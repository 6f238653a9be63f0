"""Drop-in boundary checks that need no GPU: parameter tree, init known-answers, state_dict round trip,
shim import path, loud failure on CPU tensors (SURVEY.md section 8 rows a1, a13, a14, b)."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLD, ROOT, build_module, manifest
from oracle import dstformer_oracle as O


@pytest.mark.parametrize("cfg", [O.BASE, O.LITE], ids=["base", "lite"])
def test_state_dict_names_shapes_order(cfg):
    m = build_module(cfg)
    sd = m.state_dict()
    ref = O.param_shapes(cfg)
    assert list(sd.keys()) == list(ref.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == ref[k], k
    assert all(isinstance(p, torch.nn.Parameter) for p in m.parameters())
    assert [p.data_ptr() for p in m._ordered_params()] == [v.data_ptr() for v in sd.values()]


@pytest.mark.parametrize("which,cfg", [("base", O.BASE), ("lite", O.LITE)])
def test_seeded_init_is_bit_identical_to_reference(which, cfg):
    """torch.manual_seed(0) + construction must reproduce the reference's init (SURVEY.md 8c checksums)."""
    kat = manifest()["init_kat"][which]
    torch.manual_seed(0)
    m = build_module(cfg)
    sd = m.state_dict()
    sha = hashlib.sha256(b"".join(v.contiguous().numpy().tobytes() for v in sd.values())).hexdigest()[:16]
    assert len(sd) == kat["n_tensors"] and sha == kat["sha16"]
    assert abs(sum(float(v.double().sum()) for v in sd.values()) - kat["sum"]) < 1e-6
    for i in range(cfg.depth):                       # DSTformer.py:306-311
        assert float(m.ts_attn[i].weight.abs().sum()) == 0.0 and torch.all(m.ts_attn[i].bias == 0.5)


def test_strict_load_module_prefix_and_partial_train():
    cfg = O.LITE
    P = O.make_params(cfg, 5)
    m = build_module(cfg, P)
    # DataParallel-style checkpoint keys (lib/utils/learning.py:57-58 strips 'module.')
    ck = {"module." + k: torch.from_numpy(v) for k, v in P.items()}
    m2 = build_module(cfg)
    md = m2.state_dict()
    md.update({k[7:]: v for k, v in ck.items()})
    m2.load_state_dict(md, strict=True)
    for (k, a), b in zip(m.state_dict().items(), m2.state_dict().values()):
        assert torch.equal(a, b), k
    # partial_train_layers-style freezing by name substring (learning.py:69-77)
    for name, p in m.named_parameters():
        p.requires_grad = "head" in name
    assert sum(p.requires_grad for p in m.parameters()) == 2


def test_api_surface():
    m = build_module(O.BASE)
    for attr in ("dim_out", "dim_feat", "joints_embed", "pos_drop", "blocks_st", "blocks_ts", "norm", "pre_logits",
                 "head", "temp_embed", "pos_embed", "att_fuse", "ts_attn"):
        assert hasattr(m, attr), attr
    assert m.get_classifier() is m.head
    assert m.eps == pytest.approx(1e-6)
    m.reset_classifier(5)
    assert m.head.out_features == 5 and m.head.in_features == m.dim_feat


def test_cpu_tensor_fails_loudly_no_fallback():
    m = build_module(O.LITE)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 4, 17, 3))
    with pytest.raises(RuntimeError, match="maxlen"):
        m(torch.zeros(1, 244, 17, 3))
    with pytest.raises(RuntimeError, match="num_joints"):
        m(torch.zeros(1, 4, 16, 3))


# lib/utils/learning.py of the stand-in checkout: constructs the backbone with recorded constructor arguments
_STANDIN_FACTORY = '''
import importlib
from functools import partial

from lib.model.DSTformer import DSTformer


def _arg(v):
    if isinstance(v, dict) and "partial" in v:
        mod, _, name = v["partial"].rpartition(".")
        return partial(getattr(importlib.import_module(mod), name), *v["args"], **v["keywords"])
    return v


def load_backbone(recorded_kwargs):
    return DSTformer(**{k: _arg(v) for k, v in recorded_kwargs.items()})
'''

_SHIM_CHECK = '''
import json, sys
import motionbert_b200
import lib.model.drop as dr
from lib.utils.learning import load_backbone
from oracle import dstformer_oracle as O
gold = json.load(open(sys.argv[1]))
for name, c in gold["configs"].items():
    m = load_backbone(c["kwargs"])
    assert type(m) is motionbert_b200.DSTformer, name
    assert m.eps == c["kwargs"]["norm_layer"]["keywords"]["eps"] == 1e-6, name
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert shapes == O.param_shapes({"base": O.BASE, "lite": O.LITE}[name]), name
assert dr.__file__.startswith(sys.argv[2]), dr.__file__
print("ok")
'''


def test_shim_shadows_exactly_the_reference_module(tmp_path):
    """lib/ is a namespace package in the reference: shim first on sys.path replaces only lib.model.DSTformer.

    The reference's side is a stand-in checkout laid out as tests/golden/load_backbone.json records the real one
    (oracle/make_golden_backbone.py): the same namespace packages and lib/model modules, a DSTformer module that must
    never be imported, and a factory passing the constructor arguments the reference's load_backbone was recorded
    passing for DSTformer-base and -Lite."""
    code = ("import lib.model.DSTformer as D, motionbert_b200; "
            "assert D.DSTformer is motionbert_b200.DSTformer; print('ok')")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "shim"), ROOT]))
    r = subprocess.run([sys.executable, "-P", "-c", code], capture_output=True, text=True, env=env)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr
    gold_path = os.path.join(GOLD, "load_backbone.json")
    with open(gold_path) as f:
        gold = json.load(f)
    assert gold["namespace_packages"] == ["lib", "lib.model", "lib.utils"]
    ref = tmp_path / "MotionBERT"
    for pkg in gold["namespace_packages"]:
        (ref / pkg.replace(".", os.sep)).mkdir(parents=True, exist_ok=True)
    for mod in gold["lib_model_modules"]:
        (ref / "lib" / "model" / f"{mod}.py").write_text("")
    (ref / "lib" / "model" / "DSTformer.py").write_text("raise ImportError('the shim did not shadow lib.model.DSTformer')\n")
    (ref / "lib" / "utils" / "learning.py").write_text(_STANDIN_FACTORY)
    env["PYTHONPATH"] += os.pathsep + str(ref)
    r = subprocess.run([sys.executable, "-P", "-c", _SHIM_CHECK, gold_path, str(ref)], capture_output=True, text=True,
                       env=env)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr


def test_backward_phase_of_every_parameter_matches_its_name():
    """`_param_phases` lays the flat gradient bucket out in the order mb_backward finishes the gradients
    (tail, depth d-1 ... 0, embed); check it against the parameter names."""
    import re

    from motionbert_b200 import DSTformer
    m = DSTformer(dim_feat=256, depth=3, num_heads=8, mlp_ratio=2)
    names = {id(p): n for n, p in m.named_parameters()}
    ph = m._param_phases()
    ps = m._ordered_params()
    assert len(ph) == len(ps) == 4 + 2 * 3 * 24 + 6 + 2 * 3
    for p, k in zip(ps, ph):
        n = names[id(p)]
        mt = re.match(r"(blocks_st|blocks_ts|ts_attn)\.(\d+)\.", n)
        if mt:
            assert k == 1 + (3 - 1 - int(mt.group(2))), n
        elif n in ("temp_embed", "pos_embed") or n.startswith("joints_embed"):
            assert k == 3 + 1, n
        else:
            assert k == 0 and (n.startswith("norm.") or n.startswith("pre_logits") or n.startswith("head.")), n


def test_gradient_allreduce_needs_a_process_group_and_can_be_switched_off():
    from motionbert_b200 import DSTformer
    m = DSTformer(dim_feat=256, depth=1, num_heads=8, mlp_ratio=2)
    assert m._grad_sync is None
    with pytest.raises(RuntimeError, match="process group"):
        m.enable_gradient_allreduce()
    assert m.enable_gradient_allreduce(enabled=False) is m and m._grad_sync is None


def test_native_backward_eligibility_is_decided_on_the_host_and_unsupported_configurations_raise():
    """There is no PyTorch-op fallback backward: configurations mb_backward does not cover raise on the host."""
    import torch

    from motionbert_b200 import DSTformer
    m = DSTformer(dim_feat=256, depth=1, num_heads=8, mlp_ratio=2)
    x = torch.zeros(1, 2, 17, 3)
    m._check_native_backward(x)                                # fp32 contiguous parameters on x's device: fine
    m.ts_attn[0].weight.data = m.ts_attn[0].weight.data.double()
    with pytest.raises(NotImplementedError, match="fp32"):
        m._check_native_backward(x)
    m2 = DSTformer(dim_feat=256, depth=1, num_heads=8, mlp_ratio=2, att_fuse=False)
    m2._check_native_backward(x)                               # no fusion head: native (constant 0.5 / 0.5 fusion)
    assert m2._head_param_slots() == (56, 57) and len([p for p in m2._ordered_params() if p is None]) == 2
    m3 = DSTformer(dim_feat=256, depth=1, num_heads=8, mlp_ratio=2, dim_out=17)
    with pytest.raises(NotImplementedError, match="dim_out"):
        m3._check_native_backward(x)


def test_data_parallel_replicas_still_see_their_parameters_for_the_gradient_decision():
    """nn.DataParallel replicas keep their parameters as plain attributes (`_parameters` is empty), so the
    needs-gradient decision must not go through `self.parameters()` (train.py:256-258 wraps the backbone)."""
    import torch

    from motionbert_b200 import DSTformer
    m = DSTformer(dim_feat=256, depth=1, num_heads=8, mlp_ratio=2)
    rep = m._replicate_for_data_parallel()
    for name, sub in m.named_modules():
        if name:
            parent = rep
            *path, leaf = name.split(".")
            for t in path:
                parent = parent._modules[t]
            parent._modules[leaf] = sub._replicate_for_data_parallel()
    # what torch.nn.parallel.replicate does: parameters become non-leaf attribute tensors
    for name, sub in rep.named_modules():
        src = dict(m.named_modules())[name]
        for k, p in src._parameters.items():
            if p is not None:
                setattr(sub, k, p * 1.0)
    assert len(list(rep.parameters())) == 0
    ps = rep._ordered_params()
    assert len(ps) == 60 and all(p.requires_grad for p in ps)


def test_math_modes_are_a_host_side_switch():
    from motionbert_b200 import DSTformer, _lib
    m = DSTformer(dim_feat=256, depth=1, num_heads=8, mlp_ratio=2)
    assert (m.math_mode, m.train_math_mode) == (_lib.MB_MATH_F16C, _lib.MB_MATH_BF16X3)
    m.set_math_mode("bf16")
    assert (m.math_mode, m.train_math_mode) == (_lib.MB_MATH_BF16, _lib.MB_MATH_BF16)
    m.set_math_mode("bf16x3")
    assert (m.math_mode, m.train_math_mode) == (_lib.MB_MATH_BF16X3, _lib.MB_MATH_BF16X3)
    with pytest.raises(KeyError):
        m.set_math_mode("fp64")
