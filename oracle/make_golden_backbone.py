"""Generate tests/golden/load_backbone.json from a checkout of the reference (MotionBERT).

    python oracle/make_golden_backbone.py /path/to/MotionBERT

Records what the shim (shim/lib/model/DSTformer.py) relies on: which of `lib`, `lib.model`, `lib.utils` are namespace
packages (no __init__.py, so a directory earlier on sys.path can supply one module of them), the modules next to
`lib/model/DSTformer.py`, and the arguments the reference's own factory `lib.utils.learning.load_backbone` passes to
the DSTformer constructor for DSTformer-base and DSTformer-Lite.  The constructor is replaced by a recorder while the
factory runs.  No reference source is copied: only names and the arguments it produced.
"""
from __future__ import annotations

import functools
import json
import os
import sys
import types
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "load_backbone.json")

# the two shipped encoders (configs/pretrain/MB_pretrain.yaml and MB_lite.yaml)
CONFIGS = {
    "base": dict(backbone="DSTformer", dim_feat=512, dim_rep=512, depth=5, num_heads=8, mlp_ratio=2, maxlen=243,
                 num_joints=17),
    "lite": dict(backbone="DSTformer", dim_feat=256, dim_rep=512, depth=5, num_heads=8, mlp_ratio=4, maxlen=243,
                 num_joints=17),
}


def _jsonable(v):
    if isinstance(v, functools.partial):
        return {"partial": f"{v.func.__module__}.{v.func.__qualname__}", "args": [_jsonable(a) for a in v.args],
                "keywords": {k: _jsonable(a) for k, a in v.keywords.items()}}
    if isinstance(v, (bool, int, float, str)) or v is None:
        return v
    raise TypeError(f"cannot record a {type(v).__name__} argument")


def main(ref: str) -> None:
    calls = []

    class Recorder:
        def __init__(self, *args, **kwargs):
            calls.append((args, kwargs))

    stub = types.ModuleType("lib.model.DSTformer")
    stub.DSTformer = Recorder
    sys.modules["lib.model.DSTformer"] = stub
    sys.path.insert(0, ref)
    from lib.utils.learning import load_backbone

    out = {"namespace_packages": [p for p in ("lib", "lib.model", "lib.utils")
                                  if not os.path.exists(os.path.join(ref, *p.split("."), "__init__.py"))],
           "lib_model_modules": sorted(f[:-3] for f in os.listdir(os.path.join(ref, "lib", "model")) if f.endswith(".py")),
           "configs": {}}
    for name, args in CONFIGS.items():
        calls.clear()
        load_backbone(SimpleNamespace(**args))
        assert len(calls) == 1, calls
        pos, kw = calls[0]
        assert not pos, pos
        out["configs"][name] = {"args": args, "kwargs": {k: _jsonable(v) for k, v in kw.items()}}
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", OUT)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
