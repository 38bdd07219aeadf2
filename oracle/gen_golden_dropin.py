"""Generate tests/golden/dropin_reference.npz from the REAL reference (needs its source tree, see oracle/ref_shim.py).

    python -m oracle.gen_golden_dropin

What the drop-in tests (tests/test_dropin_cpu.py, tests/test_host_logic_cpu.py) compare against:
  * ckpt      -- a full-object checkpoint written by the reference itself (``torch.save({'model': model})`` of a half()
                 yolov5s_Transfusion_kaist Model, train.py:424-435), as raw bytes.  The weights are the periodic fill of
                 `fill_state_dict` rather than seeded noise: the file then compresses to a few hundred kB while every
                 tensor still holds distinct, fp16-exact values.
  * meta.sd   -- the reference's own state_dict layout (name, shape, dtype) of that model; the Detect anchor buffers are
                 stored as arrays ("sd:<name>"), every other entry is `fill_state_dict` of its name and shape.
  * meta.signatures -- constructor parameters (name, repr of the default) of the classes the Transfusion YAMLs and pickles
                 name, from models/common.py and models/yolo_test.py.
  * meta.cfg  -- the keys of models/transformer/yolov5{s,l}_Transfusion_kaist.yaml that icafusion_b200.cfg regenerates.
"""
from __future__ import annotations

import inspect
import io
import json
import os
import sys
import zlib
from collections import OrderedDict

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

OUT = os.path.join(ROOT, "tests", "golden", "dropin_reference.npz")
COMMON_CLASSES = ("Conv", "Bottleneck", "C3", "SPPF", "Concat", "TransformerFusionBlock", "CrossTransformerBlock", "CrossAttention",
                  "LearnableCoefficient", "LearnableWeights", "AdaptivePool2d")
YOLO_CLASSES = ("Model", "Detect")
CFG_KEYS = ("nc", "depth_multiple", "width_multiple", "anchors", "backbone", "head")


def fill_tensor(name: str, shape, dtype: str) -> torch.Tensor:
    """Deterministic weights of period 17 along the flattened tensor, offset per name; every value is k/64 (exact in
    fp16), BatchNorm weights sit around 1 and running variances are positive."""
    n = int(np.prod(shape, dtype=np.int64))
    if dtype == "int64":
        return torch.zeros(shape, dtype=torch.int64)
    k = (np.arange(n, dtype=np.int64) * 5 + zlib.crc32(name.encode())) % 17 - 8
    a = k.astype(np.float32) / 64.0
    if name.endswith("running_var"):
        a = 0.75 + np.abs(a) * 2.0
    elif ".bn.weight" in name:
        a = 1.0 + a
    return torch.from_numpy(a.reshape(shape))


def fill_state_dict(layout) -> "OrderedDict[str, torch.Tensor]":
    """`layout`: [(name, shape, dtype), ...]; the Detect anchor buffers are skipped."""
    return OrderedDict((k, fill_tensor(k, tuple(s), d)) for k, s, d in layout if not k.endswith(("anchors", "anchor_grid")))


def init_signature(cls):
    """[(parameter name, repr of its default)] of cls.__init__."""
    return [[p.name, repr(p.default)] for p in inspect.signature(cls.__init__).parameters.values()]


def main():
    import warnings
    import yaml
    from oracle.ref_shim import REF_ROOT, load_reference
    warnings.filterwarnings("ignore")
    common, yolo = load_reference()
    cfg_path = os.path.join(REF_ROOT, "models", "transformer", "yolov5s_Transfusion_kaist.yaml")
    model = yolo.Model(cfg_path, ch=3, nc=1)
    assert type(model).__module__ == "models.yolo_test"
    layout = [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in model.state_dict().items()]
    res = model.load_state_dict(fill_state_dict(layout), strict=False)
    assert not res.unexpected_keys and all(k.endswith(("anchors", "anchor_grid")) for k in res.missing_keys), res
    model.half()                                   # train.py:427 saves the half() model object
    buf = io.BytesIO()
    torch.save({"epoch": 3, "model": model, "optimizer": None}, buf)
    sd = model.float().state_dict()
    want = fill_state_dict(layout)                 # the test rebuilds the state_dict from the layout: it must be exact
    for k, v in sd.items():
        assert k in want or k.endswith(("anchors", "anchor_grid")), k
        assert k not in want or torch.equal(v, want[k].to(v.dtype)), k
    src_common = open(os.path.join(REF_ROOT, "models", "common.py")).read()
    sigs = {}
    for name in COMMON_CLASSES:
        assert f"class {name}(" in src_common, name
        sigs[name] = init_signature(getattr(common, name))
    for name in YOLO_CLASSES:
        sigs[name] = init_signature(getattr(yolo, name))
    cfg = {}
    for size in ("s", "l"):
        with open(os.path.join(REF_ROOT, "models", "transformer", f"yolov5{size}_Transfusion_kaist.yaml")) as f:
            ref = yaml.safe_load(f)
        cfg[size] = {k: ref[k] for k in CFG_KEYS}
        assert json.loads(json.dumps(cfg[size])) == cfg[size], size
    meta = dict(kind="dropin", sd=layout, signatures=sigs, cfg=cfg, torch=torch.__version__,
                reference="models/yolo_test.py Model(yolov5s_Transfusion_kaist.yaml, nc=1).half() pickled by torch.save; "
                          "models/common.py, models/yolo_test.py constructors; models/transformer/*.yaml")
    arrays = {f"sd:{k}": v.numpy() for k, v in sd.items() if k.endswith(("anchors", "anchor_grid"))}
    np.savez_compressed(OUT, meta=np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8),
                        ckpt=np.frombuffer(buf.getvalue(), dtype=np.uint8), **arrays)
    print(f"wrote {OUT}  ({os.path.getsize(OUT) / 1e6:.2f} MB; checkpoint {len(buf.getvalue()) / 1e6:.1f} MB uncompressed)")


if __name__ == "__main__":
    main()
