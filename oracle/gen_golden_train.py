"""Generate tests/golden/train_yolov5s_320.npz by executing the REAL reference's training step (build container only).

    python -m oracle.gen_golden_train

One step of train.py:334-344 on CPU fp32: reference ``Model`` in ``train()`` (BatchNorm batch statistics, nearest DMFF tail),
every ``nn.Dropout`` set to p = 0 (torch's dropout masks cannot be reproduced by another implementation), reference
``ComputeLoss``, ``loss.backward()``.  Stored: the loss, a fingerprint (L2 norm + two seeded projections, float64) of every
parameter gradient and of the three Detect outputs, and the updated running statistics of three BatchNorm layers.  Weights,
images and targets are seeded (oracle/synth.py, gen_golden_loss.synth_targets) and rebuilt by the tests.
"""
from __future__ import annotations

import json
import os
import sys
import warnings
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import synth  # noqa: E402
from oracle.ref_shim import REF_ROOT, load_reference  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
HYP = dict(box=0.05, obj=1.0, cls=0.5, cls_pw=1.0, obj_pw=1.0, anchor_t=4.0, fl_gamma=0.0)
CASE = dict(name="train_yolov5s_320", size="s", B=2, H=320, W=320, nt=12, seed=1234)
BN_PROBES = ["model.0.bn", "model.4.cv3.bn", "model.10.bn", "model.22.conv1x1_out.bn"]
# intra-op threads of the stored run.  The step's gradients move by up to ~1.5e-3 of their norm with the CPU summation order
# (BatchNorm batch statistics in the backward), so whoever replays the step on the CPU uses the same thread count.
THREADS = 8


def synth_targets(nt: int, B: int, seed: int) -> np.ndarray:
    g = np.random.Generator(np.random.PCG64([seed, 77]))
    t = np.zeros((nt, 6), dtype=np.float32)
    t[:, 0] = g.integers(0, B, nt)
    t[:, 2:4] = g.uniform(0.1, 0.9, (nt, 2))
    t[:, 4:6] = np.exp(g.uniform(np.log(0.04), np.log(0.5), (nt, 2)))
    return t


def fingerprint(a: np.ndarray, key: str) -> np.ndarray:
    """[||a||_2, <a, w1>, <a, w2>] in float64, w seeded by `key`."""
    r = np.random.Generator(np.random.PCG64([23, zlib.crc32(key.encode())]))
    v = a.astype(np.float64).reshape(-1)
    return np.array([np.sqrt((v * v).sum()), v @ r.standard_normal(v.size), v @ r.standard_normal(v.size)], dtype=np.float64)


def main():
    warnings.filterwarnings("ignore")
    torch.set_num_threads(THREADS)
    _, yolo = load_reference()
    from utils.loss import ComputeLoss
    c = CASE
    cfg = os.path.join(REF_ROOT, "models", "transformer", f"yolov5{c['size']}_Transfusion_kaist.yaml")
    model = yolo.Model(cfg, ch=3, nc=1)
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    sd = synth.synth_state_dict(shapes, c["seed"])
    missing = model.load_state_dict(sd, strict=False)
    assert all(k.endswith(("anchors", "anchor_grid")) for k in missing.missing_keys) and not missing.unexpected_keys
    model.train()
    for m in model.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    model.hyp, model.gr = dict(HYP), 1.0
    rgb, ir = synth.synth_images(c["B"], c["H"], c["W"], c["seed"])
    t = synth_targets(c["nt"], c["B"], c["seed"])
    pred = model(rgb, ir)                                                        # train.py:336
    loss, items = ComputeLoss(model)(pred, torch.from_numpy(t))                  # train.py:338
    loss.backward()                                                              # train.py:344
    arrays = {"targets": t, "out": np.concatenate([loss.detach().numpy().reshape(1), items.numpy()]).astype(np.float32)}
    names, dead = [], []
    for k, p in model.named_parameters():
        if p.grad is None:
            dead.append(k)
            continue
        names.append(k)
        arrays["g:" + k] = fingerprint(p.grad.numpy(), k)
    for i, x in enumerate(pred):
        arrays[f"pred{i}"] = fingerprint(x.detach().numpy(), f"pred{i}")
    state = model.state_dict()
    for k in BN_PROBES:
        arrays["rm:" + k] = state[k + ".running_mean"].numpy().copy()
        arrays["rv:" + k] = state[k + ".running_var"].numpy().copy()
    meta = dict(c, hyp=HYP, gr=1.0, params=names, dead_params=dead, bn_probes=BN_PROBES,
                reference="models/yolo_test.py Model.train() forward + utils/loss.py ComputeLoss + backward (train.py:334-344), dropout p=0, fp32 CPU",
                torch=torch.__version__)
    path = os.path.join(OUT, c["name"] + ".npz")
    np.savez_compressed(path, meta=np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8), **arrays)
    print(f"loss {arrays['out']}  {len(names)} live / {len(dead)} dead parameters  -> {path} ({os.path.getsize(path) / 1e3:.0f} kB)")


if __name__ == "__main__":
    main()
