"""Pins oracle/icaf_oracle.py to outputs of the real reference (tests/golden/*.npz, produced by
oracle/gen_golden.py in the build container).  CPU only."""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_golden, normwise
from icafusion_b200.cfg import load_cfg
from oracle import icaf_oracle as O
from oracle import synth

DMFF = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "dmff_*.npz")))
MODELS = ["yolov5s_320", "yolov5s_512x640"]   # yolov5l replay is in the gpu suite (CPU time)

TOL_FP32 = 2e-5   # fp32 vs fp32, different op order only


@pytest.mark.parametrize("name", DMFF)
def test_dmff_oracle_matches_reference(name):
    m, d = load_golden(name)
    sd = synth.synth_state_dict(synth.dmff_param_shapes(m["C"], m["va"] * m["ha"], "blk"), m["seed"])
    rgb, ir = synth.synth_features(m["B"], m["C"], m["H"], m["W"], m["seed"])
    with torch.no_grad():
        r, _, _ = O.dmff_tokens(rgb, sd, "blk", "vis", m["va"], m["ha"])
        i, _, _ = O.dmff_tokens(ir, sd, "blk", "ir", m["va"], m["ha"])
        tr, ti = O.cross_transformer_block(r, i, sd, "blk.crosstransformer.0", m["loops"])
        out = O.dmff_block(rgb, ir, sd, "blk", m["va"], m["ha"], m["loops"], bn_eps=m["bn_eps"])
    assert normwise(tr.numpy(), d["tok_vis"]) < TOL_FP32
    assert normwise(ti.numpy(), d["tok_ir"]) < TOL_FP32
    assert normwise(out.numpy(), d["out"]) < TOL_FP32


@pytest.mark.parametrize("name", MODELS)
def test_model_oracle_matches_reference(name):
    m, d = load_golden(name)
    cfg = load_cfg(f"yolov5{m['size']}_Transfusion_kaist")
    sd = synth.synth_state_dict(synth.model_param_shapes(cfg), m["seed"])
    rgb, ir = synth.synth_images(m["B"], m["H"], m["W"], m["seed"])
    with torch.no_grad():
        z, lg, xs = O.model_forward(sd, cfg, rgb, ir)
        zf = O.model_forward(O.fold_bn(sd), cfg, rgb, ir)[0]
    assert z.shape == d["z"].shape
    assert normwise(z.numpy(), d["z"]) < TOL_FP32
    assert normwise(lg.numpy(), d["logits"]) < TOL_FP32
    assert normwise(zf.numpy(), d["z_fused"]) < TOL_FP32       # fold_bn == Model.fuse()
    for j in range(3):
        assert normwise(xs[j].numpy(), d[f"x{j}"].astype(np.float32)) < 2e-3   # stored as fp16


def test_flop_accounting_matches_survey():
    # SURVEY.md section 8(a): hook-counted on the reference: 24.61 / 155.82 GFLOP per 512x640 pair
    s = O.model_conv_flops(load_cfg("yolov5s_Transfusion_kaist"), 512, 640) / 1e9
    l = O.model_conv_flops(load_cfg("yolov5l_Transfusion_kaist"), 512, 640) / 1e9
    assert abs(s - 24.61) < 0.02 and abs(l - 155.82) < 0.05, (s, l)
    assert abs(O.dmff_flops(1, 256, 64, 80, 400) / 1e9 - 2.928) < 0.01


def test_nms_oracle_matches_reference_golden():
    """oracle.non_max_suppression (incl. its restated greedy NMS) reproduces the REAL reference's output rows exactly
    (tests/golden/nms_cases.npz from oracle/gen_golden_nms.py), and the greedy NMS equals torchvision's on random boxes."""
    m, d = load_golden("nms_cases")
    pred = torch.from_numpy(d["pred"])
    for st in m["settings"]:
        out = O.non_max_suppression(pred, st["conf"], st["iou"], classes=st["classes"], agnostic=st["agnostic"])
        for b, o in enumerate(out):
            want = d[f"{st['name']}_{b}"]
            assert o.shape[0] == st["counts"][b] == want.shape[0]
            assert np.array_equal(o.numpy(), want), (st["name"], b)
    try:
        import torchvision
    except Exception:  # noqa: BLE001
        return
    g = torch.Generator().manual_seed(0)
    xy = torch.rand(3000, 2, generator=g) * 600
    wh = torch.rand(3000, 2, generator=g) * 120 + 2
    boxes, scores = torch.cat([xy, xy + wh], 1), (torch.rand(3000, generator=g) * 64).round() / 64     # many score ties
    for thr in (0.3, 0.45, 0.6):
        assert torch.equal(O.greedy_nms(boxes, scores, thr), torchvision.ops.nms(boxes, scores, thr))


def test_loss_oracle_matches_reference_golden():
    """oracle.compute_loss reproduces the REAL reference's ComputeLoss outputs (tests/golden/loss_cases.npz,
    oracle/gen_golden_loss.py) on the seeded predictions / stored targets."""
    from oracle.gen_golden_loss import synth_case
    m, d = load_golden("loss_cases")
    for cs in m["cases"]:
        p, t = synth_case(cs["name"], cs["nc"], cs["B"], cs["nt"])
        assert np.array_equal(t, d[f"{cs['name']}_targets"])
        pt = [torch.from_numpy(x).requires_grad_(True) for x in p]
        loss, items = O.compute_loss(pt, torch.from_numpy(t), torch.from_numpy(d[f"{cs['name']}_anchors"]), cs["hyp"], cs["gr"])
        got = np.concatenate([loss.detach().numpy().reshape(1), items.detach().numpy()])
        assert np.allclose(got, d[f"{cs['name']}_out"], rtol=2e-5, atol=1e-6), (cs["name"], got, d[f"{cs['name']}_out"])
        # the oracle's autograd graph equals the reference's (tobj and CIoU's alpha detached): its backward reproduces the
        # reference's loss.backward() -- coarsest level in full, every level through the stored fingerprint
        from oracle.gen_golden_loss import grad_fingerprint
        loss.sum().backward()
        g2 = d[f"{cs['name']}_grad2"]
        assert np.abs(pt[2].grad.numpy() - g2).max() <= 2e-5 * np.abs(g2).max(), cs["name"]
        for lvl, x in enumerate(pt):
            want = d[f"{cs['name']}_gproj{lvl}"]
            assert np.allclose(grad_fingerprint(x.grad.numpy(), lvl), want, rtol=1e-4, atol=1e-6 * want[0]), (cs["name"], lvl)


def test_training_step_oracle_matches_reference_golden():
    """oracle.train_step (train-mode forward with BatchNorm batch statistics and the nearest DMFF tail, loss, autograd backward)
    reproduces the REAL reference's training step (tests/golden/train_yolov5s_320.npz, oracle/gen_golden_train.py): loss, a
    fingerprint of every parameter gradient, the set of parameters that receive no gradient, updated BN running statistics."""
    from oracle.gen_golden_train import THREADS, fingerprint, synth_targets
    m, d = load_golden("train_yolov5s_320")
    cfg = load_cfg(f"yolov5{m['size']}_Transfusion_kaist")
    sd = synth.synth_state_dict(synth.model_param_shapes(cfg), m["seed"])
    rgb, ir = synth.synth_images(m["B"], m["H"], m["W"], m["seed"])
    t = synth_targets(m["nt"], m["B"], m["seed"])
    assert np.array_equal(t, d["targets"])
    n_threads = torch.get_num_threads()
    torch.set_num_threads(THREADS)                                  # the stored run's summation order
    try:
        loss, items, grads, pred, state = O.train_step(sd, cfg, rgb, ir, torch.from_numpy(t), m["hyp"], m["gr"])
    finally:
        torch.set_num_threads(n_threads)
    got = np.concatenate([loss.numpy().reshape(1), items.numpy()])
    assert np.allclose(got, d["out"], rtol=1e-4, atol=1e-6), (got, d["out"])
    assert sorted(grads) == sorted(m["params"])                     # the same 30 parameters stay without a gradient
    worst = 0.0
    for k in m["params"]:
        want = d["g:" + k]
        fp = fingerprint(grads[k].numpy(), k)
        # floor: key-projection biases (softmax is shift invariant) and the last MLP biases (a per-channel constant in front of
        # a batch-statistics BatchNorm) have mathematically zero gradients -- 1e-8 rounding noise on both sides
        worst = max(worst, float(np.abs(fp - want).max() / max(want[0], 1e-3)))
    assert worst < 2e-4, worst                                      # fp32 CPU both sides (observed 4e-5)
    for i in range(3):
        want = d[f"pred{i}"]
        assert np.abs(fingerprint(pred[i].numpy(), f"pred{i}") - want).max() < 1e-4 * want[0]
    for k in m["bn_probes"]:
        assert np.allclose(state[k + ".running_mean"].numpy(), d["rm:" + k], rtol=1e-4, atol=1e-6)
        assert np.allclose(state[k + ".running_var"].numpy(), d["rv:" + k], rtol=1e-4, atol=1e-6)
