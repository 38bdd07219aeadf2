"""Host-side logic that needs no GPU: config generation, graph building, state_dict parity with the reference,
filter packing layout, BN folding, pooling geometry."""
import pytest
import torch

from conftest import load_golden
from icafusion_b200 import Model, TransformerFusionBlock, ops
from icafusion_b200.cfg import load_cfg, transfusion_kaist_cfg
from icafusion_b200.common import AdaptivePool2d, Conv
from icafusion_b200.yolo_test import fuse_conv_and_bn
from oracle import icaf_oracle as O
from oracle import synth


@pytest.mark.parametrize("size", ["s", "l"])
def test_state_dict_layout_matches_reference(size):
    """Keys/shapes equal oracle.synth.model_param_shapes, which gen_golden loaded into the real reference with strict
    matching -- so reference checkpoints load here with strict=True."""
    if size == "l":
        with torch.device("meta"):
            m = Model(f"yolov5{size}_Transfusion_kaist")
    else:
        m = Model(f"yolov5{size}_Transfusion_kaist")
    own = {k: tuple(v.shape) for k, v in m.state_dict().items() if not k.endswith(("anchors", "anchor_grid"))}
    want = {k: tuple(v) for k, v in synth.model_param_shapes(load_cfg(f"yolov5{size}_Transfusion_kaist")).items()}
    assert own == want
    assert m._ir_start == 10 and len(m.model) == 38
    n_params = sum(p.numel() for p in m.parameters())
    assert abs(n_params / 1e6 - (23.26 if size == "s" else 120.25)) < 0.01     # SURVEY.md section 8(a)


@pytest.mark.parametrize("size", ["s", "l"])
def test_generated_cfg_equals_reference_yaml(size):
    """models/transformer/yolov5{s,l}_Transfusion_kaist.yaml as the reference parses it (stored by oracle/gen_golden_dropin.py)."""
    ref = load_golden("dropin_reference")[0]["cfg"][size]
    mine = transfusion_kaist_cfg(size)
    for k in ("nc", "depth_multiple", "width_multiple", "anchors", "backbone", "head"):
        assert mine[k] == ref[k], k


def test_dmff_block_state_dict_and_defaults():
    blk = TransformerFusionBlock(128, 10, 10)
    assert {f"blk.{k}": tuple(v.shape) for k, v in blk.state_dict().items()} == \
        {k: tuple(v) for k, v in synth.dmff_param_shapes(128, 100, "blk").items()}
    assert blk.crosstransformer[0].loops == 1 and blk.crosstransformer[0].crossatt.h == 8   # common.py:691,763


def test_pack_conv_weight_layout():
    w = torch.randn(20, 16, 3, 3)
    pk = ops.pack_conv_weight(w, torch.zeros(20), 1, 1, ops.ACT_SILU)
    assert pk.w.shape == (32, 192) and pk.cin == 16 and pk.cout == 20
    # K order is (ky, kx, c): element [n, (ky*3+kx)*16 + c] == w[n, c, ky, kx]
    assert torch.equal(pk.w[:20, :144].float().view(20, 3, 3, 16), w.half().float().permute(0, 2, 3, 1))
    assert float(pk.w[20:].abs().max()) == 0 and float(pk.w[:, 144:].abs().max()) == 0
    stem = ops.pack_conv_weight(torch.randn(32, 3, 6, 6), None, 2, 2, ops.ACT_SILU)
    assert stem.cin == 4 and stem.w.shape == (32, 192)
    assert float(stem.w[:, :144].view(32, 36, 4)[..., 3].abs().max()) == 0        # padded 4th input channel


def test_fuse_conv_and_bn_matches_oracle_fold():
    c = Conv(16, 24, 3, 1).eval()
    sd = synth.synth_state_dict({f"m.{k}": tuple(v.shape) for k, v in c.state_dict().items()}, 1)
    c.load_state_dict({k[2:]: v for k, v in sd.items()})
    c.bn.eps = 1e-3
    f = fuse_conv_and_bn(c.conv, c.bn)
    folded = O.fold_bn(sd, 1e-3)
    assert torch.allclose(f.weight, folded["m.conv.weight"], atol=1e-6)
    assert torch.allclose(f.bias, folded["m.conv.bias"], atol=1e-6)


def test_adaptive_pool_geometry():
    p = AdaptivePool2d(20, 20)
    assert p.out_size(64, 80) == (20, 20) and p.out_size(16, 20) == (16, 20) and p.out_size(20, 20) == (20, 20)
    with pytest.raises(ValueError):
        AdaptivePool2d(16, 16).out_size(8, 20)        # the reference divides by zero here (common.py:880)


def test_model_fuse_removes_bn_and_rebinds_forward():
    m = Model("yolov5s_Transfusion_kaist").eval().fuse()
    convs = [x for x in m.modules() if type(x) is Conv]
    assert convs and not any(hasattr(c, "bn") for c in convs) and all(c.conv.bias is not None for c in convs)
    assert not any(".bn." in k for k in m.state_dict())


def test_stem_space_to_depth_repack_is_the_same_convolution():
    """ops.pack_stem_weight: the 6x6 / stride 2 / pad 2 image stem (models/common.py:36-60 with the YAML row
    [-1, 1, Conv, [c, 6, 2, 2]]) equals a 3x3 / stride 1 / pad 1 convolution over the space-to-depth frame that
    icaf_pack_image_s2d produces (channel (dy*2+dx)*4 + c).  Pure fp32 torch on the CPU: the identity is exact up to
    summation order."""
    import torch.nn.functional as F
    from icafusion_b200 import ops
    g = torch.Generator().manual_seed(3)
    img = torch.rand(2, 3, 32, 48, generator=g)
    w = torch.randn(8, 3, 6, 6, generator=g)
    b = torch.randn(8, generator=g)
    ref = F.conv2d(img, w, b, stride=2, padding=2)
    pk = ops.pack_stem_weight(w, b, ops.ACT_NONE, device="cpu")
    assert (pk.cin, pk.kh, pk.kw, pk.stride, pk.pad) == (16, 3, 3, 1, 1)
    # unpack the GEMM filter matrix [Cout^32][K^64], K order (ky, kx, c), back to (Cout, 16, 3, 3)
    ws = pk.w[:8, :144].float().view(8, 3, 3, 16).permute(0, 3, 1, 2)
    # space-to-depth frame exactly as icaf_pack_image_s2d lays it out: channel (dy*2+dx)*4 + c, c = r,g,b,0
    B, _, H, W = img.shape
    x4 = torch.cat([img, img.new_zeros(B, 1, H, W)], 1)
    s2d = x4.view(B, 4, H // 2, 2, W // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(B, 16, H // 2, W // 2)
    out = F.conv2d(s2d, ws, b, stride=1, padding=1)
    assert out.shape == ref.shape
    # the packed filter is fp16: compare against the fp16-rounded 6x6 filter
    ref16 = F.conv2d(img, w.half().float(), b, stride=2, padding=2)
    assert float((out - ref16).abs().max()) < 1e-4


def test_resize_taps_reproduce_cv2_bilinear():
    """icafusion_b200/datasets.py:resize_taps + the kernel's integer arithmetic (restated in numpy) == cv2.resize(INTER_LINEAR)
    on uint8, bit for bit -- the host half of the device letterbox (utils/datasets.py:1404-1427)."""
    cv2 = pytest.importorskip("cv2")
    import numpy as np
    from icafusion_b200.datasets import letterbox_geometry, resize_taps
    g = np.random.Generator(np.random.PCG64(1))
    for (H0, W0), (h, w) in (((300, 400), (480, 640)), ((1080, 1920), (360, 640)), ((333, 517), (412, 640)), ((64, 80), (640, 800)),
                             ((720, 1280), (378, 672)), ((517, 333), (640, 412))):
        img = g.integers(0, 256, (H0, W0, 3), dtype=np.uint8)
        xt, yt = resize_taps(W0, w).astype(np.int64), resize_taps(H0, h, vertical=True).astype(np.int64)
        src = img.astype(np.int64)
        rows = src[:, xt[:, 0]] * xt[:, 2][None, :, None] + src[:, xt[:, 1]] * xt[:, 3][None, :, None]        # (H0, w, 3)
        out = (((yt[:, 2][:, None, None] * (rows[yt[:, 0]] >> 4)) >> 16) + ((yt[:, 3][:, None, None] * (rows[yt[:, 1]] >> 4)) >> 16) + 2) >> 2
        want = cv2.resize(img, (w, h), interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(out.astype(np.uint8), want), (H0, W0, h, w, int(np.abs(out - want).max()))
    (nw, nh), ratio, (dw, dh), (top, bottom, left, right) = letterbox_geometry((512, 640), (640, 640))
    assert (nw, nh, top, bottom, left, right) == (640, 512, 64, 64, 0, 0) and ratio == (1.0, 1.0)      # the KAIST frame: bands only
