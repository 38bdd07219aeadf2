"""Drop-in proof for INTEGRATION.md section 2 (CPU only): a full-object checkpoint written by the REAL reference
(``torch.save({'model': model})``, train.py:424-435; stored in tests/golden/dropin_reference.npz by
oracle/gen_golden_dropin.py) is unpickled into the shadow modules (``sys.modules['models.common'] = icafusion_b200.common``
etc.), goes through what ``attempt_load`` does (models/experimental.py:113-121: ``ckpt['model'].float().fuse().eval()``),
loads the reference's state_dict with ``strict=True`` and walks the product path (dry run: meta tensors, every kernel launch
planned, none issued)."""
import subprocess
import sys
import textwrap

import torch

from conftest import ROOT, load_golden
from oracle.gen_golden_dropin import COMMON_CLASSES, fill_state_dict, init_signature


def _write_reference_checkpoint(path, sd_path):
    """The reference's checkpoint bytes and its state_dict (rebuilt from the stored layout, exactly what it held)."""
    m, d = load_golden("dropin_reference")
    with open(path, "wb") as f:
        f.write(d["ckpt"].tobytes())
    fill = fill_state_dict(m["sd"])
    torch.save({k: fill[k] if k in fill else torch.from_numpy(d["sd:" + k]) for k, _, _ in m["sd"]}, sd_path)


def test_reference_checkpoint_unpickles_into_shadow_modules(tmp_path):
    ckpt, sdp = str(tmp_path / "last.pt"), str(tmp_path / "sd.pt")
    _write_reference_checkpoint(ckpt, sdp)
    code = textwrap.dedent(f"""
        import sys, torch
        sys.path.insert(0, {ROOT!r})
        import icafusion_b200.common as C, icafusion_b200.yolo_test as Y
        import types
        pkg = types.ModuleType("models"); pkg.__path__ = []
        sys.modules["models"] = pkg                    # INTEGRATION.md section 2: shadow before anything imports the reference
        sys.modules["models.common"] = C
        sys.modules["models.yolo_test"] = Y
        from icafusion_b200 import ops
        ck = torch.load({ckpt!r}, map_location="cpu", weights_only=False)
        m = ck["model"]
        assert type(m) is Y.Model and type(m.model[0]) is C.Conv and type(m.model[-1]) is Y.Detect, type(m)
        assert type(m.model[20]) is C.TransformerFusionBlock and type(m.model[20].crosstransformer[0].crossatt) is C.CrossAttention
        m = m.float().fuse().eval()                    # models/experimental.py:118
        assert not hasattr(m.model[0], "bn") and m.model[0].conv.bias is not None
        # the reference's own state_dict (unfused layout) loads strictly into a freshly built shadow model
        fresh = Y.Model("yolov5s_Transfusion_kaist")
        sd = torch.load({sdp!r}, map_location="cpu")
        missing = fresh.load_state_dict(sd, strict=True)
        assert not missing.missing_keys and not missing.unexpected_keys
        fresh = fresh.eval().fuse()
        for (ka, va), (kb, vb) in zip(sorted(m.state_dict().items()), sorted(fresh.state_dict().items())):
            assert ka == kb and va.shape == vb.shape and torch.allclose(va.float(), vb.float(), atol=2e-3, rtol=2e-3), ka
        # the unpickled object drives the product path: dry-run walk (nothing launched), every conv plan accepted
        from icafusion_b200 import _lib
        import ctypes
        img = torch.empty(1, 3, 512, 640, dtype=torch.uint8, device="meta")
        with torch.no_grad(), ops.dry_run() as dr:
            z, logits, xs = m.half()(img, img)
        assert tuple(z.shape) == (1, 20160, 6) and len(xs) == 3
        convs = [w for n, a, w in dr.records if n == "icaf_conv2d_fwd"]
        assert len(convs) >= 60
        for w in convs:
            pl = _lib.ConvPlan()
            assert _lib.lib().icaf_conv2d_plan(ctypes.byref(w["geom"]), w["n_io"], 148, -1, ctypes.byref(pl)) == 0
        print("ok", len(dr.records))
    """)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-1000:], out.stderr[-3000:])
    assert out.stdout.strip().startswith("ok")


def test_shadow_modules_export_the_reference_names():
    """Every class the Transfusion YAMLs / pickles name exists in the shadow modules with the reference's constructor
    signature (parameter names and defaults)."""
    import icafusion_b200.common as C
    import icafusion_b200.yolo_test as Y
    ref = load_golden("dropin_reference")[0]["signatures"]
    for name in COMMON_CLASSES:
        assert name in ref and hasattr(C, name), name
    for name in ("Conv", "Bottleneck", "C3", "SPPF", "Concat", "TransformerFusionBlock", "CrossTransformerBlock", "CrossAttention",
                 "AdaptivePool2d"):
        assert init_signature(getattr(C, name)) == ref[name], name
    for name in ("Model", "Detect"):
        assert hasattr(Y, name)
    assert [p for p, _ in init_signature(Y.Detect)] == [p for p, _ in ref["Detect"]]
