"""GPU, at the BENCHMARKED sizes: parity against outputs of the UNMODIFIED reference (tests/golden/make_golden_fullsize.py:
Sigma-tiny 480x640 = BASELINE config 2, Sigma-small 480x640 = config 3's forward, Sigma-base 720x960 = config 5 with its odd
45 -> 46 -> 23 stage), and against the oracle port run on the GPU box's host cores at B = 2 (no golden involved: fresh seeded
inputs, so nothing can be tuned to a fixture).

Bars (BASELINE.json north_star: "logits/mIoU match on a fixed synthetic batch"):
  composed path (fp32 dense math, op-level scan kernel): logits within 1e-3 of the logit scale, >= 99.9 % labels, mIoU 5e-4
  fused path (precision follows torch.backends.cuda.matmul.allow_tf32, sigma_b200.fused.precision()): logits within the bar stated per precision mode below; a label may
  differ from the reference's only where the reference's own top-2 margin is below twice the logit error bar."""
import contextlib
import io

import numpy as np
import pytest
import torch

import procedural as P
from helpers import SEED, cfg_tiny, golden, record
from oracle import sigma_ref

pytestmark = pytest.mark.gpu

CASES = {
    "tiny": ("sigma_tiny_480x640", "sigma_tiny", 480, 640, 9),
    "small": ("sigma_small_480x640", "sigma_small", 480, 640, 40),
    "base": ("sigma_base_720x960", "sigma_base", 720, 960, 5),
}


def _have(tag):
    import os
    from helpers import GOLDEN
    return os.path.exists(os.path.join(GOLDEN, tag + ".npz"))


def _model(backbone, H, W, ncls, seed=SEED):
    from sigma_b200 import modules as M
    with contextlib.redirect_stdout(io.StringIO()):
        model = M.EncoderDecoder(cfg_tiny(H, W, num_classes=ncls, backbone=backbone), criterion=None)
    P.fill_state_dict(model, seed)
    return model.cuda().eval()


def _check(logits, g, ncls, tag, bar, min_agree, miou_tol, H, W):
    scale = float(g["logits_absmax"])
    y0, x0, s = (int(v) for v in g["logits_step"])
    sub = logits[:, :, y0::s, x0::s].float().cpu().numpy()
    err = float(np.abs(sub - g["logits_sub"]).max())
    assert err <= bar * scale, f"{tag}: logits differ from the reference by {err:.3e} = {err / scale:.2e} of the scale {scale:.3e} (bar {bar:g})"
    pred = logits.argmax(1).cpu().numpy().astype(np.uint8)
    ref = g["argmax"]
    diff = pred != ref
    agree = 1.0 - float(diff.mean())
    assert agree >= min_agree, f"{tag}: only {agree:.5f} of the arg-max labels equal the reference's"
    # a flipped label is only acceptable at a near-tie of the REFERENCE's own logits; the fixture keeps the margin of the
    # pixels where it is at most tie_bound of the scale, everywhere else a flip fails
    assert 2.5 * bar <= float(g["tie_bound"])
    tie = np.unpackbits(g["tie_mask"], count=diff.size).astype(bool)
    margin = np.full(diff.size, np.inf, np.float32)
    margin[tie] = g["tie_margin"]
    margin = margin.reshape(diff.shape)
    worst = float(margin[diff].max()) if diff.any() else 0.0
    assert worst <= 2.5 * bar * scale, f"{tag}: a label flipped where the reference's top-2 margin is {worst:.3e}"
    gt = (P.rand(SEED, tag + "/gt", (1, H, W)) * ncls).long().clamp(max=ncls - 1).numpy()
    _, miou = sigma_ref.mean_iou(pred, gt, ncls)
    assert abs(miou - float(g["miou"])) <= miou_tol, f"{tag}: mIoU {miou} vs reference {float(g['miou'])}"
    return err / scale, agree


@pytest.mark.parametrize("which", ["tiny", "small", "base"])
@pytest.mark.parametrize("path", ["fused_tf32x3", "fused_tf32x3_cudnn_tf32", "fused_tf32", "composed"])
def test_logits_vs_reference_golden_fullsize(which, path):
    tag, backbone, H, W, ncls = CASES[which]
    if not _have(tag):
        pytest.skip(f"{tag}.npz not generated")
    if path in ("composed", "fused_tf32x3_cudnn_tf32") and which != "tiny":
        pytest.skip("covered at the tiny size; small/base run the two fused precisions")
    from sigma_b200 import fused, modules as M
    torch.backends.cuda.matmul.allow_tf32 = path == "fused_tf32"    # the fused path's precision follows torch's switch
    # "fused_tf32x3_cudnn_tf32" is EXACTLY bench.py's default configuration: fp32-grade projections, and cuDNN left at torch's
    # (and the reference's) default for the three library convolutions still on the path (patch embed, the CAB's 3x3 pair)
    torch.backends.cudnn.allow_tf32 = path == "fused_tf32x3_cudnn_tf32"
    g = golden(tag)
    model = _model(backbone, H, W, ncls)
    rgb = P.randn(SEED, tag + "/rgb", (1, 3, H, W)).cuda()
    mx = P.randn(SEED, tag + "/x", (1, 3, H, W)).cuda()
    with torch.no_grad(), M.composed_path(path == "composed"):
        logits = model(rgb, mx)
    assert tuple(logits.shape) == (1, ncls, H, W)
    if path == "composed":
        bar, agree, mtol = 1e-3, 0.999, 5e-4
    else:
        bar, agree, mtol = fused.logits_bar(), (0.995 if path == "fused_tf32" else 0.999), (2e-3 if path == "fused_tf32" else 5e-4)
    e, a = _check(logits, g, ncls, tag, bar, agree, mtol, H, W)
    record("fullsize_golden", tag=tag, path=path, precision=fused.precision(), logits_err_of_scale=e, labels_equal=a)
    # the encoder maps too (fused path returns NCHW views like the reference)
    with torch.no_grad(), M.composed_path(path == "composed"):
        feats = model.backbone(rgb, mx)
    fc, fs = (int(v) for v in g["feat_step"])
    for i, f in enumerate(feats):
        sub = f[:, ::fc, ::fs, ::fs].float().cpu().numpy()
        sc = float(g[f"feat{i}_absmax"])
        ferr = float(np.abs(sub - g[f"feat{i}_sub"]).max())
        assert ferr <= bar * sc * 2, f"{tag} {path}: encoder map {i} differs by {ferr / sc:.2e} of its scale"


@pytest.mark.parametrize("tf32", [False, True])
def test_fused_vs_oracle_port_480x640_b2(tf32):
    """Fresh seeded inputs and weights (not the fixture's), B = 2 at the benchmarked size: the CUDA path against the CPU
    oracle port (oracle/sigma_ref.py + the C selective scan) computed on this box's host cores (~3 s per image)."""
    from oracle import scan_oracle
    from sigma_b200 import fused
    scan_oracle.build()
    torch.backends.cuda.matmul.allow_tf32 = tf32
    torch.backends.cudnn.allow_tf32 = False
    H, W, ncls = 480, 640, 9
    model = _model("sigma_tiny", H, W, ncls, seed=SEED + 5)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    rgb = P.randn(SEED + 5, "o2/rgb", (2, 3, H, W))
    mx = P.randn(SEED + 5, "o2/x", (2, 3, H, W))
    with torch.no_grad():
        got = model(rgb.cuda(), mx.cuda()).cpu()
        ref = torch.cat([sigma_ref.encoder_decoder(rgb[i:i + 1], mx[i:i + 1], sd) for i in range(2)])
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max())
    agree = float((got.argmax(1) == ref.argmax(1)).float().mean())
    record("fullsize_oracle_b2", precision=fused.precision(), logits_err_of_scale=err / scale, labels_equal=agree)
    assert err <= fused.logits_bar() * scale, f"logits differ by {err:.3e} ({err / scale:.2e} of scale)"
    assert agree >= (0.995 if tf32 else 0.999)
