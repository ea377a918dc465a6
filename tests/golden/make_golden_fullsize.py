"""Goldens at the BENCHMARKED sizes from the UNMODIFIED reference (run in the build container; slow).

    python tests/golden/make_golden_fullsize.py tiny     # Sigma-tiny 480x640 B=1 (BASELINE config 2), ~4 min on 8 cores
    python tests/golden/make_golden_fullsize.py small    # Sigma-small 480x640 B=1, 40 classes (config 3 forward)
    python tests/golden/make_golden_fullsize.py base     # Sigma-base 720x960 B=1, 5 classes (config 5; odd 45->46->23 stage)

Same recipe as make_golden.py (reference classes through ref_shim, procedural weights / inputs); because a
full logits tensor is 11-14 MB and a fixture stays below 1 MB, it keeps: logits sub-sampled on a fixed pixel lattice
(all classes; every 8th pixel, every 16th for the 40 classes of small; `logits_step`), the FULL arg-max map (uint8),
the top-2 logit margin quantised to fp16 at the pixels where it is at most TIE of the logit scale (`tie_mask` packed
bits, `tie_margin`; so a test can tell a flipped label at a near-tie from a real error), the 4 encoder stage outputs
sub-sampled (`feat_step`), and hist/mIoU from the reference's own utils/metric.py.
"""
import os
import sys
import time
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [HERE, os.path.dirname(HERE)]
import procedural as P  # noqa: E402
import ref_shim  # noqa: E402

SEED = 7
CASES = {
    "tiny": ("sigma_tiny_480x640", "sigma_tiny", 480, 640, 9),
    "small": ("sigma_small_480x640", "sigma_small", 480, 640, 40),
    "base": ("sigma_base_720x960", "sigma_base", 720, 960, 5),
}
STEPS = {"tiny": (8, 3), "small": (16, 3), "base": (8, 6)}   # logits lattice step, encoder-map spatial step
TIE = 0.025                                                   # 2.5 x the largest logits bar of the tests (1e-2)


@torch.no_grad()
def main():
    torch.set_num_threads(8)
    ns = ref_shim.install()
    sys.path.insert(0, ref_shim.REF_ROOT)
    from utils.metric import hist_info, compute_score
    for which in sys.argv[1:]:
        tag, backbone, H, W, ncls = CASES[which]
        cfg = types.SimpleNamespace(backbone=backbone, decoder="MambaDecoder", num_classes=ncls,
                                    image_height=H, image_width=W, pretrained_model=None,
                                    bn_eps=1e-3, bn_momentum=0.1)
        model = ns.builder.EncoderDecoder(cfg, criterion=None, norm_layer=nn.BatchNorm2d)
        P.fill_state_dict(model, SEED)
        model.eval()
        ns.stub.calls.clear()
        rgb = P.randn(SEED, tag + "/rgb", (1, 3, H, W))
        mx = P.randn(SEED, tag + "/x", (1, 3, H, W))
        t0 = time.time()
        feats = model.backbone(rgb, mx)
        logits = model.decode_head.forward(feats)
        dec_shape = tuple(logits.shape)
        logits = torch.nn.functional.interpolate(logits, size=(H, W), mode="bilinear", align_corners=False)  # builder.py:136
        dt = time.time() - t0
        assert logits.shape == (1, ncls, H, W), logits.shape
        pred = logits.argmax(1)
        top2 = logits.topk(2, dim=1).values
        margin = (top2[:, 0] - top2[:, 1]).to(torch.float16)
        gt = (P.rand(SEED, tag + "/gt", (1, H, W)) * ncls).long().clamp(max=ncls - 1).numpy()
        hist, labeled, correct = hist_info(ncls, pred.numpy(), gt)
        iou, mean_iou, _, _, _, _ = compute_score(hist, correct, labeled)
        ls, fs = STEPS[which]
        tie = (margin.float() <= TIE * logits.abs().max()).reshape(-1).numpy()
        out = dict(logits_sub=logits[:, :, 3::ls, 5::ls].contiguous().numpy(), logits_step=np.asarray([3, 5, ls]),
                   argmax=pred.numpy().astype(np.uint8), tie_bound=np.float32(TIE), tie_mask=np.packbits(tie),
                   tie_margin=margin.reshape(-1).numpy()[tie], logits_absmax=np.float32(logits.abs().max()),
                   miou=np.float64(mean_iou), iou=np.asarray(iou), hist=np.asarray(hist),
                   ncalls=len(ns.stub.calls), dec_shape=np.asarray(dec_shape), ref_seconds=np.float64(dt))
        out["feat_step"] = np.asarray([4, fs])
        for i, f in enumerate(feats):
            out[f"feat{i}_sub"] = f[:, ::4, ::fs, ::fs].contiguous().numpy()
            out[f"feat{i}_absmax"] = np.float32(f.abs().max())
        np.savez_compressed(os.path.join(HERE, tag + ".npz"), **out)
        print(tag, "mIoU", mean_iou, "scan calls", len(ns.stub.calls), f"{dt:.0f} s",
              {k: getattr(v, "shape", None) for k, v in out.items()}, flush=True)


if __name__ == "__main__":
    main()
