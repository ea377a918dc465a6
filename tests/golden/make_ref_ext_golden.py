"""Golden outputs of the UNMODIFIED reference CUDA extension for tests/test_ref_ext_gpu.py (run once on a B200).

    SIGMA_REFERENCE_DIR=<checkout of the original Sigma project> python oracle/build_ref_ext.py   # -> oracle/_ref/
    python tests/golden/make_ref_ext_golden.py [OUT.npz]                                         # default tests/golden/ref_ext.npz

Inputs are the test's own seeded tensors (tests/procedural.py), so only the extension's OUTPUTS are stored, summarized
per tensor by test_ref_ext_gpu.summarize (shape, dtype, largest and mean |value|, a fixed seeded element sample).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE), os.path.join(ROOT, "oracle", "_ref")]
import selective_scan_cuda_core as ext  # noqa: E402
import test_ref_ext_gpu as T  # noqa: E402


@torch.no_grad()
def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_ext.npz")
    out = {}
    for dn, dt in T.DTYPES.items():
        for i, (b, d, n, L, g) in enumerate(T.SHAPES):
            u, dl, A, Bm, Cm, D, bias = T._inputs(b, d, n, L, g, dt)
            o, x = ext.fwd(u, dl, A, Bm, Cm, D, bias, True, 1)
            tag = T.fwd_tag(b, d, n, L, g, dn)
            out.update(T.summarize(tag + "/out", o, T.K_OUT))
            out.update(T.summarize(tag + "/x", x, T.K_GRAD))
            out[tag + "/x|ystate_absmax"] = np.float32(float(x[..., 1::2].abs().max()))
            if i < 8:
                grads = ext.bwd(u, dl, A, Bm, Cm, D, bias, T._dout(b, d, L, dt), x, True, 1)
                for nm, r in zip(T.GRADS, grads):
                    out.update(T.summarize(f"{T.bwd_tag(b, d, n, L, g, dn)}/{nm}", r, T.K_GRAD))
    for case in T.FUSED:
        tag, ref = T.extension_fused_reference(ext, *case)
        out.update(T.summarize(tag, ref, T.K_OUT))
    np.savez_compressed(out_path, **out)
    print(out_path, len(out), "arrays", os.path.getsize(out_path), "bytes")


if __name__ == "__main__":
    main()
