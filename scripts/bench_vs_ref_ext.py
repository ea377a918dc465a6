"""Same box, same tensors: the reference CUDA extension rebuilt for sm_100a (oracle/_ref, recipe oracle/build_ref_ext.py)
next to sigma_b200's op-level kernels and the fused SS2D scan, on every a1 shape of SURVEY.md App. B.

    python scripts/bench_vs_ref_ext.py [--batch 1 8] [--dtypes f32 bf16] [--bwd] [--out gpurun_out/ref_ext_compare.json]

For each (shape, batch, dtype): parity of `sigma_scan_fwd` (and, with --bwd, `sigma_scan_bwd`) against the EXTENSION on
identical inputs (max abs error over the output scale), time of both (CUDA events, L2 flush between repetitions, median of
5), algorithmic GB/s by the SURVEY.md §8d formula.  The reference is timed with nrows=1 and, where the model uses it
(vmamba.py:183-191: nrows=4 when D % 4 == 0), nrows=4; the faster one is the baseline.  The fused scan is timed on the
channels-last formulation of the same problem (same algorithmic bytes) for the kinds that exist in the model.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle", "_ref")]
from sigma_b200 import _lib, fused, ops  # noqa: E402

# name, KD, L, N, K, (fused kind, H, W, D, R) or None
SHAPES = [
    ("enc0", 768, 19200, 16, 4, ("cross4", 120, 160, 192, 6)), ("enc1", 1536, 4800, 16, 4, ("cross4", 60, 80, 384, 12)),
    ("enc2", 3072, 1200, 16, 4, ("cross4", 30, 40, 768, 24)), ("enc3", 6144, 300, 16, 4, ("cross4", 15, 20, 1536, 48)),
    ("cromb0", 192, 19200, 4, 1, None), ("cromb1", 384, 4800, 4, 1, None), ("cromb2", 768, 1200, 4, 1, None),
    ("cromb3", 1536, 300, 4, 1, None),
    ("conmb0", 384, 38400, 4, 2, ("seq2", 120, 160, 192, 6)), ("conmb1", 768, 9600, 4, 2, ("seq2", 60, 80, 384, 12)),
    ("conmb2", 1536, 2400, 4, 2, ("seq2", 30, 40, 768, 24)), ("conmb3", 3072, 600, 4, 2, ("seq2", 15, 20, 1536, 48)),
    ("dec0", 768, 19200, 4, 4, ("cross4", 120, 160, 192, 6)), ("dec1", 1536, 4800, 4, 4, ("cross4", 60, 80, 384, 12)),
    ("dec2", 3072, 1200, 4, 4, ("cross4", 30, 40, 768, 24)),
]
KID = {"cross4": _lib.DIRS_CROSS4, "seq2": _lib.DIRS_SEQ2}
DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


def algo_bytes(B, KD, L, N, K, s):
    return s * (3 * B * KD * L + 2 * B * K * N * L) + 4 * (KD * N + 2 * KD)


def timeit(fn, flush, reps=5):
    fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[1, 8])
    ap.add_argument("--dtypes", nargs="+", default=["f32", "bf16"])
    ap.add_argument("--bwd", action="store_true")
    ap.add_argument("--only", nargs="*", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "ref_ext_compare.json"))
    a = ap.parse_args()
    import selective_scan_cuda_core as ref  # the reference extension, rebuilt for sm_100a
    peak = 6486.1
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rows = []
    g = torch.Generator(device="cuda").manual_seed(11)
    for B in a.batch:
        for name, KD, L, N, K, fz in SHAPES:
            if a.only and name not in a.only:
                continue
            for dn in a.dtypes:
                dt = DT[dn]
                s = 4 if dn == "f32" else 2
                u = torch.randn(B, KD, L, device="cuda", generator=g).to(dt)
                dl = (torch.randn(B, KD, L, device="cuda", generator=g) * 0.7).to(dt)     # pre-softplus dt_proj output scale
                A = -(torch.rand(KD, N, device="cuda", generator=g) * N + 0.3)
                Bm = torch.randn(B, K, N, L, device="cuda", generator=g).to(dt)
                Cm = torch.randn(B, K, N, L, device="cuda", generator=g).to(dt)
                D = torch.randn(KD, device="cuda", generator=g)
                bias = torch.rand(KD, device="cuda", generator=g) * 4 - 6                # softplus(bias) in [0.0025, 0.13]
                byt = algo_bytes(B, KD, L, N, K, s)
                row = dict(shape=name, batch=B, dtype=dn, KD=KD, L=L, N=N, K=K, algo_MB=round(byt / 1e6, 2))
                # ---- forward
                o_ref, x_ref = ref.fwd(u, dl, A, Bm, Cm, D, bias, True, 1)
                o_our, _ = ops.selective_scan_cuda_core_fwd(u, dl, A, Bm, Cm, D, bias, True, 1)
                scale = float(o_ref.float().abs().max())
                row["fwd_err_vs_ext"] = float((o_our.float() - o_ref.float()).abs().max()) / scale
                t_ref = {1: timeit(lambda: ref.fwd(u, dl, A, Bm, Cm, D, bias, True, 1), flush)}
                if (KD // K) % 4 == 0 and K > 1:
                    t_ref[4] = timeit(lambda: ref.fwd(u, dl, A, Bm, Cm, D, bias, True, 4), flush)
                t_our = timeit(lambda: ops.selective_scan_cuda_core_fwd(u, dl, A, Bm, Cm, D, bias, True, 1), flush)
                best = min(t_ref.values())
                row.update(ref_fwd_ms={str(k): round(v, 4) for k, v in t_ref.items()}, ref_fwd_GBps=round(byt / best / 1e6, 1),
                           our_fwd_ms=round(t_our, 4), our_fwd_GBps=round(byt / t_our / 1e6, 1),
                           our_fwd_frac=round(byt / t_our / 1e6 / peak, 4), fwd_speedup=round(best / t_our, 3))
                # ---- fused SS2D scan on the channels-last formulation of the same call (fp32 only)
                if fz is not None and dn == "f32":
                    kind, H, W, Dd, R = fz
                    Ls = 2 * H * W if kind == "seq2" else H * W
                    Cp = _lib.lib().sigma_ss2d_padded_cp(N, R)
                    xc = torch.randn(B, Ls, Dd, device="cuda", generator=g)
                    xdbl = torch.randn(B, Ls, K, Cp, device="cuda", generator=g)
                    dtw = (torch.rand(K, Dd, R, device="cuda", generator=g) * 2 - 1) * R ** -0.5
                    dtb = torch.rand(K, Dd, device="cuda", generator=g) * 4 - 6
                    Af = -(torch.rand(K * Dd, N, device="cuda", generator=g) * N + 0.3)
                    Dsf = torch.randn(K * Dd, device="cuda", generator=g)
                    t_f = timeit(lambda: fused.ss2d_scan(KID[kind], xc, xdbl, dtw, dtb, Af, Dsf, B, H, W, Dd, N, R, Cp), flush)
                    row.update(fused_ms=round(t_f, 4), fused_GBps=round(byt / t_f / 1e6, 1), fused_speedup=round(best / t_f, 3))
                    del xc, xdbl
                # ---- backward
                if a.bwd:
                    dout = torch.randn(B, KD, L, device="cuda", generator=g).to(dt)
                    try:
                        r = ref.bwd(u, dl, A, Bm, Cm, D, bias, dout, x_ref, True, 1)
                        o = ops.selective_scan_cuda_core_bwd(u, dl, A, Bm, Cm, D, bias, dout, None, True, 1)
                        errs = {}
                        for nm, tr, to in zip(("du", "ddelta", "dA", "dB", "dC", "dD", "dbias"), r, o):
                            sc = float(tr.float().abs().max()) + 1e-20
                            errs[nm] = float((tr.float() - to.float()).abs().max()) / sc
                        row["bwd_err_vs_ext"] = {k: float(f"{v:.3e}") for k, v in errs.items()}
                        tb_ref = timeit(lambda: ref.bwd(u, dl, A, Bm, Cm, D, bias, dout, x_ref, True, 1), flush, reps=3)
                        tb_our = timeit(lambda: ops.selective_scan_cuda_core_bwd(u, dl, A, Bm, Cm, D, bias, dout, None, True, 1), flush, reps=3)
                        row.update(ref_bwd_ms=round(tb_ref, 4), our_bwd_ms=round(tb_our, 4), bwd_speedup=round(tb_ref / tb_our, 3))
                    except Exception as e:  # report, keep going
                        row["bwd_error"] = f"{type(e).__name__}: {e}"[:300]
                    del dout
                rows.append(row)
                print(json.dumps(row), flush=True)
                del u, dl, Bm, Cm
                torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    json.dump(dict(peak_GBps=peak, gpu=torch.cuda.get_device_name(0), rows=rows), open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
