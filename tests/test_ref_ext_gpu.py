"""GPU: parity against the reference CUDA EXTENSION itself (selective_scan_cuda_core rebuilt for sm_100a by
oracle/build_ref_ext.py, BASELINE.json north_star: "outputs match the reference selective_scan extension on identical
inputs within 1e-3 fp32 / 1e-2 bf16").  The extension's outputs on these seeded inputs are stored in
tests/golden/ref_ext.npz (tests/golden/make_ref_ext_golden.py, run once on a B200): for every output tensor its shape,
dtype, largest |value|, mean |value| and a fixed seeded sample of its elements.  The extension is built with
--use_fast_math (setup.py:94); errors are measured against the output scale."""
import numpy as np
import pytest
import torch

import procedural as P
from helpers import golden
from test_ss2d_scan_gpu import _dir_index

pytestmark = pytest.mark.gpu
S = 41
K_OUT, K_GRAD = 512, 256     # sampled elements stored per output / per gradient or chunk-state tensor


def sample_index(tag, n, k):
    """k flat element indices of an n-element tensor, a pure function of the tag (numpy PCG64, as tests/procedural.py)."""
    return np.sort((P._rng(S, tag + "/sample").random(k) * n).astype(np.int64))


def summarize(tag, t, k):
    """What tests/golden/ref_ext.npz keeps of one output tensor `t` under the key prefix `tag`."""
    f = t.detach().float().reshape(-1)
    idx = torch.from_numpy(sample_index(tag, f.numel(), k)).to(f.device)
    return {tag + "|shape": np.asarray(t.shape, np.int64), tag + "|dtype": np.asarray(str(t.dtype)),
            tag + "|absmax": np.float32(float(f.abs().max())), tag + "|meanabs": np.float64(float(f.abs().double().mean())),
            tag + "|idx_sample": f[idx].cpu().numpy()}


def compare(G, tag, got, k, bar, what):
    """Relative error of `got` against the stored extension output: on the sampled elements and on the tensor-wide
    largest and mean |value|, all against the extension's largest |value|.  Returns the sampled error."""
    assert tuple(got.shape) == tuple(G[tag + "|shape"]) and str(got.dtype) == str(G[tag + "|dtype"]), what
    f = got.detach().float().reshape(-1)
    scale = float(G[tag + "|absmax"]) + 1e-20
    idx = torch.from_numpy(sample_index(tag, f.numel(), k)).to(f.device)
    err = float(np.abs(f[idx].cpu().numpy() - G[tag + "|idx_sample"]).max()) / scale
    assert err <= bar, f"{what}: {err:.3e} of the extension's output scale"
    assert abs(float(f.abs().max()) - scale) / scale <= bar, f"{what}: largest |value| {float(f.abs().max()):.6e} vs {scale:.6e}"
    assert abs(float(f.abs().double().mean()) - float(G[tag + "|meanabs"])) / scale <= bar, f"{what}: mean |value|"
    return err


@pytest.fixture(scope="module")
def G():
    return golden("ref_ext")


def _inputs(b, d, n, L, g, dt):
    tag = f"ext/{b}/{d}/{n}/{L}/{g}"
    u = P.randn(S, tag + "/u", (b, d, L)).to(dt).cuda()
    dl = P.randn(S, tag + "/dl", (b, d, L), 0.7).to(dt).cuda()
    A = (-P.rand(S, tag + "/A", (d, n), 0.3, n + 0.5)).cuda()
    Bm = P.randn(S, tag + "/B", (b, g, n, L)).to(dt).cuda()
    Cm = P.randn(S, tag + "/C", (b, g, n, L)).to(dt).cuda()
    D = P.randn(S, tag + "/D", (d,)).cuda()
    bias = P.rand(S, tag + "/bias", (d,), -6.0, -2.0).cuda()
    return u, dl, A, Bm, Cm, D, bias


def _dout(b, d, L, dt):
    return P.randn(S, f"ext/dout/{b}/{d}/{L}", (b, d, L)).to(dt).cuda()


SHAPES = [  # b, d, n, L, g: Sigma shapes (App. B) and ragged ones
    (2, 3072, 16, 1200, 4), (1, 768, 16, 4800, 4), (2, 6144, 16, 300, 4), (2, 768, 4, 1200, 1), (1, 384, 4, 9600, 2),
    (2, 3072, 4, 1200, 4), (2, 24, 8, 372, 2), (1, 40, 16, 2077, 1), (3, 36, 4, 4100, 3), (1, 8192, 16, 690, 4),
]
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
GRADS = ("du", "ddelta", "dA", "dB", "dC", "dD", "dbias")
FUSED = [("cross4", 2, 30, 40, 768, 16, 24), ("cross4", 1, 60, 80, 384, 4, 12), ("seq2", 1, 30, 40, 768, 4, 24),
         ("cross4", 1, 23, 30, 256, 16, 16)]


def fwd_tag(b, d, n, L, g, dn):
    return f"fwd/{b}/{d}/{n}/{L}/{g}/{dn}"


def bwd_tag(b, d, n, L, g, dn):
    return f"bwd/{b}/{d}/{n}/{L}/{g}/{dn}"


@pytest.mark.parametrize("b,d,n,L,g", SHAPES)
@pytest.mark.parametrize("dn", ["f32", "bf16", "f16"])
def test_fwd_matches_extension(G, b, d, n, L, g, dn):
    from sigma_b200 import ops
    u, dl, A, Bm, Cm, D, bias = _inputs(b, d, n, L, g, DTYPES[dn])
    got, xg = ops.selective_scan_cuda_core_fwd(u, dl, A, Bm, Cm, D, bias, True, 1)
    tag = fwd_tag(b, d, n, L, g, dn)
    compare(G, tag + "/out", got, K_OUT, 1e-3 if dn == "f32" else 1e-2, f"fwd vs extension ({dn})")
    assert tuple(xg.shape) == tuple(G[tag + "/x|shape"])
    if dn == "f32":   # chunk-end states (only .y = h is consumed, selective_scan_bwd_kernel.cuh:114-116); running prefix in .x
        xf = xg.reshape(-1)
        idx = sample_index(tag + "/x", xf.numel(), K_GRAD)
        got_s, ref_s = xf[torch.from_numpy(idx).to(xf.device)].cpu().numpy(), G[tag + "/x|idx_sample"]
        odd = idx % 2 == 1                        # the last dimension interleaves (.x, .y)
        xs = float(G[tag + "/x|ystate_absmax"]) + 1e-20
        assert float(np.abs(got_s[odd] - ref_s[odd]).max()) / xs <= 1e-3
        assert abs(float(xg[..., 1::2].abs().max()) - xs) / xs <= 1e-3
        assert float(np.abs(got_s[~odd] - ref_s[~odd]).max()) <= 1e-3, "running-prefix component of x"


@pytest.mark.parametrize("b,d,n,L,g", SHAPES[:8])
@pytest.mark.parametrize("dn", ["f32", "bf16", "f16"])
def test_bwd_matches_extension(G, b, d, n, L, g, dn):
    from sigma_b200 import ops
    u, dl, A, Bm, Cm, D, bias = _inputs(b, d, n, L, g, DTYPES[dn])
    got = ops.selective_scan_cuda_core_bwd(u, dl, A, Bm, Cm, D, bias, _dout(b, d, L, DTYPES[dn]), None, True, 1)
    bar = 2e-3 if dn == "f32" else 2e-2   # fast-math reference, atomics in a different order
    for nm, o in zip(GRADS, got):
        compare(G, f"{bwd_tag(b, d, n, L, g, dn)}/{nm}", o, K_GRAD, bar, f"{nm} vs extension ({dn})")


def fused_inputs(kind, B, H, W, D, N, R):
    from sigma_b200 import _lib
    L = H * W
    K = 4 if kind == "cross4" else 2
    Ls = 2 * L if kind == "seq2" else L
    Cp = _lib.lib().sigma_ss2d_padded_cp(N, R)
    tag = f"extf/{kind}/{B}/{H}/{W}/{D}/{N}/{R}"
    xc = P.randn(S, tag + "/xc", (B, Ls, D)).cuda()
    xdbl = P.randn(S, tag + "/xdbl", (B, Ls, K, Cp))
    xdbl[..., 2 * N + R:] = 0.0
    xdbl = xdbl.cuda()
    dtw = P.rand(S, tag + "/dtw", (K, D, R), -R ** -0.5, R ** -0.5).cuda()
    dtb = P.rand(S, tag + "/dtb", (K, D), -6.0, -1.0).cuda()
    A = (-P.rand(S, tag + "/A", (K * D, N), 0.3, N + 0.5)).cuda()
    Ds = P.randn(S, tag + "/Ds", (K * D,)).cuda()
    return tag, K, Ls, Cp, xc, xdbl, dtw, dtb, A, Ds


@pytest.mark.parametrize("kind,B,H,W,D,N,R", FUSED)
def test_fused_scan_matches_extension(G, kind, B, H, W, D, N, R):
    """The fused channels-last scan against CrossScan + dt einsum (fp32) + the EXTENSION + un-flip, on the device."""
    from sigma_b200 import _lib, fused
    torch.backends.cuda.matmul.allow_tf32 = False
    tag, K, Ls, Cp, xc, xdbl, dtw, dtb, A, Ds = fused_inputs(kind, B, H, W, D, N, R)
    kid = {"cross4": _lib.DIRS_CROSS4, "seq2": _lib.DIRS_SEQ2}[kind]
    y = fused.ss2d_scan(kid, xc, xdbl, dtw, dtb, A, Ds, B, H, W, D, N, R, Cp)
    compare(G, tag, y, K_OUT, 1e-3, "fused scan vs extension")


def extension_fused_reference(ext, kind, B, H, W, D, N, R):
    """What test_fused_scan_matches_extension compares with: the reference's composition around the extension."""
    torch.backends.cuda.matmul.allow_tf32 = False
    tag, K, Ls, Cp, xc, xdbl, dtw, dtb, A, Ds = fused_inputs(kind, B, H, W, D, N, R)
    idx = [torch.from_numpy(ix.copy()).cuda() for ix in _dir_index(kind, H, W)]
    us = torch.cat([xc[:, ix].transpose(1, 2) for ix in idx], 1).contiguous()
    dts = torch.cat([torch.einsum("blr,dr->bdl", xdbl[:, ix, k, 2 * N:2 * N + R], dtw[k]) for k, ix in enumerate(idx)], 1).contiguous()
    Bs = torch.stack([xdbl[:, ix, k, 0:N].transpose(1, 2) for k, ix in enumerate(idx)], 1).contiguous()
    Cs = torch.stack([xdbl[:, ix, k, N:2 * N].transpose(1, 2) for k, ix in enumerate(idx)], 1).contiguous()
    o, _ = ext.fwd(us, dts, A, Bs, Cs, Ds, dtb.reshape(-1).contiguous(), True, 1)
    ref = torch.zeros((K, B, Ls, D), device="cuda")
    for k, ix in enumerate(idx):
        ref[k][:, ix] = o[:, k * D:(k + 1) * D].transpose(1, 2)
    return tag, ref
