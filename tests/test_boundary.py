"""CPU: the drop-in boundary.  The C-ABI library loads without a GPU or libcuda, exports every symbol that
include/sigma_b200.h declares, the ctypes binding declares the same set, and the reference's import paths resolve to
our modules.  No compute calls (there is no GPU here)."""
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib_path():
    from sigma_b200 import build
    return build.build()


def _declared():
    src = open(os.path.join(ROOT, "include", "sigma_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return set(re.findall(r"\b(sigma_[a-z0-9_]+)\s*\(", src))


def test_library_exports_every_declared_symbol(lib_path):
    out = subprocess.run(["nm", "-D", "--defined-only", lib_path], capture_output=True, text=True, check=True).stdout
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    declared = _declared()
    assert declared, "no declarations parsed"
    assert declared <= exported, f"declared but not exported: {sorted(declared - exported)}"
    extra = {s for s in exported - declared if s.startswith("sigma_")}
    assert extra <= {"sigma_scan_fwd_f32_split", "sigma_scan_bwd_split", "sigma_ss2d_scan_fwd_split", "sigma_ss2d_scan_bwd_split",
                     "sigma_test_pick_segments", "sigma_test_pick_bn"}, f"undeclared exports: {sorted(extra)}"


def test_library_has_no_runtime_dependency_on_cuda_libs(lib_path):
    out = subprocess.run(["ldd", lib_path], capture_output=True, text=True, check=True).stdout
    assert "libcuda" not in out and "libcudart" not in out and "libtorch" not in out, out


def test_ctypes_binding_matches_header(lib_path):
    from sigma_b200 import _lib
    L = _lib.lib()
    n0 = L.sigma_launch_count()        # GPU tests earlier in this process may have launched kernels
    assert L.sigma_abi_version() == 1
    assert set(_lib.SIGNATURES) >= _declared()
    assert L.sigma_ss2d_padded_cp(16, 6) == 40 and L.sigma_ss2d_padded_cp(4, 24) == 32 and L.sigma_ss2d_padded_cp(4, 65) == -1
    assert L.sigma_scan_fwd_workspace_bytes(2, 768, 1024, 16, 4, 0) > 0
    assert L.sigma_launch_count() == n0
    # a freshly loaded library has launched nothing
    r = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); from sigma_b200 import _lib; print(_lib.launch_count())" % ROOT],
                       capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.split() == ["0"], r.stdout + r.stderr


def test_sm100a_tma_in_sass(lib_path):
    """the fused scan really is a TMA kernel (UTMALDG) compiled for sm_100a."""
    out = subprocess.run(["cuobjdump", "-lelf", lib_path], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run(["cuobjdump", "-sass", os.path.join(ROOT, "sigma_b200", "build", "ss2d_scan_rp8.o")],
                          capture_output=True, text=True).stdout
    assert "UTMALDG" in sass and "SYNCS" in sass and "MUFU.EX2" in sass


def test_dropin_import_paths_resolve():
    code = ("import sys; sys.path[:0] = [%r, %r];"
            "import selective_scan_cuda_core as c, selective_scan as s;"
            "from models.builder import EncoderDecoder;"
            "from models.encoders.vmamba import SS2D, VSSBlock, ConMB_SS2D, CrossScan, SelectiveScan, Backbone_VSSM;"
            "from models.encoders.dual_vmamba import vssm_tiny, vssm_small, vssm_base;"
            "from models.decoders.MambaDecoder import MambaDecoder;"
            "import sigma_b200.modules as M;"
            "assert EncoderDecoder is M.EncoderDecoder and SS2D is M.SS2D and callable(c.fwd) and callable(c.bwd);"
            "assert callable(s.selective_scan_fn) and callable(s.selective_scan_ref); print('ok')") % (
        ROOT, os.path.join(ROOT, "sigma_b200", "dropin"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr


def test_no_cpu_fallback():
    """product modules refuse CPU tensors instead of silently computing on the host."""
    import torch
    from sigma_b200 import modules as M, ops
    with pytest.raises(RuntimeError):
        ops.selective_scan_cuda_core_fwd(torch.zeros(1, 4, 8), torch.zeros(1, 4, 8), torch.zeros(4, 4),
                                         torch.zeros(1, 1, 4, 8), torch.zeros(1, 1, 4, 8), None, None, False, 1)
    blk = M.VSSBlock(hidden_dim=16, mlp_ratio=0.0, d_state=4)
    with pytest.raises(RuntimeError), torch.no_grad():
        blk(torch.zeros(1, 4, 4, 16))


def test_dropin_selective_scan_ref_matches_oracle():
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "sigma_b200", "dropin"))
    try:
        import selective_scan as s
    finally:
        sys.path.pop(0)
    import procedural as P
    from oracle import scan_oracle
    u, dl, A, Bm, Cm, D, bias = P.scan_inputs(3, 2, 8, 4, 40, 2)
    got = s.selective_scan_ref(u, dl, A, Bm, Cm, D, bias, True)
    ref = scan_oracle.scan_fwd(u.numpy(), dl.numpy(), A.numpy(), Bm.numpy(), Cm.numpy(), D.numpy(), bias.numpy(), True)
    assert np.abs(got.numpy() - ref).max() < 1e-4
