"""CPU-side checks: the C-ABI library loads and exports exactly what include/morfem_b200.h declares, argument
validation answers without touching a GPU, and the host-side helpers mirror the reference's behaviour."""
import ctypes
import math
import os
import re
import subprocess
import sys
import textwrap
import warnings

import numpy as np
import pytest
from scipy.sparse import csc_array

from morfem_b200 import _ffi, implementation as impl, test_helpers as th, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    text = open(os.path.join(ROOT, "include", "morfem_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mf_[a-z0-9_]+)\s*\(", text)))


def test_header_library_and_binding_agree():
    names = header_functions()
    assert len(names) >= 20
    assert sorted(_ffi.SIGNATURES) == names
    lib = _ffi.load()
    for n in names:
        assert hasattr(lib, n), n
    assert lib.mf_version() == 100


def test_argument_validation_without_gpu():
    lib = _ffi.load()
    # NULL operands: every entry point must answer with -(argument index) and a message, never crash
    st = lib.mf_gemm_tn_c128(None, 4, 4, None, 4, 4, 10, 0, None, 4, None, 0, None)
    assert st == -1 and b"mf_gemm_tn_c128" in lib.mf_last_error()
    st = lib.mf_spmm_csr_c128(None, None, None, 1, 10, None, 4, 4, None, 4, None)
    assert st == -1
    st = lib.mf_sweep_lu_gsm_c128(None, None, None, 8, None, 2, 8, 2, None, None, None, None, None, 4, None, None, None, 0,
                                  None, 0, None)
    assert st == -1
    with pytest.raises(_ffi.MorfemB200Error):
        _ffi.check(st, "mf_sweep_lu_gsm_c128")
    assert lib.mf_gemm_tn_ws_bytes(64, 64, 100000) >= 64 * 64 * 16
    assert lib.mf_jacobi_svd_ws_bytes(64) > 2 * 64 * 64 * 16
    # the real float64 twins and the row-grouped SpMM entries validate the same way
    assert lib.mf_gemm_tn_f64(None, 4, 4, None, 4, 4, 10, None, 4, None, 0, None) == -1 and b"mf_gemm_tn_f64" in lib.mf_last_error()
    assert lib.mf_gemm_nn_f64(None, 4, 10, 4, None, 4, 4, None, 4, None) == -1
    assert lib.mf_trmm_nn_f64(None, 4, 10, 4, None, 4, None, 4, None) == -1
    assert lib.mf_trmm_nn_c128(None, 4, 10, 4, None, 4, None, 4, None) == -1
    assert lib.mf_chol_inv_upper_c128(None, 4, 4, None, 4, None, None, 0, None) == -1
    assert lib.mf_chol_inv_ws_bytes(256) >= 128
    assert lib.mf_spmm_csr2_c128(None, None, None, None, 1, 10, None, 4, 4, None, 4, None, 4, None) == -1
    assert lib.mf_spmm_csr2_f64(None, None, None, None, 10, None, 4, 4, None, 4, None, 4, None) == -1
    assert lib.mf_spmm_csr_f64(None, None, None, 10, None, 4, 4, None, 4, None) == -1
    assert lib.mf_spmm_group_count(None, None, 10, 4, None, None) == -1
    assert lib.mf_spmm_grouped_c128(None, None, None, 10, 4, None, 4, 4, None, 4, None) == -1
    assert lib.mf_sweep_lu_gsm_f64(None, None, None, 8, None, 2, 8, 2, None, None, None, None, None, 4, None, None, None, 0, None, 0, None) == -1
    assert lib.mf_jacobi_svd_f64(None, 4, 4, None, 4, None, 10, 1e-15, None, None) == -1
    assert lib.mf_gemm_tn_f64_ws_bytes(64, 64, 100000) >= 64 * 64 * 8
    # shape support queries (host only): which kernel family serves which (r, m)
    assert lib.mf_spmm_group_size(64) == 4 and lib.mf_spmm_group_size(256) == 2 and lib.mf_spmm_group_size_f64(256) == 4
    assert lib.mf_sweep_f64_supported(64, 2) == 1 and lib.mf_sweep_f64_supported(256, 4) == 1 and lib.mf_sweep_f64_supported(513, 4) == 0
    assert lib.mf_sweep_f64_variant_supported(256, 4, 3) == 0 and lib.mf_sweep_f64_variant_supported(256, 4, 5) == 1
    assert lib.mf_sweep_f64_ws_bytes(64, 2, 1000, 0) == 256 and lib.mf_sweep_f64_ws_bytes(256, 4, 1000, 0) >= 148 * 2 * 256 * 256 * 8
    assert lib.mf_sweep_variant_supported(256, 4, 4) == 1 and lib.mf_sweep_variant_supported(64, 2, 4) == 0 and lib.mf_sweep_variant_supported(64, 2, 5) == 1
    assert lib.mf_jacobi_svd_f64_supported(64) == 1 and lib.mf_jacobi_svd_f64_supported(65) == 0
    assert all(lib.mf_sweep_variant_supported(r, 4, 3) == 1 for r in (1, 64, 112, 113, 256, 512))
    assert lib.mf_sweep_variant_supported(600, 4, 3) == 0 and lib.mf_sweep_variant_supported(600, 4, 1) == 1
    assert lib.mf_sweep_ws_bytes(256, 4, 1000, 0) >= 148 * 2 * 256 * 256 * 16 and lib.mf_sweep_ws_bytes(64, 2, 1000, 0) == 256
    assert lib.mf_sweep_ws_bytes(256, 4, 1000, 4) >= 148 * 256 * 264 * 16


def test_product_path_refuses_to_run_without_cuda():
    """No CPU fallback on the hot path.  Runs in a child process with every GPU hidden, so that it checks the same thing on a
    machine that has one."""
    script = textwrap.dedent("""
        import numpy as np, torch
        from morfem_b200 import _ffi, implementation as impl, test_helpers as th, synthetic
        assert not torch.cuda.is_available()
        a0, a1, a2, b = synthetic.reduced_model(8, 2, seed=0)
        md = impl.ModelDefinition(np.linspace(3e9, 5e9, 4), a0, a1, a2, b, lambda t: 1.0, lambda t: t, lambda t: t ** 2, th.b_coefficient)
        try:
            impl.solve_finite_element_method(md)
        except _ffi.MorfemB200Error:
            raise SystemExit(0)
        raise SystemExit("solve_finite_element_method returned without a CUDA device")
    """)
    out = subprocess.run([sys.executable, "-c", script], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]


def test_b_coefficient_scalar_and_array_forms_agree():
    """test_helpers.py:70-72: scalar form identical to the reference's formula (math.sqrt, ValueError below cutoff); the array
    form agrees to 1 ulp and raises for a point below the cutoff like the scalar loop would."""
    import math
    from scipy.constants import pi, c
    f = np.linspace(3e9, 5e9, 2001)
    ref = np.array([math.sqrt(math.sqrt(((2 * pi * t) / c) ** 2 - 54.5976295582387 ** 2) / t) for t in f])
    assert np.array_equal(np.array([th.b_coefficient(float(t)) for t in f]), ref)
    vec = th.b_coefficient(f)
    assert np.max(np.abs(vec - ref) / ref) <= 2 * np.finfo(float).eps
    assert np.max(np.abs(impl.coefficient_array(th.b_coefficient, f) - ref) / ref) <= 2 * np.finfo(float).eps
    with pytest.raises(ValueError):
        th.b_coefficient(1e9)
    with pytest.raises(ValueError):
        th.b_coefficient(np.array([4e9, 1e9]))
    with pytest.raises(ValueError):
        impl.coefficient_array(th.b_coefficient, np.array([4e9, 1e9]))


def test_coefficient_array_vectorised_and_scalar_fallback():
    dom = np.linspace(3e9, 5e9, 17)
    assert np.array_equal(impl.coefficient_array(lambda t: t ** 2, dom), dom ** 2)
    assert np.array_equal(impl.coefficient_array(lambda t: 1.0, dom), np.ones(17))
    cb = impl.coefficient_array(th.b_coefficient, dom)            # math.sqrt: scalar-only callable
    assert np.array_equal(cb, np.array([th.b_coefficient(t) for t in dom]))
    with pytest.raises(ValueError):
        impl.coefficient_array(th.b_coefficient, np.array([1e9, 3e9]))   # below cutoff: the reference's ValueError
    # a callable whose vectorised form is *different* from its scalar form must fall back to scalar evaluation
    odd = lambda t: float(np.sum(t))  # noqa: E731
    assert np.array_equal(impl.coefficient_array(odd, dom), dom)


def test_host_helpers_match_reference_semantics():
    rng = np.random.default_rng(0)
    a = rng.standard_normal((5, 5))
    md = impl.ModelDefinition(np.array([2.0]), a, 2 * a, 3 * a, rng.standard_normal((5, 2)), lambda t: 1.0, lambda t: t,
                              lambda t: t ** 2, lambda t: t)
    s = impl.system_matrix(2.0, md)
    full = a + 2.0 * 2 * a + 4.0 * 3 * a
    assert np.allclose(s, (full + full.T) / 2)
    assert np.allclose(impl.impulse_vector(2.0, md), 2.0 * md.b)
    with pytest.raises(Exception):
        impl.h(np.zeros(3))
    z = rng.standard_normal((3, 2)) + 1j * rng.standard_normal((3, 2))
    assert np.array_equal(impl.h(z), z.conj().T)
    assert th.b_coefficient(4e9) == math.sqrt(math.sqrt(((2 * math.pi * 4e9) / 299792458.0) ** 2 - 54.5976295582387 ** 2) / 4e9)
    pts = th.equally_distributed_points(np.arange(10), 4)
    assert list(pts) == [0, 3, 6, 9]
    with pytest.raises(Exception):
        th.equally_distributed_points(np.arange(3), 4)


def test_full_order_branch_stays_on_scipy():
    """solve_fem_point on sparse operators is the SuperLU call of implementation.py:475 (outside the hot path)."""
    ct, tt = synthetic.waveguide_operators(3, 2, 6)
    wp = synthetic.port_matrix(ct.shape[0], 2, 5)
    in_c, in_gamma, in_b = synthetic.driver_scaled(ct, tt, wp)
    md = impl.ModelDefinition(np.array([4e9]), in_c, csc_array(in_c.shape), in_gamma, in_b, lambda t: 1.0, lambda t: t,
                              lambda t: t ** 2, th.b_coefficient)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        x = impl.solve_fem_point(4e9, md)
    a = in_c + (4e9) ** 2 * in_gamma
    assert np.allclose(a @ x, th.b_coefficient(4e9) * in_b.toarray(), atol=1e-9 * np.abs(in_b.toarray()).max())


def test_streamed_sweep_geometry_from_workspace_sizes(monkeypatch):
    """The streamed sweep (113 <= r <= 512) sizes its workspace as one R x LD complex slot per resident CTA: three CTAs per SM
    up to r = 128, two up to r = 256, one above (148 SMs assumed when no device is visible); MF_STREAM_CFG=0 forces one."""
    from morfem_b200 import _ffi
    lib = _ffi.load()
    monkeypatch.delenv("MF_STREAM_CFG", raising=False)
    slot = lambda r, m: 16 * ((r + 31) // 32 * 32) * ((r + 31) // 32 * 32 + (m + 7) // 8 * 8)
    big = 10 ** 6
    per_sm = {(113, 1): 3, (128, 4): 3, (129, 4): 2, (256, 4): 2, (257, 4): 1, (512, 8): 1}
    sms = lib.mf_sweep_ws_bytes(512, 8, big, 4) // slot(512, 8)
    assert sms >= 1
    for (r, m), ctas in per_sm.items():
        assert lib.mf_sweep_ws_bytes(r, m, big, 4) == ctas * sms * slot(r, m), (r, m)
        assert lib.mf_sweep_ws_bytes(r, m, 10, 4) == 10 * slot(r, m)          # never more slots than points
    monkeypatch.setenv("MF_STREAM_CFG", "0")
    assert lib.mf_sweep_ws_bytes(256, 4, big, 4) == sms * slot(256, 4)
    assert lib.mf_sweep_ws_bytes(64, 2, big, 3) <= 256                         # r <= 64: matrix lives in shared memory
    assert lib.mf_sweep_ws_bytes(80, 2, 10, 3) == 10 * 16 * (2 * 80 * 80 + 32 * 80)     # above: the left-looking kernel's slots


def test_left_looking_sweep_workspace_sizes():
    """The left-looking sweep (variant 5; what variant 3 runs above r = 112) keeps, per resident CTA, the multiplier panels
    (R x R, indexed by original row), the U blocks (R x R, fragment order) and the inverted 16 x 16 diagonal blocks of L and U
    (2 x 16 R), R = r rounded up to 16; float64 slots are half the size of complex128 ones."""
    from morfem_b200 import _ffi
    lib = _ffi.load()
    slot = lambda r: ((r + 15) // 16 * 16) ** 2 * 2 + 32 * ((r + 15) // 16 * 16)
    for r, m in ((113, 1), (160, 4), (256, 4), (300, 2), (512, 8)):
        assert lib.mf_sweep_ws_bytes(r, m, 10, 5) == 10 * 16 * slot(r)
        assert lib.mf_sweep_ws_bytes(r, m, 10, 3) == 10 * 16 * slot(r)
        assert lib.mf_sweep_f64_ws_bytes(r, m, 10, 0) == 10 * 8 * slot(r)                          # float64: left-looking kernel from r = 73
        assert lib.mf_sweep_f64_ws_bytes(r, m, 10, 5) == 10 * 8 * slot(r)
    assert lib.mf_sweep_ws_bytes(64, 2, 10, 5) == 10 * 16 * slot(64) and lib.mf_sweep_f64_ws_bytes(64, 2, 10, 5) == 10 * 8 * slot(64)


def test_reference_host_helpers_of_the_opm_mode():
    """orthonormalize_to_base / orthonormalize_vector_to_base / expand_matrix / OfflinePhaseMatrices / TimeStatistics
    (implementation.py:57-96, :455-523) keep their names and semantics (host helpers, outside the hot path)."""
    rng = np.random.default_rng(3)
    base = np.linalg.qr(rng.standard_normal((40, 5)))[0]
    v = rng.standard_normal((40, 3))
    one = impl.orthonormalize_vector_to_base(v[:, 0], base)
    ref = v[:, 0] - sum(base[:, i] * np.inner(v[:, 0], base[:, i]) for i in range(5))        # implementation.py:517-521
    assert np.allclose(one, ref / np.linalg.norm(ref), rtol=0, atol=1e-15)
    new = impl.orthonormalize_to_base(v, base)
    assert new.shape == (40, 3) and np.abs(base.T @ new).max() < 1e-14 and np.abs(new.T @ new - np.eye(3)).max() < 1e-14
    mid = rng.standard_normal((40, 40))
    full = np.hstack((base, new))
    assert np.allclose(impl.expand_matrix(base.T @ mid @ base, base, mid, new), full.T @ mid @ full, rtol=0, atol=1e-13)
    with pytest.raises(Exception):
        impl.orthonormalize_to_base(v[:, 0], base)
    with pytest.raises(Exception):
        impl.orthonormalize_vector_to_base(v, base)
    assert impl.OfflinePhaseMatrices().bh_b is None
    ts = impl.TimeStatistics()
    ts.start_clock(); ts.add_time("Offline"); ts.add_custom_time("Whole", ts.clock)
    assert "Offline" in impl.TimeStatistics.times                 # class-level dict, shared like the reference's (implementation.py:77)
