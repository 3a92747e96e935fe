"""The complex128 DMMA contractions (gemm_tn, gemm_nn, trmm) form each complex block product in Gauss's three-multiplication
form (cmma3 in csrc/common.cuh).  3M is normwise stable but not componentwise: with |Im| >> |Re| (or the reverse) the small part
of a product only carries the absolute error of the large one.  So the checks here are normwise,

    ||C - C_ref||_F <= c k eps ||op(A)||_F ||B||_F,   c = 2,

with k the reduction length, on inputs with balanced parts, with |Im| << |Re| and with |Im| >> |Re|.  numpy's product (the
reference) has an error of the same order, which the factor 2 covers.  Real data embedded in complex128 must give exactly
zero imaginary parts: there k2 = -k1 and k3 = 0 exactly."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
C_3M = 2.0

# (scale of the real part, scale of the imaginary part)
PARTS = {"balanced": (1.0, 1.0), "im_small": (1.0, 1e-9), "im_large": (1e-9, 1.0)}


@pytest.fixture(scope="module")
def dv():
    from morfem_b200 import device
    device.require_cuda()
    return device


def cplx(rng, shape, parts):
    sr, si = PARTS[parts]
    return sr * rng.standard_normal(shape) + 1j * si * rng.standard_normal(shape)


def assert_normwise(out, ref, k, na, nb):
    err = np.linalg.norm(out - ref)
    bound = C_3M * k * EPS * na * nb
    assert err <= bound, f"||C - C_ref|| = {err:.3e} > {bound:.3e} (c = {C_3M}, k = {k})"


@pytest.mark.parametrize("parts", sorted(PARTS))
@pytest.mark.parametrize("conj", [False, True])
@pytest.mark.parametrize("n,ra,rb", [(1000, 24, 40), (50000, 256, 256), (20011, 130, 7), (17, 64, 64)])
def test_gemm_tn_normwise(dv, n, ra, rb, conj, parts):
    rng = np.random.default_rng(n + ra + rb + 2 * conj)
    a, b = cplx(rng, (n, ra), parts), cplx(rng, (n, rb), parts)
    out = dv.gemm_tn(dv.to_device_c128(a), dv.to_device_c128(b), conj=conj).cpu().numpy()
    ref = (a.conj().T if conj else a.T) @ b
    assert_normwise(out, ref, n, np.linalg.norm(a), np.linalg.norm(b))


@pytest.mark.parametrize("parts", sorted(PARTS))
@pytest.mark.parametrize("n,r", [(40000, 256), (3001, 130), (999, 17)])
def test_gram_matrix_normwise_and_real_diagonal_error(dv, n, r, parts):
    """A^H A takes the Hermitian path (upper tiles only, mirrored in the reduction).  Its diagonal is real in exact arithmetic;
    3M leaves an imaginary part of rounding size there, which the Cholesky kernels never read."""
    rng = np.random.default_rng(n + r)
    a = cplx(rng, (n, r), parts)
    ad = dv.to_device_c128(a)
    g = dv.gemm_tn(ad, ad, conj=True).cpu().numpy()
    ref = a.conj().T @ a
    na = np.linalg.norm(a)
    assert_normwise(g, ref, n, na, na)
    col2 = np.sum(np.abs(a) ** 2, axis=0)
    assert np.all(np.abs(np.diag(g).imag) <= C_3M * n * EPS * col2)
    assert np.allclose(g, g.conj().T, rtol=0, atol=C_3M * n * EPS * na * na)


@pytest.mark.parametrize("parts", sorted(PARTS))
@pytest.mark.parametrize("n,ra,rb", [(100003, 256, 256), (1000, 24, 40), (5000, 100, 7), (130, 256, 130)])
def test_gemm_nn_normwise(dv, n, ra, rb, parts):
    rng = np.random.default_rng(n + ra + rb)
    a, w = cplx(rng, (n, ra), parts), cplx(rng, (ra, rb), parts)
    out = dv.gemm_nn(dv.to_device_c128(a), dv.to_device_c128(w)).cpu().numpy()
    assert_normwise(out, a @ w, ra, np.linalg.norm(a), np.linalg.norm(w))


@pytest.mark.parametrize("parts", sorted(PARTS))
@pytest.mark.parametrize("n,r", [(70001, 256), (700, 130), (150, 512)])
def test_trmm_normwise(dv, n, r, parts):
    rng = np.random.default_rng(n + r)
    a, w = cplx(rng, (n, r), parts), np.triu(cplx(rng, (r, r), parts))
    out = dv.gemm_nn(dv.to_device_c128(a), dv.to_device_c128(w), w_upper=True).cpu().numpy()
    assert_normwise(out, a @ w, r, np.linalg.norm(a), np.linalg.norm(w))


@pytest.mark.parametrize("n,ra,rb", [(30000, 256, 256), (4097, 130, 64), (333, 7, 5)])
def test_real_embedded_inputs_give_exactly_zero_imaginary_parts(dv, n, ra, rb):
    rng = np.random.default_rng(n + ra)
    a, b = rng.standard_normal((n, ra)), rng.standard_normal((n, rb))
    w, wt = rng.standard_normal((ra, rb)), np.triu(rng.standard_normal((ra, ra)))
    ad, bd = dv.to_device_c128(a), dv.to_device_c128(b)
    outs = {
        "gemm_tn": dv.gemm_tn(ad, bd),
        "gemm_tn conj": dv.gemm_tn(ad, bd, conj=True),
        "gram": dv.gemm_tn(ad, ad, conj=True),
        "gemm_nn": dv.gemm_nn(ad, dv.to_device_c128(w)),
        "trmm": dv.gemm_nn(ad, dv.to_device_c128(wt), w_upper=True),
    }
    for name, o in outs.items():
        o = o.cpu().numpy()
        assert np.abs(o.imag).max() == 0.0, name
    # conjugation is a no-op on real data: the two gemm_tn forms agree bit for bit
    assert np.array_equal(outs["gemm_tn"].cpu().numpy(), outs["gemm_tn conj"].cpu().numpy())


@pytest.mark.parametrize("parts", sorted(PARTS))
def test_cholesky_qr_of_complex_block_is_orthonormal(dv, parts):
    """CholeskyQR2 on genuinely complex data: the Gram diagonals carry rounding-level imaginary parts from 3M."""
    rng = np.random.default_rng(11)
    s = cplx(rng, (20000, 96), parts)
    q, _ = dv.orthonormalize(dv.to_device_c128(s))
    q = q.cpu().numpy()
    assert np.linalg.norm(q.conj().T @ q - np.eye(q.shape[1])) < 1e-12
    # span(q) = span(s): s is recovered from its projection onto q
    assert np.linalg.norm(s - q @ (q.conj().T @ s)) / np.linalg.norm(s) < 1e-12
