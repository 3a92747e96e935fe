"""The sweep tests' reference on its own, without torch or a GPU: every float64 and complex128 model builds a refined reference that
passes its own self-check (getrf's unrefined solution within the LAPACK test ratios), and the ratios reject a solution that is
wrong by far less than the sweep tests could miss."""
import numpy as np
import pytest
from scipy.linalg import lapack

from sweep_reference import (EPS, F64_MODELS, THRESH, Reference, backward_ratios, coefficients, complex_model, frequencies, real_model,
                             sample, singular_block, singular_columns, symmetrised)

COMPLEX_MODELS = (("balanced", 1e-2), ("balanced", 1e-6), ("near_real", 1e-9), ("near_imag", 1e-9))
SIZES = [(9, 2), (64, 4), (130, 9), (7, 9)]


def _models():
    out = [pytest.param(name, r, m, id=f"f64-{name}-r{r}-m{m}") for name in F64_MODELS for r, m in SIZES]
    out += [pytest.param(key, r, m, id=f"c128-{key[0]}{key[1]:g}-r{r}-m{m}") for key in COMPLEX_MODELS for r, m in SIZES]
    out += [pytest.param("real", r, m, id=f"c128-real-r{r}-m{m}") for r, m in SIZES]
    return out


def build(key, r, m):
    if key in F64_MODELS:
        ops, br = F64_MODELS[key](r, m)
        assert all(a.dtype == np.float64 for a in ops) and br.dtype == np.float64
    else:
        ops, br = real_model(r, m) if key == "real" else complex_model(*key, r, m)
    return symmetrised(ops), br


@pytest.mark.parametrize("key,r,m", _models())
def test_reference_passes_its_own_check(key, r, m):
    nf = 12
    sops, br = build(key, r, m)
    ref = Reference(sops, br, coefficients(frequencies(nf)), sample(nf, r))      # asserts the self-check
    assert ref.xs.dtype == (np.float64 if key in F64_MODELS else np.complex128)
    assert np.all(np.isfinite(ref.cond)) and ref.has_s == (m <= r)
    # a solution perturbed by 1e3 eps cond2 relative fails the forward ratio; one perturbed by 1e2 r eps in a random direction fails
    # the backward ratio whenever A is well conditioned
    rng = np.random.default_rng(r + m)
    d = rng.standard_normal(ref.xs.shape)
    norm = lambda a: np.linalg.norm(a.reshape(len(ref.idx), -1), axis=1)[:, None, None]      # noqa: E731
    nrm = norm(ref.xs) / norm(d)
    bad = ref.xs + 1e3 * EPS * ref.cond[:, None, None] * nrm * d
    assert np.all(ref.forward(bad) > THRESH)
    if key == "exchange":
        sub = [c[ref.idx] for c in ref.coef]
        assert np.all(backward_ratios(sops, sub, br, ref.xs + 1e2 * r * EPS * nrm * d) > THRESH)


@pytest.mark.parametrize("r", [2, 17, 33, 130, 512])
def test_singular_block_gives_known_info(r):
    for k in singular_columns(r) or [0]:
        assert lapack.dgetrf(singular_block(r, k, float))[2] == k + 2
        assert lapack.zgetrf(singular_block(r, k))[2] == k + 2
