"""The refined LAPACK reference of the reduced sweep (stages 3 + 4), shared by the float64 and complex128 sweep tests.

Reference.  Per point, A(t) = c0 A0 + c1 A1 + c2 A2 from the same symmetrised operators the kernels receive, solved by getrf
(scipy ``lu_factor`` / ``lu_solve``: dgetrf on float64 models, zgetrf on complex ones) and two steps of iterative refinement with
the residual in long double (``np.longdouble`` / ``np.clongdouble``): x*.  S* = 2 (I + Z*^-1)^-1 - I with Z* = j zs x*^T (cb Br).
The unrefined getrf solution must pass the same checks before x* is used, so that a failure points at the kernel and not at the test.

Checks (LAPACK's test ratios, with the threshold 30 of its dchkge / zchkge suites):
  backward error, every point     ||b - A x||_1 / (r ||A||_1 ||x||_1 eps)            per column, residual in long double
  forward error, sampled points   ||x - x*||_F / (||x*||_F cond2(A) eps)
  S-parameters, sampled points    ||S - S*||_F / (||S*||_F eps kappa)
                                  kappa = cond2(A) (||x*|| ||B|| / ||x*^T B||) cond(Z*) cond(I + Z*^-1)
  info == 0 on every point.
At most 16 points per run are sampled (cond2 costs an SVD per point); the backward error needs no reference and runs on all of them.

This module needs neither torch nor a GPU: the models and the reference are plain numpy / scipy."""
from collections import defaultdict

import numpy as np
import pytest
from scipy.constants import epsilon_0, pi
from scipy.linalg import lu_factor, lu_solve

from oracle import reference_path as orc

EPS = np.finfo(np.float64).eps
THRESH = 30.0

# the switches the sweep reads on every call; each run sets exactly the ones it names and clears the others
SWITCHES = ("MF_LEFT_VER", "MF_LEFT_CFG", "MF_LEFT_CHUNK", "MF_LEFT_LOOKAHEAD", "MF_STREAM_CFG", "MF_STREAM_FUSE",
            "MF_SWEEP_FORCE_SMEM", "MF_SWEEP_FORCE_LEFT")

WORST = defaultdict(lambda: np.zeros(3))      # family -> largest (backward, forward, S) ratio


@pytest.fixture(scope="module", autouse=True)
def report():
    """Prints (``pytest -s``) and forgets the largest ratios per family seen by the module that uses it."""
    yield
    if WORST:
        print("\nlargest ratios per family (threshold %g):  backward  forward  S" % THRESH)
        for fam in sorted(WORST):
            b, f, s = WORST[fam]
            print(f"  {fam:<22s} {b:9.3f} {f:8.3f} {s:8.3f}")
        WORST.clear()


def set_switches(monkeypatch, env):
    for k in SWITCHES:
        if k in env and env[k] is not None:
            monkeypatch.setenv(k, str(env[k]))
        else:
            monkeypatch.delenv(k, raising=False)


# ------------------------------------------------------------------------------------------------------------ models
def _sym(rng, r):
    """Symmetric, 2-norm ~ 1."""
    g = rng.standard_normal((r, r))
    return (g + g.T) / (2.0 * np.sqrt(2.0 * r))


def complex_model(regime, loss, r, m):
    """Host operators ``[a0, a1, a2]`` (complex, not symmetrised) and the port matrix ``br`` (r x m, complex): a seeded reduced
    waveguide model with a loss term on all three operators, in the regime ``balanced`` (times a phase), ``near_real`` or
    ``near_imag`` (times i)."""
    from morfem_b200 import synthetic
    seed = 1000 + 7 * r + m
    a0, _, a2, b = synthetic.reduced_model(r, m, seed=seed)
    rng = np.random.default_rng(seed)
    sym = lambda: _sym(rng, r)                              # noqa: E731
    n0, n2 = np.abs(a0).max(), np.abs(a2).max()
    a1 = (sym() + 1j * loss * sym()) * 1e-3 * n0 / 4e9       # c1(t) = t: a conductor-like term, 1e-3 of a0 at 4 GHz
    a0 = a0 + 1j * loss * n0 * sym()
    a2 = a2 + 1j * loss * n2 * sym()
    b2 = rng.standard_normal(b.shape) * np.sqrt(np.mean(b ** 2))
    phase, bre, bim = {"balanced": (np.exp(0.6j), 1.0, 1.0), "near_real": (1.0, 1.0, 1e-9), "near_imag": (1j, 1e-9, 1.0)}[regime]
    return [phase * a for a in (a0, a1, a2)], bre * b + 1j * bim * b2


def real_model(r, m):
    """The float64 waveguide model (``waveguide_f64``) embedded in complex128."""
    ops, br = waveguide_f64(r, m)
    return [a.astype(complex) for a in ops], br.astype(complex)


def waveguide_f64(r, m):
    """A seeded reduced waveguide model (real, not symmetrised) with a real symmetric conductor term ``a1`` of 1e-3 |a0| at 4 GHz
    (c1(t) = t)."""
    from morfem_b200 import synthetic
    a0, _, a2, b = synthetic.reduced_model(r, m, seed=2000 + r)
    rng = np.random.default_rng(r)
    a1 = 1e-3 * np.abs(a0).max() / 4e9 * _sym(rng, r)
    return [a0, a1, a2], b


def exchange_f64(r, m):
    """2 fliplr(I) + 1e-3 noise (real, not symmetrised), with small a1 and a2 terms: the anti-diagonal makes partial pivoting
    exchange rows in each of the first r / 2 columns, the noise decides the later pivots.  cond2 stays ~1."""
    rng = np.random.default_rng(3000 + 7 * r + m)
    a0 = 2.0 * np.fliplr(np.eye(r)) + 1e-3 * rng.standard_normal((r, r))
    a1 = 1e-3 / 4e9 * rng.standard_normal((r, r))
    a2 = 1e-3 / 1.6e19 * rng.standard_normal((r, r))
    return [a0, a1, a2], rng.standard_normal((r, m))


F64_MODELS = {"waveguide": waveguide_f64, "exchange": exchange_f64}


def singular_block(r, k, dtype=complex):
    """Identity with the symmetric block [[2, 1], [1, 0.5]] (times 1 + i for complex) at rows/columns k, k+1: the pivot is 2, the
    multiplier exactly 0.5 and U[k+1, k+1] exactly 0, so LU reports info = k + 2."""
    a = np.eye(r, dtype=dtype)
    z = (1 + 1j) if np.dtype(dtype).kind == "c" else 1.0
    a[k:k + 2, k:k + 2] = [[2 * z, z], [z, 0.5 * z]]
    return a


def singular_columns(r):
    """k such that columns k, k+1 straddle an 8-column register panel, a 16-column block column and a deep panel."""
    deep = 16 * ((r - 1) // 16) - 1
    return sorted({k for k in (7, 15, deep - 8, deep) if 0 <= k and k + 1 < r})


def frequencies(nf):
    return np.array([4e9]) if nf == 1 else np.linspace(3e9, 5e9, nf)


def coefficients(f):
    """(c0, c1, c2, cb, zs) of the waveguide sweep at the points f."""
    return np.ones_like(f), f.copy(), f ** 2, np.array([orc.b_coefficient(t) for t in f]), 2 * pi * f * epsilon_0


def symmetrised(ops):
    return [None if a is None else (a + a.T) / 2 for a in ops]


# --------------------------------------------------------------------------------------------------------- reference
def _is_complex(sops, br):
    return np.iscomplexobj(br) or any(s is not None and np.iscomplexobj(s) for s in sops)


def _types(sops, br):
    """(working type, long-double type) of a model: float64 / longdouble, or complex128 / clongdouble."""
    return (complex, np.clongdouble) if _is_complex(sops, br) else (np.float64, np.longdouble)


def system(sops, coef, i, dtype=None):
    if dtype is None:
        dtype = complex if _is_complex(sops, np.zeros(1)) else np.float64
    a = None
    for c, s in zip(coef[:3], sops):
        if s is not None:
            t = dtype(c[i]) * s.astype(dtype, copy=False)
            a = t if a is None else a + t
    return a


def cond2(a):
    s = np.linalg.svd(a, compute_uv=False)
    return s[0] / s[-1]


def sample(nf, r, extra=()):
    n = min(nf, 16 if r <= 256 else (8 if r <= 512 else 3))
    return np.unique(np.concatenate([np.linspace(0, nf - 1, n).round().astype(int), np.asarray(extra, dtype=int)]))


def backward_ratios(sops, coef, br, x):
    """Per point: max over the right-hand sides of ||b - A x||_1 / (r ||A||_1 ||x||_1 eps), the residual in long double."""
    nf, r, m = x.shape
    ld = np.clongdouble if (np.iscomplexobj(x) or _is_complex(sops, br)) else np.longdouble
    xl = np.moveaxis(x, 0, 1).reshape(r, nf * m).astype(ld)
    res = (coef[3][:, None, None] * br[None].astype(ld)).astype(ld)
    for c, s in zip(coef[:3], sops):
        if s is not None:
            res = res - c[:, None, None] * np.moveaxis((s.astype(ld) @ xl).reshape(r, nf, m), 1, 0)
    rn = np.abs(res).sum(axis=1).astype(np.float64)                                   # (nf, m) column 1-norms
    xn = np.abs(x).sum(axis=1)
    an = np.array([np.abs(system(sops, coef, i)).sum(axis=0).max() for i in range(nf)])
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.max(rn / (r * an[:, None] * xn * EPS), axis=1)


def gsm_host(x, br, cb, zs):
    z = 1j * zs * (x.T @ (cb * br))
    ident = np.eye(z.shape[0])
    return z, 2 * np.linalg.inv(ident + np.linalg.inv(z)) - ident


class Reference:
    """The refined reference of one model at the points ``idx`` of a coefficient set (x*, cond2, S*, kappa per point)."""

    def __init__(self, sops, br, coef, idx):
        self.sops, self.br, self.coef, self.idx = sops, br, coef, np.asarray(idx)
        r, m = br.shape
        wt, ld = _types(sops, br)
        self.has_s = m <= r            # for m > r, Z = j zs x^T B has rank r < m: no S-parameters to compare
        self.xs, self.cond, self.ss, self.kappa, x0s = [], [], [], [], []
        for i in self.idx:
            a, al = system(sops, coef, i, wt), system(sops, coef, i, ld)
            b = coef[3][i] * br
            lu = lu_factor(a)
            x0 = lu_solve(lu, b)
            xl = x0.astype(ld)
            for _ in range(2):
                xl = xl + lu_solve(lu, (b.astype(ld) - al @ xl).astype(wt))
            xs = xl.astype(wt)
            c = cond2(a)
            self.xs.append(xs); self.cond.append(c); x0s.append(x0)
            if self.has_s:
                bb = coef[3][i] * br
                z, s = gsm_host(xs, br, coef[3][i], coef[4][i])
                self.ss.append(s)
                self.kappa.append(c * np.linalg.norm(xs, 2) * np.linalg.norm(bb, 2) / np.linalg.norm(xs.T @ bb, 2) * np.linalg.cond(z) *
                                  np.linalg.cond(np.eye(m) + np.linalg.inv(z)))
        self.xs, self.ss = np.array(self.xs), np.array(self.ss)
        self.cond, self.kappa = np.array(self.cond), np.array(self.kappa)
        # getrf's own solution must pass every check against x* (else the reference could not tell a kernel error)
        x0s = np.array(x0s)
        sub = [c[self.idx] for c in coef]
        assert np.all(backward_ratios(sops, sub, br, x0s) < THRESH)
        assert np.all(self.forward(x0s) < THRESH)
        if self.has_s:
            s0 = np.array([gsm_host(x0, br, coef[3][i], coef[4][i])[1] for x0, i in zip(x0s, self.idx)])
            assert np.all(self.s_ratios(s0) < THRESH)

    def forward(self, x):
        """||x - x*||_F / (||x*||_F cond2(A) eps) at the reference points (x indexed like ``idx``)."""
        d = np.linalg.norm((x - self.xs).reshape(len(self.idx), -1), axis=1)
        return d / (np.linalg.norm(self.xs.reshape(len(self.idx), -1), axis=1) * self.cond * EPS)

    def s_ratios(self, s):
        if not self.has_s:
            return np.zeros(1)
        d = np.linalg.norm((s - self.ss).reshape(len(self.idx), -1), axis=1)
        return d / (np.linalg.norm(self.ss.reshape(len(self.idx), -1), axis=1) * self.kappa * EPS)


def check(family, ref, x, s, info, points=None):
    """Every check on one run; ``points`` restricts the backward error and the info check to a subset (default: all)."""
    points = np.arange(x.shape[0]) if points is None else np.asarray(points)
    assert not np.any(info[points]), (family, np.flatnonzero(info))
    coef = [c[points] for c in ref.coef]
    bw = backward_ratios(ref.sops, coef, ref.br, x[points])
    fw = ref.forward(x[ref.idx])
    sr = ref.s_ratios(s[ref.idx])
    w = WORST[family]
    w[:] = np.maximum(w, [bw.max(), fw.max(), sr.max()])
    assert np.all(bw < THRESH), (family, "backward", bw.max(), int(points[np.argmax(bw)]))
    assert np.all(fw < THRESH), (family, "forward", fw.max(), int(ref.idx[np.argmax(fw)]))
    assert np.all(sr < THRESH), (family, "S", sr.max(), int(ref.idx[np.argmax(sr)]))
