"""The complex128 sweep (stages 3 + 4: LU with partial pivoting per point, then the S-parameters) on genuinely complex models, for
every kernel family and launch geometry, against a refined LAPACK reference.

Models.  A seeded reduced waveguide model (``synthetic.reduced_model``) with a loss term on all three operators (``a1`` non-zero,
``c1(t) = t``) and a complex port matrix, in three regimes of the imaginary parts: balanced (the lossy model times a phase, loss 1e-2
and 1e-6), near-real (|Im| ~ 1e-9 |Re|: the kernels must not take their real fast paths) and near-imaginary (the same model times i:
pivots that are almost purely imaginary).  The loss sets how close the points come to a resonance: cond2(A(t)) runs from ~1e3 to ~1e7.

Reference.  Per point, A(t) = c0 A0 + c1 A1 + c2 A2 from the same symmetrised operators the kernels receive, solved by zgetrf
(scipy ``lu_factor`` / ``lu_solve``) and two steps of iterative refinement with the residual in clongdouble: x*.  S* = 2 (I + Z*^-1)^-1 - I
with Z* = j zs x*^T (cb Br).  The unrefined zgetrf solution must pass the same checks before x* is used, so that a failure points at
the kernel and not at the test.

Checks (LAPACK's test ratios, with the threshold 30 of its zchkge suite):
  backward error, every point     ||b - A x||_1 / (r ||A||_1 ||x||_1 eps)            per column, residual in clongdouble
  forward error, sampled points   ||x - x*||_F / (||x*||_F cond2(A) eps)
  S-parameters, sampled points    ||S - S*||_F / (||S*||_F eps kappa)
                                  kappa = cond2(A) (||x*|| ||B|| / ||x*^T B||) cond(Z*) cond(I + Z*^-1)
  info == 0 on every point.
At most 16 points per run are sampled (cond2 costs an SVD per point); the backward error needs no reference and runs on all of them.
The largest ratios seen per family are printed at the end of the module (``pytest -s``)."""
import ctypes
import os
import subprocess
import sys
import textwrap
from collections import defaultdict

import numpy as np
import pytest
from scipy.constants import epsilon_0, pi
from scipy.linalg import lapack, lu_factor, lu_solve

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import reference_path as orc   # noqa: E402  (checker only)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = np.finfo(np.float64).eps
THRESH = 30.0
CLD = np.clongdouble

# the switches the sweep reads on every call; each run sets exactly the ones it names and clears the others
SWITCHES = ("MF_LEFT_VER", "MF_LEFT_CFG", "MF_LEFT_CHUNK", "MF_LEFT_LOOKAHEAD", "MF_STREAM_CFG", "MF_STREAM_FUSE",
            "MF_SWEEP_FORCE_SMEM", "MF_SWEEP_FORCE_LEFT")

# (regime, relative loss)
MODELS = (("balanced", 1e-2), ("balanced", 1e-6), ("near_real", 1e-9), ("near_imag", 1e-9))

WORST = defaultdict(lambda: np.zeros(3))      # family -> largest (backward, forward, S) ratio


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if WORST:
        print("\nlargest ratios per family (threshold %g):  backward  forward  S" % THRESH)
        for fam in sorted(WORST):
            b, f, s = WORST[fam]
            print(f"  {fam:<22s} {b:9.3f} {f:8.3f} {s:8.3f}")


@pytest.fixture(scope="module")
def dv():
    from morfem_b200 import device
    device.require_cuda()
    return device


@pytest.fixture(scope="module")
def lib():
    from morfem_b200 import _ffi
    return _ffi.load()


# ------------------------------------------------------------------------------------------------------------ models
def complex_model(regime, loss, r, m):
    """Host operators ``[a0, a1, a2]`` (complex, not symmetrised) and the port matrix ``br`` (r x m, complex)."""
    from morfem_b200 import synthetic
    seed = 1000 + 7 * r + m
    a0, _, a2, b = synthetic.reduced_model(r, m, seed=seed)
    rng = np.random.default_rng(seed)

    def sym():                                              # symmetric, 2-norm ~ 1
        g = rng.standard_normal((r, r))
        return (g + g.T) / (2.0 * np.sqrt(2.0 * r))

    n0, n2 = np.abs(a0).max(), np.abs(a2).max()
    a1 = (sym() + 1j * loss * sym()) * 1e-3 * n0 / 4e9       # c1(t) = t: a conductor-like term, 1e-3 of a0 at 4 GHz
    a0 = a0 + 1j * loss * n0 * sym()
    a2 = a2 + 1j * loss * n2 * sym()
    b2 = rng.standard_normal(b.shape) * np.sqrt(np.mean(b ** 2))
    phase, bre, bim = {"balanced": (np.exp(0.6j), 1.0, 1.0), "near_real": (1.0, 1.0, 1e-9), "near_imag": (1j, 1e-9, 1.0)}[regime]
    return [phase * a for a in (a0, a1, a2)], bre * b + 1j * bim * b2


def real_model(r, m):
    from morfem_b200 import synthetic
    a0, _, a2, b = synthetic.reduced_model(r, m, seed=2000 + r)
    rng = np.random.default_rng(r)
    g = rng.standard_normal((r, r))
    a1 = 1e-3 * np.abs(a0).max() / 4e9 * (g + g.T) / (2.0 * np.sqrt(2.0 * r))
    return [a0.astype(complex), a1.astype(complex), a2.astype(complex)], b.astype(complex)


def singular_block(r, k):
    """Identity with the symmetric block [[2+2i, 1+i], [1+i, 0.5+0.5i]] at rows/columns k, k+1: under |re|+|im| pivoting the multiplier is
    exactly 0.5 and U[k+1, k+1] exactly 0, so LU reports info = k + 2."""
    a = np.eye(r, dtype=complex)
    a[k:k + 2, k:k + 2] = [[2 + 2j, 1 + 1j], [1 + 1j, 0.5 + 0.5j]]
    return a


def frequencies(nf):
    return np.array([4e9]) if nf == 1 else np.linspace(3e9, 5e9, nf)


def coefficients(f):
    """(c0, c1, c2, cb, zs) of the waveguide sweep at the points f."""
    return np.ones_like(f), f.copy(), f ** 2, np.array([orc.b_coefficient(t) for t in f]), 2 * pi * f * epsilon_0


def symmetrised(ops):
    return [None if a is None else (a + a.T) / 2 for a in ops]


# --------------------------------------------------------------------------------------------------------- reference
def system(sops, coef, i, dtype=complex):
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
    """Per point: max over the right-hand sides of ||b - A x||_1 / (r ||A||_1 ||x||_1 eps), the residual in clongdouble."""
    nf, r, m = x.shape
    xl = np.moveaxis(x, 0, 1).reshape(r, nf * m).astype(CLD)
    res = (coef[3][:, None, None] * br[None].astype(CLD)).astype(CLD)
    for c, s in zip(coef[:3], sops):
        if s is not None:
            res = res - c[:, None, None] * np.moveaxis((s.astype(CLD) @ xl).reshape(r, nf, m), 1, 0)
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
        self.has_s = m <= r            # for m > r, Z = j zs x^T B has rank r < m: no S-parameters to compare
        self.xs, self.cond, self.ss, self.kappa, x0s = [], [], [], [], []
        for i in self.idx:
            a, al = system(sops, coef, i), system(sops, coef, i, CLD)
            b = coef[3][i] * br
            lu = lu_factor(a)
            x0 = lu_solve(lu, b)
            xl = x0.astype(CLD)
            for _ in range(2):
                xl = xl + lu_solve(lu, (b.astype(CLD) - al @ xl).astype(complex))
            xs = xl.astype(complex)
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
        # zgetrf's own solution must pass every check against x* (else the reference could not tell a kernel error)
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


_models, _refs, _dev = {}, {}, {}


def model_case(key, r, m, nf):
    """Host operators (symmetrised), port matrix, coefficients and refined reference of one model; computed once per process."""
    if (key, r, m) not in _models:
        ops, br = real_model(r, m) if key == "real" else complex_model(*key, r, m)
        _models[(key, r, m)] = (symmetrised(ops), br, ops)
    sops, br, ops = _models[(key, r, m)]
    if (key, r, m, nf) not in _refs:
        coef = coefficients(frequencies(nf))
        _refs[(key, r, m, nf)] = Reference(sops, br, coef, sample(nf, r))
    return _refs[(key, r, m, nf)]


def device_operands(dv, key, r, m):
    """The raw operators uploaded and symmetrised by ``device.symmetrize`` (bit-equal to the host's (a + a^T) / 2), and the port matrix."""
    if (key, r, m) not in _dev:
        sops, br, ops = _models[(key, r, m)]
        dops = [dv.symmetrize(dv.to_device_c128(a)) for a in ops]
        for d, s in zip(dops, sops):
            assert np.array_equal(d.cpu().numpy(), s)
        _dev[(key, r, m)] = (dops, dv.to_device_c128(br))
    return _dev[(key, r, m)]


def set_switches(monkeypatch, env):
    for k in SWITCHES:
        if k in env and env[k] is not None:
            monkeypatch.setenv(k, str(env[k]))
        else:
            monkeypatch.delenv(k, raising=False)


def run_sweep(dv, dops, dbr, coef, variant, want_gsm=True):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()  # noqa: E731
    res = dv.sweep(*dops, dbr, *(t(c) for c in coef), want_x=True, want_gsm=want_gsm, variant=variant)
    torch.cuda.synchronize()
    return res.x.cpu().numpy(), (res.gsm.cpu().numpy() if want_gsm else None), res.info.cpu().numpy()


def check(family, ref, x, s, info, points=None):
    """Every check of the module on one run; ``points`` restricts the backward error to a subset (default: all)."""
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


# ------------------------------------------------------------------------------------------------ families and cases
# family -> (variant, switches)
FAMILIES = {
    "generic": (1, {}),
    "register_panel": (2, {}),
    "smem_blocked": (3, {}),
    "smem_blocked_large": (3, {"MF_SWEEP_FORCE_SMEM": 1}),
    "left_forced": (5, {}),
    "left_auto": (0, {}),
    "left_plain_body": (5, {"MF_LEFT_VER": 2}),
    "left_lookahead_body": (5, {"MF_LEFT_VER": 3}),
    "left_8warps_4blocks": (5, {"MF_LEFT_CFG": 4}),
    "left_two_point_cta": (5, {"MF_LEFT_CFG": 8}),
    "stream": (4, {}),
}

_R_M_F = {
    # generic: F = 300 > 296 resident CTAs of its workspace mode
    "generic": [(1, 1, 3), (5, 9, 4), (64, 16, 6), (200, 3, 300), (512, 2, 4), (700, 4, 3), (1024, 5, 2)],
    "register_panel": [(1, 2, 5), (2, 1, 7), (17, 8, 2000), (33, 4, 9), (64, 16, 6)],
    "smem_blocked": [(1, 3, 4), (8, 9, 6), (15, 2, 5), (16, 16, 4), (17, 5, 7), (40, 4, 9), (63, 1, 5), (64, 8, 1500)],
    # R = 128 never fits in shared memory (test_shared_memory_kernel_limit); F = 500 > one CTA per SM
    "smem_blocked_large": [(65, 2, 500), (80, 5, 6), (112, 16, 4), (112, 9, 5)],
    "left_forced": [(1, 4, 3), (16, 2, 6), (33, 9, 5), (64, 3, 700)],
    # every left_geom boundary (R = 112 | 128 | 256 | 512) and the left_chunk boundary at R = 192 / 208; F = 300 > 296 resident CTAs
    "left_auto": [(65, 1, 5), (112, 2, 6), (113, 3, 4), (128, 4, 5), (129, 5, 300), (192, 8, 4), (193, 9, 3), (208, 16, 4), (255, 1, 5),
                  (256, 2, 4), (257, 3, 3), (400, 4, 3), (511, 5, 2), (512, 8, 3)],
    "left_plain_body": [(65, 1, 600), (128, 4, 5), (200, 9, 4), (256, 16, 3), (257, 2, 4), (512, 5, 2)],
    "left_lookahead_body": [(65, 1, 600), (128, 4, 5), (200, 9, 4), (256, 16, 3), (257, 2, 4), (512, 5, 2)],
    "left_8warps_4blocks": [(129, 2, 150), (256, 5, 4), (300, 8, 3), (512, 16, 2)],
    # F = 1, odd F, F > 2 x SMs
    "left_two_point_cta": [(17, 2, 1), (40, 3, 7), (130, 5, 301), (256, 4, 5)],
}
STREAM_M = {113: 1, 128: 4, 200: 9, 256: 16, 257: 3, 512: 8}


def _cases():
    out = []
    for fam, rows in _R_M_F.items():
        for i, (r, m, nf) in enumerate(rows):
            variant, env = FAMILIES[fam]
            if fam == "left_auto":
                variant = (0, 3)[i % 2]
            model = MODELS[i % len(MODELS)]
            out.append(pytest.param(fam, variant, env, model, r, m, nf, id=f"{fam}-r{r}-m{m}-F{nf}-{model[0]}{model[1]:g}"))
    i = 0
    for r, m in STREAM_M.items():
        for cfg in ((None, 0, 1, 2, 3) if r <= 256 else (None,)):
            for fuse in (0, 1):
                nf = 450 if (r, cfg, fuse) == (128, None, 1) else 5          # F = 450 > three CTAs per SM
                env = {"MF_STREAM_CFG": cfg, "MF_STREAM_FUSE": fuse}
                model = MODELS[i % len(MODELS)]
                out.append(pytest.param("stream", 4, env, model, r, m, nf, id=f"stream-r{r}-m{m}-F{nf}-cfg{cfg}-fuse{fuse}-{model[0]}{model[1]:g}"))
                i += 1
    return out


@pytest.mark.parametrize("family,variant,env,model,r,m,nf", _cases())
def test_family_matches_refined_reference(dv, lib, monkeypatch, family, variant, env, model, r, m, nf):
    set_switches(monkeypatch, env)
    assert lib.mf_sweep_variant_supported(r, m, variant)
    if family == "smem_blocked_large":
        assert lib.mf_sweep_ws_bytes(r, m, nf, 3) == 256          # the shared-memory kernel runs, not the left-looking one
    ref = model_case(model, r, m, nf)
    dops, dbr = device_operands(dv, model, r, m)
    x, s, info = run_sweep(dv, dops, dbr, ref.coef, variant)
    check(family, ref, x, s, info)


def test_shared_memory_kernel_limit(lib, monkeypatch):
    """The shared-memory kernel is built for R <= 128 but its matrix only fits up to r = 112 (R = 120 and 128 need more than 226 KiB)."""
    set_switches(monkeypatch, {"MF_SWEEP_FORCE_SMEM": 1})
    assert all(lib.mf_sweep_ws_bytes(112, m, 10, 3) == 256 for m in (1, 8, 9, 16))
    assert all(lib.mf_sweep_ws_bytes(r, m, 10, 3) > 256 for r in (113, 120, 128) for m in (1, 16))


@pytest.mark.parametrize("r,m,ver,model", [(208, 3, 2, MODELS[0]), (208, 3, 3, MODELS[3]), (256, 4, 2, MODELS[2]), (256, 4, 3, MODELS[1])])
def test_short_launches_are_bit_equal_and_match_reference(dv, monkeypatch, r, m, ver, model):
    """F = 700 points: several launches of chunk x resident CTAs with a ragged last one; the same body gives the same bits whatever the
    launch length, and the library's own choice passes the checks too."""
    nf = 700
    ref = model_case(model, r, m, nf)
    dops, dbr = device_operands(dv, model, r, m)
    set_switches(monkeypatch, {"MF_LEFT_VER": ver, "MF_LEFT_CHUNK": 0})
    x, s, info = run_sweep(dv, dops, dbr, ref.coef, 5)
    check("left_short_launches", ref, x, s, info)
    for chunk in (1, 2):
        set_switches(monkeypatch, {"MF_LEFT_VER": ver, "MF_LEFT_CHUNK": chunk})
        xc, sc, ic = run_sweep(dv, dops, dbr, ref.coef, 5)
        assert np.array_equal(xc, x) and np.array_equal(sc, s) and np.array_equal(ic, info), chunk
    set_switches(monkeypatch, {})
    x, s, info = run_sweep(dv, dops, dbr, ref.coef, 0)
    check("left_short_launches", ref, x, s, info)


# ------------------------------------------------------------------------------------------------ complex properties
# one representative (r, m) per family: (family, r, m)
PROPERTY_CASES = [("generic", 200, 3), ("generic", 40, 2), ("register_panel", 33, 4), ("smem_blocked", 40, 5),
                  ("smem_blocked_large", 80, 2), ("left_forced", 64, 3), ("left_auto", 256, 4), ("left_plain_body", 200, 9),
                  ("left_lookahead_body", 257, 2), ("left_8warps_4blocks", 300, 8), ("left_two_point_cta", 130, 5), ("stream", 200, 4),
                  ("stream", 512, 16)]


def _pair_ratio(a, b, ref):
    d = np.linalg.norm((a - b).reshape(a.shape[0], -1), axis=1)
    return d / (np.linalg.norm(b.reshape(b.shape[0], -1), axis=1) * ref.cond * EPS)


@pytest.mark.parametrize("family,r,m", PROPERTY_CASES)
def test_rotation_by_i_and_conjugation(dv, monkeypatch, family, r, m):
    """i A x' = b has x' = -i x with the same |re|+|im| pivots (every real pivot becomes purely imaginary); conj(A) x' = conj(b) has
    x' = conj(x).  Neither is bit-exact (host zgetrf differs by ~1e-14 under the rotation too), so the forward-error ratio applies."""
    variant, env = FAMILIES[family]
    set_switches(monkeypatch, env)
    nf = 5
    real = model_case("real", r, m, nf)
    assert len(real.idx) == nf
    dops, dbr = device_operands(dv, "real", r, m)
    x, s, info = run_sweep(dv, dops, dbr, real.coef, variant)
    check(family, real, x, s, info)
    xr, _, info_r = run_sweep(dv, [1j * o for o in dops], dbr, real.coef, variant, want_gsm=False)
    assert np.array_equal(info_r, info)
    rot = _pair_ratio(xr, -1j * x, real)
    assert np.all(rot < THRESH), ("rotation", rot.max())

    cplx = model_case(MODELS[0], r, m, nf)
    dops, dbr = device_operands(dv, MODELS[0], r, m)
    x, s, info = run_sweep(dv, dops, dbr, cplx.coef, variant)
    check(family, cplx, x, s, info)
    xc, _, info_c = run_sweep(dv, [o.conj().resolve_conj() for o in dops], dbr.conj().resolve_conj(), cplx.coef, variant, want_gsm=False)
    assert np.array_equal(info_c, info)
    cj = _pair_ratio(xc, x.conj(), cplx)
    assert np.all(cj < THRESH), ("conjugation", cj.max())
    WORST[family][1] = max(WORST[family][1], rot.max(), cj.max())


def singular_columns(r):
    """k such that columns k, k+1 straddle an 8-column register panel, a 16-column block column and a deep panel."""
    deep = 16 * ((r - 1) // 16) - 1
    return sorted({k for k in (7, 15, deep - 8, deep) if 0 <= k and k + 1 < r})


@pytest.mark.parametrize("family,r,m", PROPERTY_CASES)
def test_complex_singular_points(dv, monkeypatch, family, r, m):
    variant, env = FAMILIES[family]
    set_switches(monkeypatch, env)
    f = np.array([3e9, 4e9, 5e9])
    coef = (np.ones(3), f, f ** 2, np.ones(3), np.ones(3))
    ks = singular_columns(r)
    assert ks
    for k in ks:
        a = singular_block(r, k)
        for rot in (1.0, 1j):
            assert lapack.zgetrf(rot * a)[2] == k + 2
            _, _, info = run_sweep(dv, [dv.to_device_c128(rot * a), None, None], dv.to_device_c128(np.ones((r, m))), coef, variant,
                                   want_gsm=False)
            assert list(info) == [k + 2] * 3, (k, rot)


# --------------------------------------------------------------------------------------- per-point state inside one CTA
def abi_sweep(lib, dops, dbr, coef, variant, ws_bytes):
    """mf_sweep_lu_gsm_c128 through ctypes with a workspace of exactly ``ws_bytes`` (the launchers shrink the grid to fit it)."""
    from morfem_b200 import _ffi
    nf = coef[0].size
    r, m = dbr.shape
    cd = [torch.from_numpy(np.ascontiguousarray(c, dtype=np.float64)).cuda() for c in coef]
    x = torch.empty((nf, r, m), dtype=torch.complex128, device="cuda")
    s = torch.empty((nf, m, m), dtype=torch.complex128, device="cuda")
    info = torch.zeros(nf, dtype=torch.int32, device="cuda")
    ws = torch.empty(max(int(ws_bytes), 1), dtype=torch.uint8, device="cuda")
    p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())  # noqa: E731
    _ffi.check(lib.mf_sweep_lu_gsm_c128(p(dops[0]), p(dops[1]), p(dops[2]), dops[0].stride(0), p(dbr), dbr.stride(0), r, m,
                                        *(p(c) for c in cd), nf, p(x), p(s), p(info), variant, p(ws), int(ws_bytes),
                                        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "mf_sweep_lu_gsm_c128")
    torch.cuda.synchronize()
    return x.cpu().numpy(), s.cpu().numpy(), info.cpu().numpy()


@pytest.mark.parametrize("family,variant,env,r,m,slots", [
    ("generic", 1, {}, 130, 3, 1),                         # workspace mode (the matrix no longer fits in shared memory)
    ("left_auto", 3, {}, 80, 2, 1),
    ("stream", 4, {}, 200, 4, 1),
    ("left_forced", 5, {}, 256, 5, 1),                     # short launches of two points each
    ("left_two_point_cta", 5, {"MF_LEFT_CFG": 8}, 130, 2, 2),
])
def test_one_cta_runs_every_point_in_order(dv, lib, monkeypatch, family, variant, env, r, m, slots):
    """A workspace of one slot (two for the two-point CTA) makes one CTA run all F = 7 points in a row.  Point 2 is exactly singular
    (A = c2 E with the complex singular block in E); every later point must be unaffected by it: info flags point 2 only, the other
    points pass the checks, and x and S are bit-equal to a run with the full workspace."""
    set_switches(monkeypatch, env)
    nf, k = 7, r // 2 + 3
    ops, br = complex_model("balanced", 1e-2, r, m)
    f = frequencies(nf)
    c0, c1, _, cb, zs = coefficients(f)
    c2 = np.zeros(nf)
    c0[2], c1[2], c2[2] = 0.0, 0.0, 1.0
    coef = (c0, c1, c2, cb, zs)
    ops = [ops[0], ops[1], singular_block(r, k)]
    sops = symmetrised(ops)
    good = np.array([i for i in range(nf) if i != 2])
    ref = Reference(sops, br, coef, good)
    dops = [dv.symmetrize(dv.to_device_c128(a)) for a in ops]
    dbr = dv.to_device_c128(br)
    one = lib.mf_sweep_ws_bytes(r, m, slots, variant)
    full = lib.mf_sweep_ws_bytes(r, m, nf, variant)
    assert one < full
    x1, s1, i1 = abi_sweep(lib, dops, dbr, coef, variant, one)
    xf, sf, if_ = abi_sweep(lib, dops, dbr, coef, variant, full)
    assert list(np.flatnonzero(i1)) == [2] and i1[2] == k + 2
    assert np.array_equal(i1, if_)
    check(family, ref, x1, s1, i1, points=good)
    assert np.array_equal(x1[good], xf[good]) and np.array_equal(s1[good], sf[good])


# ------------------------------------------------------------------------------------------------- stage 4 on its own
@pytest.mark.parametrize("m", [1, 2, 3, 4, 5, 8, 9, 16])
def test_stage4_on_general_complex_impedance(dv, m):
    """mf_gsm_c128 on x with B = the first m columns of I (and zs = cb = 1), so that Z = j x[:m]^T is chosen directly: random complex Z
    and, for m > 1, a Z whose I + Z^-1 has a zero (1, 1) entry, which forces a row exchange in the epilogue's first pivot search."""
    rng = np.random.default_rng(m)
    r = m + 3
    zs_list = [rng.standard_normal((m, m)) + 1j * rng.standard_normal((m, m)) for _ in range(4)]
    zs_list.append(1e-3 * rng.standard_normal((m, m)) + 1j * 1e3 * rng.standard_normal((m, m)))
    if m > 1:
        y = rng.standard_normal((m, m)) + 1j * rng.standard_normal((m, m))
        y[0, 0] = -1.0
        zs_list.append(np.linalg.inv(y))
    nf = len(zs_list)
    x = rng.standard_normal((nf, r, m)) + 1j * rng.standard_normal((nf, r, m))       # rows >= m meet zero rows of B
    for i, z in enumerate(zs_list):
        x[i, :m] = (-1j * z).T
    b = np.eye(r, m)
    ones = torch.ones(nf, dtype=torch.float64, device="cuda")
    s = dv.gsm(dv.to_device_c128(x), dv.to_device_c128(b), ones, ones).cpu().numpy()
    for i in range(nf):
        z, s_ref = gsm_host(x[i], b, 1.0, 1.0)
        kappa = np.linalg.cond(z) * np.linalg.cond(np.eye(m) + np.linalg.inv(z))
        err = np.linalg.norm(s[i] - s_ref) / np.linalg.norm(s_ref)
        assert err < THRESH * EPS * kappa, (i, err, kappa)


# ------------------------------------------------------------------------------------- remap (read once per process)
@pytest.mark.parametrize("r,m,remap", [(200, 3, 1), (128, 4, 0)])
def test_left_looking_remap_in_child_process(dv, tmp_path, r, m, remap):
    """MF_LEFT_REMAP (panel warps on their own SM sub-partitions) is read once per process, so it runs in a child process: forced on at
    r = 200 and off at r = 128, where the library remaps by default."""
    model = MODELS[(r + remap) % 4]
    ref = model_case(model, r, m, 6)
    sops, br, ops = _models[(model, r, m)]
    np.savez(tmp_path / "in.npz", a0=ops[0], a1=ops[1], a2=ops[2], br=br, c=np.array(ref.coef))
    script = textwrap.dedent("""
        import sys, numpy as np, torch
        from morfem_b200 import device as dv
        d = np.load(sys.argv[1])
        ops = [dv.symmetrize(dv.to_device_c128(d[k])) for k in ("a0", "a1", "a2")]
        c = [torch.from_numpy(np.ascontiguousarray(v)).cuda() for v in d["c"]]
        res = dv.sweep(*ops, dv.to_device_c128(d["br"]), *c, want_x=True, want_gsm=True, variant=5)
        np.savez(sys.argv[2], x=res.x.cpu().numpy(), s=res.gsm.cpu().numpy(), info=res.info.cpu().numpy())
    """)
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env["MF_LEFT_REMAP"] = str(remap)
    out = subprocess.run([sys.executable, "-c", script, str(tmp_path / "in.npz"), str(tmp_path / "out.npz")], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    o = np.load(tmp_path / "out.npz")
    check("left_remap", ref, o["x"], o["s"], o["info"])
