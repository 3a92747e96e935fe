"""The float64 sweep (``mf_sweep_lu_gsm_f64``: LU with partial pivoting per point, then the S-parameters) for every kernel
instance and launch geometry, with a non-zero first-order term, against the refined LAPACK reference of ``sweep_reference``
(dgetrf, refinement in long double, LAPACK's test ratios with the threshold 30).

Models (real, symmetrised on the device by ``device.symmetrize``, which must be bit-equal to the host's (a + a^T) / 2):
  waveguide   a seeded reduced waveguide model plus a real symmetric conductor term a1 of ~1e-3 |a0| at 4 GHz, c1(t) = t;
              cond2(A(t)) ~ 7e2 .. 1.3e6 over the 3-5 GHz points at r = 9 .. 256.
  exchange    2 fliplr(I) + 1e-3 noise (with small a1 and a2 terms): partial pivoting exchanges rows in each of the first r / 2
              columns; cond2 ~ 1.
A case with more points than the instance has resident CTAs (multiprocessor count x the minimum CTAs per SM of its
``__launch_bounds__``) runs its points on the static operator A0 + t A1 instead, with point 1 exactly singular (A = E, the
identity with the block [[2, 1], [1, 0.5]]): with a grid-stride loop the CTA that runs that point runs later ones too, and info must
flag that point only while every other point passes the checks.

Kernel instances (``sweep_blocked_f64.cu``: shared-memory kernel by R = 8 ceil(r / 8); ``sweep_left.cu``: left-looking kernel by
geometry cfg and body MF_LEFT_VER) and their minimum CTAs per SM:
  smem   R <= 32: 12   R <= 64: 5   R <= 96: 2   R <= 128: 1
  left   cfg 1 (4 warps x 2 blocks, R <= 128): 4   cfg 5 (4 x 4, R <= 256): 4   cfg 2 (8 x 2, R <= 256): 3   cfg 4 (8 x 4): 2
         cfg 3 (16 x 2): 1;  each with the plain (2) and the look-ahead (3) body
The largest ratios seen per family are printed at the end of the module (``pytest -s``)."""
import ctypes
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
from scipy.linalg import lapack

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from sweep_reference import (F64_MODELS, Reference, backward_ratios, check, coefficients, complex_model, frequencies,  # noqa: E402,F401
                             report, sample, set_switches, singular_block, singular_columns, symmetrised, THRESH)
import test_gpu_sweep_complex as cplx_mod                                                                      # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dv():
    from morfem_b200 import device
    device.require_cuda()
    return device


@pytest.fixture(scope="module")
def lib():
    from morfem_b200 import _ffi
    return _ffi.load()


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------ kernel instances
LEFT_COVER = {1: 8, 2: 16, 3: 32, 4: 32, 5: 16}          # 16-row blocks a geometry covers (warps x blocks per warp)
LEFT_MINB = {1: 4, 2: 3, 3: 1, 4: 2, 5: 4}               # __launch_bounds__ minimum CTAs per SM of the float64 instances


def left_cfg(r, env):
    """The geometry ``left_geom<double>`` picks: the measured choice, or MF_LEFT_CFG when that geometry covers R."""
    nb = -(-r // 16)
    auto = 1 if nb <= 8 else 5 if nb <= 10 else 2 if nb <= 16 else 4
    c = int(env.get("MF_LEFT_CFG") or auto)
    return c if LEFT_COVER[c] >= nb else auto


def smem_minb(r):
    big_r = -(-r // 8) * 8
    return 12 if big_r <= 32 else 5 if big_r <= 64 else 2 if big_r <= 96 else 1


def uses_left(r, variant, env):
    if variant in (3, 5):
        return variant == 5
    if env.get("MF_SWEEP_FORCE_SMEM") and r <= 128:
        return False
    return r > 72 or bool(env.get("MF_SWEEP_FORCE_LEFT")) or r > 128


def instance(r, variant, env):
    """(name, minimum CTAs per SM) of the kernel instance a float64 sweep runs."""
    if not uses_left(r, variant, env):
        return f"smem_R{min(128, 32 * -(-r // 32))}", smem_minb(r)
    c = left_cfg(r, env)
    return f"left_cfg{c}_body{int(env.get('MF_LEFT_VER') or 2)}", LEFT_MINB[c]


def assert_instance(lib, sms, r, m, variant, env):
    """The library's workspace size confirms the kernel the case is meant to run and its resident CTA count: none for the
    shared-memory kernel, one left-looking slot per resident CTA otherwise."""
    name, minb = instance(r, variant, env)
    ws = lib.mf_sweep_f64_ws_bytes(r, m, 10 ** 6, variant)
    if name.startswith("smem"):
        assert ws == 256, (name, ws)
    else:
        nb = -(-r // 16)
        slot = 8 * (nb * 16 * nb * 16 + nb * nb * 256 + 2 * nb * 256)
        assert ws == slot * sms * minb, (name, ws, slot * sms * minb)
    return name, sms * minb


# ------------------------------------------------------------------------------------------------------------ helpers
_refs, _dev = {}, {}


def host_model(model, r, m, singular=None):
    """Host operators (raw), port matrix and coefficients of one case.  ``singular = (nf, p)``: the static operator A0 + t A1 at nf
    points, point p replaced by the exactly singular E (in the place of A2)."""
    ops, br = F64_MODELS[model](r, m)
    if singular is None:
        return ops, br, None
    nf, p = singular
    c0, c1, _, cb, zs = coefficients(frequencies(nf))
    c2 = np.zeros(nf)
    c0[p], c1[p], c2[p] = 0.0, 0.0, 1.0
    return [ops[0], ops[1], singular_block(r, (r - 2) // 2, float) if r > 1 else np.zeros((1, 1))], br, (c0, c1, c2, cb, zs)


def singular_info(r):
    return (r - 2) // 2 + 2 if r > 1 else 1


def upload(dv, ops, br):
    """The raw operators uploaded and symmetrised by ``device.symmetrize`` (bit-equal to the host's (a + a^T) / 2), and the port matrix."""
    dops = [None if a is None else dv.symmetrize(dv.real_or_complex_to_device(a)) for a in ops]
    for d, s in zip(dops, symmetrised(ops)):
        if d is not None:
            assert d.dtype == torch.float64 and np.array_equal(d.cpu().numpy(), s)
    return dops, dv.real_or_complex_to_device(br)


def case(dv, model, r, m, nf, singular_point=None):
    """(reference, device operators) of one case; computed once per process."""
    key = (model, r, m, nf, singular_point)
    if key not in _refs:
        ops, br, coef = host_model(model, r, m, None if singular_point is None else (nf, singular_point))
        if coef is None:
            coef = coefficients(frequencies(nf))
        idx = [i for i in sample(nf, r) if i != singular_point]
        _refs[key] = Reference(symmetrised(ops), br, coef, idx)
        _dev[key] = upload(dv, ops, br)
    return _refs[key], _dev[key]


def run_sweep(dv, dops, dbr, coef, variant, want_gsm=True):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()  # noqa: E731
    res = dv.sweep(*dops, dbr, *(t(c) for c in coef), want_x=True, want_gsm=want_gsm, variant=variant)
    torch.cuda.synchronize()
    return res.x.cpu().numpy(), (res.gsm.cpu().numpy() if want_gsm else None), res.info.cpu().numpy()


# ------------------------------------------------------------------------------------------------ families and cases
# family -> (variant, switches)
FAMILIES = {
    "smem": (3, {}),
    "smem_auto_forced": (0, {"MF_SWEEP_FORCE_SMEM": 1}),
    "left_auto": (0, {}),
    "left_forced_small": (0, {"MF_SWEEP_FORCE_LEFT": 1}),
    "left_cfg1": (5, {"MF_LEFT_CFG": 1}),
    "left_cfg2": (5, {"MF_LEFT_CFG": 2}),
    "left_cfg3": (5, {"MF_LEFT_CFG": 3}),
    "left_cfg4": (5, {"MF_LEFT_CFG": 4}),
    "left_cfg5": (5, {"MF_LEFT_CFG": 5}),
    "left_cfg3_body3": (5, {"MF_LEFT_CFG": 3, "MF_LEFT_VER": 3}),
    "left_body2": (5, {"MF_LEFT_VER": 2}),
    "left_body3": (5, {"MF_LEFT_VER": 3}),
}

# (r, m, F); F = "+k" means resident CTAs of the instance + k (k >= 2: those cases carry the singular point 1, and the CTA that runs
# it runs point 1 + grid too)
_R_M_F = {
    "smem": [(1, 1, 4), (7, 9, 5), (8, 16, 3), (9, 2, 6), (31, 3, "+5"), (32, 4, 7), (33, 5, 5), (63, 8, "+3"), (64, 9, 6), (65, 16, 4),
             (96, 1, "+9"), (97, 2, 5), (127, 3, "+4"), (128, 4, 6)],
    "smem_auto_forced": [(73, 5, 6), (100, 8, 5), (128, 16, 4)],
    # cfg 1 | 5 | 2 | 4 boundaries (R = 128 | 160 | 256) and the left_chunk boundary (R = 192)
    "left_auto": [(73, 1, 5), (128, 2, "+3"), (129, 3, 4), (144, 4, 5), (160, 5, "+3"), (161, 8, 4), (191, 9, 3), (192, 16, 4),
                  (256, 1, "+5"), (257, 2, 3), (511, 3, 2), (512, 1, "+3")],
    "left_forced_small": [(1, 2, 3), (16, 16, 4), (33, 9, 5), (72, 3, 6)],
    # cfg 1 is the automatic choice wherever it covers R; R = 144 falls back to cfg 5
    "left_cfg1": [(40, 5, 5), (128, 8, 4), (129, 9, 4)],
    # not the automatic choice at r = 100 (cfg 1) and 150 (cfg 5); r = 257 falls back to cfg 4
    "left_cfg2": [(100, 3, 5), (150, 4, 4), (256, 16, "+2"), (257, 1, 3)],
    "left_cfg3": [(17, 2, 4), (200, 5, 5), (512, 8, "+4")],
    "left_cfg4": [(64, 9, 4), (160, 16, 5), (300, 1, "+4")],
    # not the automatic choice at r = 100 (cfg 1) and 250 (cfg 2); r = 300 falls back to cfg 4
    "left_cfg5": [(100, 2, 5), (150, 3, "+2"), (250, 4, 4), (300, 5, 3)],
    "left_cfg3_body3": [(400, 9, "+3")],
    "left_body2": [(65, 16, 5), (160, 1, 4), (200, 2, 4), (256, 3, 3), (512, 5, 2)],
    "left_body3": [(65, 4, "+3"), (160, 5, "+2"), (200, 8, "+2"), (256, 9, 3), (512, 1, "+3")],
}


def _cases():
    out = []
    for fam, rows in _R_M_F.items():
        variant, env = FAMILIES[fam]
        for i, (r, m, nf) in enumerate(rows):
            model = ("waveguide", "exchange")[i % 2]
            out.append(pytest.param(fam, variant, env, model, r, m, nf, id=f"{fam}-r{r}-m{m}-F{nf}-{model}"))
    return out


@pytest.mark.parametrize("family,variant,env,model,r,m,nf", _cases())
def test_family_matches_refined_reference(dv, lib, sms, monkeypatch, family, variant, env, model, r, m, nf):
    set_switches(monkeypatch, env)
    assert lib.mf_sweep_f64_variant_supported(r, m, variant)
    name, resident = assert_instance(lib, sms, r, m, variant, env)
    p = None
    if isinstance(nf, str):
        nf, p = resident + int(nf), 1
        assert p + resident < nf
    ref, (dops, dbr) = case(dv, model, r, m, nf, p)
    x, s, info = run_sweep(dv, dops, dbr, ref.coef, variant)
    assert x.dtype == np.float64 and s.dtype == np.complex128
    if p is None:
        check(family, ref, x, s, info)
    else:
        assert list(np.flatnonzero(info)) == [p] and info[p] == singular_info(r), (name, np.flatnonzero(info))
        check(family, ref, x, s, info, points=np.array([i for i in range(nf) if i != p]))


def test_every_instance_runs_more_points_than_resident_ctas(sms):
    """Bookkeeping of the table above: every float64 kernel instance has a case with F > resident CTAs."""
    over = {instance(r, *FAMILIES[fam])[0] for fam, rows in _R_M_F.items() for r, m, nf in rows if isinstance(nf, str)}
    want = {f"smem_R{R}" for R in (32, 64, 96, 128)} | {f"left_cfg{c}_body{v}" for c in (1, 2, 3, 4, 5) for v in (2, 3)}
    assert over == want, want - over


# ------------------------------------------------------------------------------------------------------- properties
# one representative (r, m) per family
PROPERTY_CASES = [("smem", 40, 5), ("smem_auto_forced", 100, 8), ("left_auto", 200, 3), ("left_forced_small", 33, 4), ("left_cfg1", 100, 2),
                  ("left_cfg2", 150, 4), ("left_cfg3", 200, 5), ("left_cfg4", 300, 1), ("left_cfg5", 250, 4), ("left_cfg3_body3", 400, 9),
                  ("left_body2", 256, 3), ("left_body3", 200, 8)]

_SCALE_CASES = ([pytest.param("f64", fam, r, m, id=f"f64-{fam}-r{r}-m{m}") for fam, r, m in PROPERTY_CASES] +
                [pytest.param("c128", fam, r, m, id=f"c128-{fam}-r{r}-m{m}") for fam, r, m in cplx_mod.PROPERTY_CASES])


@pytest.mark.parametrize("kind,family,r,m", _SCALE_CASES)
def test_power_of_two_scaling_is_bit_exact(dv, monkeypatch, kind, family, r, m):
    """Every operator and cb times 2^k, zs times 2^-k (k = +-200): x and S are unchanged and, as no intermediate under- or overflows
    at these magnitudes, every operation scales exactly, so the results must be bit-equal.  An absolute threshold, or a reciprocal
    taken of the wrong quantity, breaks this."""
    variant, env = (FAMILIES if kind == "f64" else cplx_mod.FAMILIES)[family]
    set_switches(monkeypatch, env)
    nf = 5
    coef = coefficients(frequencies(nf))
    if kind == "f64":
        ops, br = F64_MODELS["waveguide"](r, m)
        up = dv.real_or_complex_to_device
    else:
        ops, br = complex_model("balanced", 1e-2, r, m)
        up = dv.to_device_c128
    ref = Reference(symmetrised(ops), br, coef, sample(nf, r))
    dbr = up(br)
    x, s, info = run_sweep(dv, [dv.symmetrize(up(a)) for a in ops], dbr, coef, variant)
    check(family if kind == "f64" else "c128_" + family, ref, x, s, info)
    for k in (200, -200):
        sc = np.ldexp(1.0, k)
        c = (coef[0], coef[1], coef[2], coef[3] * sc, coef[4] / sc)
        xk, sk, ik = run_sweep(dv, [dv.symmetrize(up(a * sc)) for a in ops], dbr, c, variant)
        assert np.array_equal(ik, info) and np.array_equal(xk, x) and np.array_equal(sk, s), (k, np.abs(xk - x).max(), np.abs(sk - s).max())


@pytest.mark.parametrize("r,m", [(1, 1), (9, 2), (33, 3), (64, 4), (65, 5), (96, 8), (112, 16), (104, 9)])
@pytest.mark.parametrize("with_a1", [True, False])
def test_shared_memory_kernel_real_equals_complex(dv, monkeypatch, r, m, with_a1):
    """The float64 shared-memory kernel runs the complex128 one's algorithm on real elements: on the same data embedded in
    complex128 the complex kernel's imaginary parts are exact zeros and x, S and info are bit-equal."""
    set_switches(monkeypatch, {"MF_SWEEP_FORCE_SMEM": 1} if r > 64 else {})
    nf = 7
    ops, br = F64_MODELS["waveguide"](r, m)
    if not with_a1:
        ops[1] = None
    coef = coefficients(frequencies(nf))
    dops, dbr = upload(dv, ops, br)
    xr, sr, ir = run_sweep(dv, dops, dbr, coef, 3)
    xc, sc, ic = run_sweep(dv, [None if d is None else d.to(torch.complex128) for d in dops], dbr.to(torch.complex128), coef, 3)
    assert xr.dtype == np.float64 and xc.dtype == np.complex128
    assert np.array_equal(ir, ic) and not np.any(ir)
    assert np.all(xc.imag == 0) and np.array_equal(xc.real, xr), np.abs(xc.real - xr).max()
    assert np.array_equal(sc, sr), np.abs(sc - sr).max()


@pytest.mark.parametrize("family,r,m", PROPERTY_CASES)
def test_singular_points(dv, monkeypatch, family, r, m):
    """A = E with the real block [[2, 1], [1, 0.5]] at columns k, k+1: the multiplier is exactly 0.5 and the next pivot exactly 0, so
    info = k + 2 as dgetrf reports; k, k+1 straddle an 8-column panel, a 16-row block column and the deepest panel."""
    variant, env = FAMILIES[family]
    set_switches(monkeypatch, env)
    f = np.array([3e9, 4e9, 5e9])
    coef = (np.ones(3), f, f ** 2, np.ones(3), np.ones(3))
    ks = singular_columns(r)
    assert ks
    for k in ks:
        a = singular_block(r, k, float)
        assert lapack.dgetrf(a)[2] == k + 2
        dops, dbr = upload(dv, [a, None, None], np.ones((r, m)))
        _, _, info = run_sweep(dv, dops, dbr, coef, variant, want_gsm=False)
        assert list(info) == [k + 2] * 3, (k, info)


# --------------------------------------------------------------------------------------- per-point state inside one CTA
def abi_sweep(lib, dops, dbr, coef, variant, ws_bytes):
    """mf_sweep_lu_gsm_f64 through ctypes with a workspace of exactly ``ws_bytes`` (the launcher shrinks the grid to fit it)."""
    from morfem_b200 import _ffi
    nf = coef[0].size
    r, m = dbr.shape
    cd = [torch.from_numpy(np.ascontiguousarray(c, dtype=np.float64)).cuda() for c in coef]
    x = torch.empty((nf, r, m), dtype=torch.float64, device="cuda")
    s = torch.empty((nf, m, m), dtype=torch.complex128, device="cuda")
    info = torch.zeros(nf, dtype=torch.int32, device="cuda")
    ws = torch.empty(max(int(ws_bytes), 1), dtype=torch.uint8, device="cuda")
    p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())  # noqa: E731
    _ffi.check(lib.mf_sweep_lu_gsm_f64(p(dops[0]), p(dops[1]), p(dops[2]), dops[0].stride(0), p(dbr), dbr.stride(0), r, m,
                                       *(p(c) for c in cd), nf, p(x), p(s), p(info), variant, p(ws), int(ws_bytes),
                                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "mf_sweep_lu_gsm_f64")
    torch.cuda.synchronize()
    return x.cpu().numpy(), s.cpu().numpy(), info.cpu().numpy()


@pytest.mark.parametrize("cfg,r,m", [(1, 100, 3), (5, 150, 2), (2, 200, 4), (4, 300, 5)])
def test_one_cta_runs_every_point_in_order(dv, lib, monkeypatch, cfg, r, m):
    """A workspace of one slot makes one left-looking CTA run all F = 7 points in a row.  Point 2 is exactly singular; every later
    point must be unaffected by it: info flags point 2 only, the other points pass the checks, and x and S are bit-equal to a run
    with the full workspace."""
    set_switches(monkeypatch, {"MF_LEFT_CFG": cfg})
    assert left_cfg(r, {"MF_LEFT_CFG": cfg}) == cfg
    nf = 7
    ref, (dops, dbr) = case(dv, "waveguide", r, m, nf, 2)
    good = np.array([i for i in range(nf) if i != 2])
    one = lib.mf_sweep_f64_ws_bytes(r, m, 1, 5)
    full = lib.mf_sweep_f64_ws_bytes(r, m, nf, 5)
    assert one < full
    x1, s1, i1 = abi_sweep(lib, dops, dbr, ref.coef, 5, one)
    xf, sf, if_ = abi_sweep(lib, dops, dbr, ref.coef, 5, full)
    assert list(np.flatnonzero(i1)) == [2] and i1[2] == singular_info(r)
    assert np.array_equal(i1, if_)
    check(f"left_cfg{cfg}_one_cta", ref, x1, s1, i1, points=good)
    assert np.array_equal(x1[good], xf[good]) and np.array_equal(s1[good], sf[good])


@pytest.mark.parametrize("r,m", [(190, 3), (256, 4), (512, 2)])
def test_chunked_launches_are_bit_equal(dv, lib, sms, monkeypatch, r, m):
    """R >= 192 cuts a long batch into launches of two points per CTA (MF_LEFT_CHUNK overrides): with F > 2 x resident CTAs the
    results are bit-equal whatever the launch length, and pass the checks."""
    set_switches(monkeypatch, {})
    _, resident = assert_instance(lib, sms, r, m, 0, {})
    nf = 2 * resident + 13
    ref, (dops, dbr) = case(dv, "waveguide", r, m, nf)
    runs = {}
    for chunk in (0, 1, 2):
        set_switches(monkeypatch, {"MF_LEFT_CHUNK": chunk})
        runs[chunk] = run_sweep(dv, dops, dbr, ref.coef, 0)
    check("left_chunked", ref, *runs[2])
    for chunk in (0, 1):
        assert all(np.array_equal(a, b) for a, b in zip(runs[chunk], runs[2])), chunk


# ------------------------------------------------------------------------------------- remap (read once per process)
@pytest.mark.parametrize("r,m", [(128, 4), (200, 3)])
def test_left_looking_remap_in_child_process(dv, tmp_path, r, m):
    """MF_LEFT_REMAP (panel warps of the look-ahead body on their own SM sub-partitions) is read once per process, so it runs in a
    child process: forced on for the 8-warp geometry (cfg 2) with the look-ahead body, at r = 128 (the library's default there) and
    r = 200 (not the default)."""
    nf = 6
    ref, _ = case(dv, "waveguide", r, m, nf)
    ops, br, _ = host_model("waveguide", r, m)
    np.savez(tmp_path / "in.npz", a0=ops[0], a1=ops[1], a2=ops[2], br=br, c=np.array(ref.coef))
    script = textwrap.dedent("""
        import sys, numpy as np, torch
        from morfem_b200 import device as dv
        d = np.load(sys.argv[1])
        ops = [dv.symmetrize(dv.real_or_complex_to_device(d[k])) for k in ("a0", "a1", "a2")]
        c = [torch.from_numpy(np.ascontiguousarray(v)).cuda() for v in d["c"]]
        res = dv.sweep(*ops, dv.real_or_complex_to_device(d["br"]), *c, want_x=True, want_gsm=True, variant=5)
        assert res.x.dtype == torch.float64
        np.savez(sys.argv[2], x=res.x.cpu().numpy(), s=res.gsm.cpu().numpy(), info=res.info.cpu().numpy())
    """)
    env = {k: v for k, v in os.environ.items() if not k.startswith("MF_")}
    env.update(MF_LEFT_REMAP="1", MF_LEFT_CFG="2", MF_LEFT_VER="3")
    out = subprocess.run([sys.executable, "-c", script, str(tmp_path / "in.npz"), str(tmp_path / "out.npz")], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    o = np.load(tmp_path / "out.npz")
    check("left_remap", ref, o["x"], o["s"], o["info"])


# ----------------------------------------------------------------------------------------- fallback and public entry
@pytest.mark.parametrize("r,m", [(513, 2), (700, 3)])
def test_real_operands_beyond_float64_kernels_run_complex(dv, monkeypatch, r, m):
    """No float64 kernel covers r > 512: ``device.sweep`` widens real operands to complex128, whose imaginary parts stay exactly 0."""
    set_switches(monkeypatch, {})
    nf = 4
    ref, (dops, dbr) = case(dv, "waveguide", r, m, nf)
    x, s, info = run_sweep(dv, dops, dbr, ref.coef, 0)
    assert x.dtype == np.complex128 and np.all(x.imag == 0)
    check("fallback_c128", ref, x, s, info)


@pytest.mark.parametrize("r,m", [(40, 3), (150, 2)])
def test_public_entry_with_first_order_term(dv, r, m):
    """``solve_finite_element_method`` on a dense real model with a non-zero a1: float64 result that passes the backward check."""
    from morfem_b200 import implementation as impl
    from oracle import reference_path as orc
    nf = 9
    f = frequencies(nf)
    ops, br = F64_MODELS["waveguide"](r, m)
    md = impl.ModelDefinition(f, *ops, br, lambda t: 1.0, lambda t: t, lambda t: t ** 2, orc.b_coefficient)
    x = impl.solve_finite_element_method(md)
    assert x.dtype == np.float64 and x.shape == (nf, r, m)
    bw = backward_ratios(symmetrised(ops), coefficients(f), br, x)
    assert np.all(bw < THRESH), bw.max()
