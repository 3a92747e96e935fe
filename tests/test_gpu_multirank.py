"""Multi-rank parity of the row-/point-sharded hot path (SURVEY.md 8e) on GPU hardware.

Two layers:

* ``test_sharded_arithmetic_emulated_on_one_gpu`` needs ONE GPU: the ranks of a 2/3/4-way job are played one after the
  other on the same device -- each rank's operator rows uploaded with window-relative column indices
  (``csr_of_transpose(row_range=, col_offset=)``), the halo-window SpMM, the r x r Gram / projection partials and the
  port-matrix partials -- and their sum is compared with the CPU oracle (what the all-reduce would deliver).
* ``test_multirank_nccl_matches_oracle`` spawns one process per GPU (NCCL) and runs ``ShardedHotPath`` -- eager with the
  point-to-point halo, eager with the slab all-gather halo, and replayed from a CUDA graph -- and rank 0 compares the
  gathered S-parameters and the reduced operators with the CPU oracle.  Skipped on a machine with fewer GPUs than ranks
  (logs of 2- and 4-GPU runs under profiles/).
"""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import reference_path as orc   # noqa: E402  (checker only)

EPS = np.finfo(float).eps


def _model(grid=(6, 5, 60), r=24, m=2, nf=96, seed=3):
    from scipy.sparse import csc_array
    from morfem_b200 import synthetic
    ct, tt = synthetic.waveguide_operators(*grid)
    n = ct.shape[0]
    wp = synthetic.port_matrix(n, m, 19)
    in_c, in_gamma, in_b = synthetic.driver_scaled(ct, tt, wp)
    f = synthetic.frequency_points(nf)
    s = synthetic.snapshot_matrix(n, r, seed=seed, decay_decades=3.0)
    return in_c, csc_array(in_c.shape), in_gamma, in_b, f, s, n


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("real", [False, True])
def test_sharded_arithmetic_emulated_on_one_gpu(world, real):
    from morfem_b200 import device as dv, dist as mfd
    dev = dv.require_cuda()
    in_c, a1, in_gamma, in_b, f, s, n = _model()
    q_host = orc.orthonormal_basis(s)
    r = q_host.shape[1]
    x = dv.real_or_complex_to_device(q_host, dev, widen=not real)
    gram = torch.zeros((r, r), dtype=x.dtype, device=dev)
    proj = {0: torch.zeros((r, r), dtype=x.dtype, device=dev), 2: torch.zeros((r, r), dtype=x.dtype, device=dev)}
    bt = torch.zeros((r, in_b.shape[1]), dtype=x.dtype, device=dev)
    b_dev = dv.csc_to_device(in_b, dev)
    halo_rows = 0
    for rank in range(world):
        row0, row1 = mfd.even_split(n, world, rank)
        x_loc = x[row0:row1].contiguous()
        gram += dv.gemm_tn(x_loc, x_loc, conj=True)
        for i, a in ((0, in_c), (2, in_gamma)):
            window = mfd.column_window(np.asarray(a.indptr), np.asarray(a.indices), row0, row1, n)
            windows = [mfd.column_window(np.asarray(a.indptr), np.asarray(a.indices), *mfd.even_split(n, world, p), n) for p in range(world)]
            plan = mfd.build_halo_plan(rank, world, n, windows)
            assert (plan.win0, plan.win1) == window
            halo_rows += plan.halo_rows
            csr = dv.csr_of_transpose(a, dev, row_range=(row0, row1), col_offset=plan.win0)
            win = x[plan.win0:plan.win1].contiguous()            # what the halo exchange assembles on this rank
            y = dv.spmm(csr, win)
            if rank == 1:
                dv.group_rows(csr, r, real=real)                 # the row-grouped operand on a window as well
                y2 = dv.spmm(csr, win)
                assert torch.allclose(y, y2, rtol=1e-13, atol=0)
            proj[i] += dv.gemm_tn(y, x_loc, conj=False)
        bt += dv.project_rhs(b_dev, x_loc, row0, conj=False)
    assert halo_rows > 0
    torch.cuda.synchronize()
    ref = orc.galerkin_projection(q_host, in_c, a1, in_gamma, in_b)
    assert orc.rel_err(gram.cpu().numpy(), q_host.T @ q_host) < 1e-12
    assert orc.rel_err(proj[0].cpu().numpy(), ref[0]) < 1e-12
    assert orc.rel_err(proj[2].cpu().numpy(), ref[2]) < 1e-12
    assert orc.rel_err(bt.cpu().numpy(), ref[3]) < 1e-12
    if not real:
        assert float(proj[0].imag.abs().max()) == 0.0


# ------------------------------------------------------------------------------------------- real NCCL ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from scipy.constants import pi, epsilon_0
    from morfem_b200 import device as dv, dist as mfd, implementation as impl, test_helpers as th
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        in_c, a1, in_gamma, in_b, f, s, n = _model(grid=(8, 6, 120), r=48, m=3, nf=257)
        cb = impl.coefficient_array(th.b_coefficient, f)
        coeffs = [np.ones_like(f), f, f ** 2, cb, 2 * pi * f * epsilon_0]
        ref = None
        if rank == 0:
            q = orc.orthonormal_basis(s)
            red = orc.galerkin_projection(q, in_c, a1, in_gamma, in_b)
            x_ref = orc.reduced_sweep(f, red[0], red[1], red[2], red[3], lambda t: 1.0, lambda t: t, lambda t: t ** 2, orc.b_coefficient)
            s_ref = orc.scattering_sweep(f, x_ref, red[3])
            cond = np.array([np.linalg.cond(orc.system_matrix(1.0, t, t ** 2, red[0], red[1], red[2])) for t in f])
            sv = np.linalg.svd(s, compute_uv=False)
            ref = (q, red, s_ref, np.maximum(1e-10, 50 * EPS * np.maximum(cond, sv[0] / sv[-1])), sv)
        row0, row1 = mfd.even_split(n, world, rank)
        results = {}
        for real in (False, True):
            s_dev = dv.real_or_complex_to_device(s[row0:row1], dev, widen=not real)
            for mode in ("allgather", "p2p", "graph"):
                path = mfd.ShardedHotPath([in_c, a1, in_gamma], in_b, n, f.size, coeffs)
                assert path.halo_mode == "allgather" and path.halo_h > 0          # banded model: the slab exchange applies
                if mode == "p2p":
                    path.halo_mode = "p2p"
                if mode == "graph":
                    for _ in range(3):                                            # replays overwrite the static outputs
                        gsm, qd, red_d, res = path.step_graph(s_dev, want_x=False)
                    assert path.verify() is None
                else:
                    gsm, qd, red_d, res = path.step(s_dev, want_x=False, gather=True)
                torch.cuda.synchronize()
                assert gsm.shape == (f.size, 3, 3)
                if rank == 0:
                    q_ref, red, s_ref, tol, sv = ref
                    err = np.linalg.norm((gsm.cpu().numpy() - s_ref).reshape(f.size, -1), axis=1) / np.linalg.norm(s_ref.reshape(f.size, -1), axis=1)
                    assert np.all(err < tol), (mode, real, err.max(), tol.max())
                    # the gathered basis rows of this rank against the oracle's subspace, reduced operators aligned with it
                    q_loc = qd.cpu().numpy()
                    results[(mode, real)] = (float(err.max()), float((err / tol).max()))
                # every rank holds the same reduced model (replicated r x r factorisations, all-reduced partials)
                a0_r = red_d[0].contiguous()
                chk = [torch.empty_like(a0_r) for _ in range(world)]
                dist.all_gather(chk, a0_r)
                assert all(torch.equal(c, chk[0]) for c in chk)
                # the basis is row-sharded: gather it and compare the subspace with the oracle's
                qs = [torch.empty((mfd.even_split(n, world, p)[1] - mfd.even_split(n, world, p)[0], qd.shape[1]), dtype=qd.dtype, device=dev)
                      for p in range(world)]
                dist.all_gather(qs, qd.contiguous())
                if rank == 0:
                    q_all = torch.cat(qs, dim=0).cpu().numpy()
                    span_tol = max(1e-10, 50 * EPS * ref[4][0] / ref[4][-1])
                    assert orc.subspace_residual(ref[0], q_all) < span_tol
                    a0_ref = orc.align_reduced(ref[1][0], ref[0], np.ascontiguousarray(q_all.real))
                    assert orc.rel_err(red_d[0].cpu().numpy().real, a0_ref) < max(1e-10, 10 * span_tol)
                del path
        if rank == 0:
            with open(os.path.join(out_dir, "result.txt"), "w") as fh:
                for k, v in results.items():
                    fh.write(f"{k}: max_rel_err {v[0]:.3e} worst_err_over_tol {v[1]:.3f}\n")
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("world", [2, 4])
def test_multirank_nccl_matches_oracle(tmp_path, world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    import torch.multiprocessing as mp
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))
    print(open(tmp_path / "result.txt").read())
