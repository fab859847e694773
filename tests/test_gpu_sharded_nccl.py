"""
The N > 1 path on the hardware: two NCCL ranks (one process per GPU) shard a batch of independent
problems through vgpa_b200.ensemble.ShardedEnsemble with the CUDA BatchEvaluator, gather F (host path:
numpy F moved to the device for NCCL; device path: eval_device + gather_device), and the result must
equal the single-GPU evaluation BIT FOR BIT (SURVEY.md 8e).  Skipped on a box with one GPU
(`gpurun --gpus 2`).
"""
import os
import socket
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu


def _problems(total):
    g = np.load(GOLDEN / "eval_L63_rk2.npz")
    rng = np.random.default_rng(7)
    obs_y = np.stack([g["obs_y"] + 0.05 * rng.standard_normal(g["obs_y"].shape) for _ in range(total)])
    sigma = np.stack([g["sigma"] * (0.8 + 0.03 * p) for p in range(total)])
    X = np.stack([g["x"] * (1.0 + 0.01 * rng.standard_normal(g["x"].size)) for _ in range(total)])
    return g, obs_y, sigma, X


def _evaluator(g, obs_y, sigma, lo, hi, device):
    from oracle import prior_kl0
    from vgpa_b200.engine import BatchEvaluator
    E0 = prior_kl0(g["m0"], g["s0"], g["mu0"], g["tau0"], False)
    return BatchEvaluator(model="L63", method="rk2", N=int(g["N"]), dt=float(g["dt"]), theta=g["theta"],
                          sigma=sigma[lo:hi], R=g["R"], obs_t=g["obs_t"], obs_y=obs_y[lo:hi], m0=g["m0"], s0=g["s0"],
                          E0=E0, B=hi - lo, dt_model=float(g["dt"]), device=device)


def _worker(rank, world, port, total, out_dir):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    import torch
    import torch.distributed as dist
    from vgpa_b200.ensemble import ShardedEnsemble
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    g, obs_y, sigma, X = _problems(total)
    ens = ShardedEnsemble(total, lambda lo, hi: _evaluator(g, obs_y, sigma, lo, hi, rank))
    F_all, G_local = ens.eval(X[ens.lo:ens.hi])                     # host buffers; F goes through the device for NCCL
    Xd = torch.from_numpy(X[ens.lo:ens.hi]).cuda()
    Fd = torch.empty(ens.hi - ens.lo, dtype=torch.float64, device="cuda")
    Gd = torch.empty_like(Xd)
    ens.eval_device(Xd, Fd, Gd, torch.cuda.current_stream().cuda_stream)
    F_dev = ens.gather_device(Fd).cpu().numpy()
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), F=F_all, F_dev=F_dev, G=G_local, G_dev=Gd.cpu().numpy(),
             lo=ens.lo, hi=ens.hi)
    ens.evaluator.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("total", [8, 9])
def test_two_rank_nccl_matches_single_gpu(tmp_path, total):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, total, str(tmp_path)), nprocs=2, join=True)
    g, obs_y, sigma, X = _problems(total)
    with _evaluator(g, obs_y, sigma, 0, total, 0) as ev:
        F_ref, G_ref = ev.eval(X)
    for r in range(2):
        z = np.load(tmp_path / f"rank{r}.npz")
        lo, hi = int(z["lo"]), int(z["hi"])
        assert np.array_equal(z["F"], F_ref) and np.array_equal(z["F_dev"], F_ref)     # bit for bit, on every rank
        assert np.array_equal(z["G"], G_ref[lo:hi]) and np.array_equal(z["G_dev"], G_ref[lo:hi])


def _scg_worker(rank, world, port, total, out_dir):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    import torch
    import torch.distributed as dist
    from vgpa_b200.batched_scg import ShardedBatchedSCG
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    g, obs_y, sigma, _ = _problems(total)
    opts = {"max_it": 20, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    ens = ShardedBatchedSCG(total, lambda lo, hi: _evaluator(g, obs_y, sigma, lo, hi, rank), opts, sub_batch=3)
    res = ens.run(keep=(0, total - 1))
    np.savez(os.path.join(out_dir, f"scg_rank{rank}.npz"), fx=res["fx"], n_it=res["n_it"], f_eval=res["f_eval"],
             kept_keys=np.array(sorted(res["kept"]), dtype=np.int64))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharded_scg_matches_single_gpu(tmp_path):
    """The device-resident ensemble OPTIMISATION sharded over two NCCL ranks (sub-batches of 3 problems):
    every rank ends with the fx / iteration counts of the whole ensemble, equal to one BatchedSCG over
    all problems on one GPU."""
    import torch
    import torch.multiprocessing as mp
    from vgpa_b200.batched_scg import BatchedSCG
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    total = 9
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_scg_worker, args=(2, port, total, str(tmp_path)), nprocs=2, join=True)
    g, obs_y, sigma, _ = _problems(total)
    opts = {"max_it": 20, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    with _evaluator(g, obs_y, sigma, 0, total, 0) as ev:
        opt = BatchedSCG(ev, opts)
        _, fx = opt(ev.initialization(0.0))
        n_it = opt.stats["MaxIt"].copy()
    for r in range(2):
        z = np.load(tmp_path / f"scg_rank{r}.npz")
        assert np.allclose(z["fx"], fx, rtol=1e-12) and np.array_equal(z["n_it"], n_it)
    assert list(np.load(tmp_path / "scg_rank0.npz")["kept_keys"]) == [0]        # each rank keeps its own problems
    assert list(np.load(tmp_path / "scg_rank1.npz")["kept_keys"]) == [total - 1]
