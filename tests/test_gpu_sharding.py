"""Sharding properties on the GPU: envs are independent, so running E envs in one launch must
equal, bit for bit, running contiguous shards separately (incl. the Philox noise stream, which
is keyed by the global env id); the additive stats vectors of the shards must sum to the
whole; and with >= 2 GPUs the NCCL all-reduce + lambda update gives every rank the same lambda."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_coverage(starts, actions, lam, gamma, thr, offset=0, fused=False):
    import safe_multiagent_rl_b200 as s
    E, A = starts.shape[:2]
    T = actions.shape[0]
    env = s.BatchedCoverageDiscrete(32, A, n_envs=E, weights=[1.0 + (i % 3) for i in range(A)], starts=starts,
                                    env_offset=offset)
    lam_d = torch.as_tensor(lam, dtype=torch.float64, device="cuda")
    act = torch.as_tensor(actions, device="cuda")
    if fused:
        act_k = torch.zeros(T, A, env.ld, dtype=torch.uint8, device="cuda")
        act_k[:, :, :E] = act.permute(0, 2, 1)
        out = env.rollout(act_k, lambdas=lam_d, gamma=gamma, thresholds=thr, g_mode=1)
    else:
        out = env.rollout_closed_loop(lambda obs, t: act[t], T, lam_d, gamma, thresholds=thr)
    return {k: out[k].cpu().numpy().copy() for k in ("R", "modR", "C", "G")}, out["stats"].vec.cpu().numpy().copy(), \
        env.state().cpu().numpy()


@pytest.mark.parametrize("fused", [False, True])
def test_coverage_shard_invariance(fused):
    rng = np.random.default_rng(0)
    E, A, T = 3000, 16, 20
    starts = rng.integers(0, 32, size=(E, A, 2))
    actions = rng.integers(0, 5, size=(T, E, A)).astype(np.uint8)
    lam, thr = np.linspace(0.1, 0.4, A), np.full(A, 7.0)
    whole, st_whole, pos_whole = run_coverage(starts, actions, lam, 0.999, thr, fused=fused)
    cuts = [0, 1000, 1777, 3000]
    st_sum = 0
    for lo, hi in zip(cuts, cuts[1:]):
        part, st, pos = run_coverage(starts[lo:hi], actions[:, lo:hi], lam, 0.999, thr, offset=lo, fused=fused)
        assert np.array_equal(pos, pos_whole[lo:hi])
        for k in ("R", "modR", "C"):
            assert np.array_equal(part[k], whole[k][lo:hi]), k              # bit-exact, any shard boundary
        assert np.array_equal(part["G"], whole["G"][:, lo:hi])
        st_sum = st_sum + st
    K = A
    assert np.array_equal(st_sum[:2 * K], st_whole[:2 * K]) and st_sum[-1] == st_whole[-1] == E
    np.testing.assert_allclose(st_sum[2 * K:-1], st_whole[2 * K:-1], rtol=1e-12)


def test_congestion_philox_shard_invariance():
    import safe_multiagent_rl_b200 as s
    rng = np.random.default_rng(1)
    E, A, T, size = 1500, 8, 30, 10
    demand = rng.random((size + 1, size + 1)) * 8 + 2
    starts = rng.integers(0, size, size=(E, A, 2)); starts[:, 0] = 0
    actions = rng.integers(0, 5, size=(T, E, A)).astype(np.uint8)

    def run(lo, hi):
        env = s.BatchedCongestion(size, A, n_envs=hi - lo, noise=0.2, starts=starts[lo:hi], demand_rate=demand,
                                  seed=99, env_offset=5_000_000_000 + lo)      # ids beyond 2^32 exercise the high word
        env.reset()
        rs, cs = [], []
        for t in range(T):
            _, r, c, _ = env.step(actions[t, lo:hi])
            rs.append(r.cpu().numpy().copy()); cs.append(c.cpu().numpy().copy())
        return env.state().cpu().numpy(), np.stack(rs), np.stack(cs)
    pos, r, c = run(0, E)
    for lo, hi in [(0, 500), (500, 501), (501, 1500)]:
        p2, r2, c2 = run(lo, hi)
        assert np.array_equal(p2, pos[lo:hi]) and np.array_equal(r2, r[:, lo:hi]) and np.array_equal(c2, c[:, lo:hi])


def _nccl_worker(rank, world, port, q, abi_comm=False):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200 import dist as sd
    sd.init_from_env(backend="nccl")
    rng = np.random.default_rng(0)
    E, A, T = 2001, 3, 25
    starts = rng.integers(0, 5, size=(E, A, 2))
    actions = rng.integers(0, 5, size=(T, E, A)).astype(np.uint8)
    off, n = sd.shard_range(E, rank, world)
    env = s.BatchedCoverageDiscrete(5, A, n_envs=n, weights=[1.0, 2.0, 3.0], starts=starts[off:off + n], env_offset=off)
    comm = sd.StatsComm.from_process_group() if abi_comm else None     # smarl_comm_* / smarl_stats_allreduce
    meta = s.BatchedMetaAgent([1] * A, 0.999, 0.05, [10.0] * A, start_learning_cycle=0, lambda_0=0.2, n_agents=A,
                              comm=comm)
    act = torch.as_tensor(actions[:, off:off + n], device="cuda")
    out = env.rollout_closed_loop(lambda obs, t: act[t], T, meta.lambdas, 0.999, thresholds=[10.0] * A)
    meta.step(out["stats"])
    glob = meta.global_stats().cpu().numpy()
    meta.update()
    q.put((rank, glob, meta.lambdas.cpu().numpy()))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


def test_abi_communicator_single_rank_is_the_identity():
    """smarl_comm_get_unique_id / _init_from_unique_id / smarl_stats_allreduce on one GPU: NCCL is loaded by
    libsmarl itself (dlopen) and a one-rank all-reduce leaves the vector as it is."""
    from safe_multiagent_rl_b200 import _lib
    from safe_multiagent_rl_b200 import dist as sd
    assert _lib.load().smarl_comm_nccl_version() >= 20000
    comm = sd.StatsComm.from_process_group()
    v = torch.arange(13, dtype=torch.float64, device="cuda") * 1.5
    want = v.clone()
    sd.allreduce_stats(v, comm=comm)
    graph = torch.cuda.CUDAGraph()                      # the call is capturable: no host sync
    torch.cuda.synchronize()
    with torch.cuda.graph(graph):
        comm.allreduce(v)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(v, want)
    comm.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("abi_comm", [False, True])
def test_two_gpu_nccl_lambda_update_matches_oracle(abi_comm):
    import torch.multiprocessing as mp
    from oracle import numpy_oracle as no
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 2000 + (7 if abi_comm else 0)
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q, abi_comm)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    rng = np.random.default_rng(0)
    E, A, T = 2001, 3, 25
    starts = rng.integers(0, 5, size=(E, A, 2))
    actions = rng.integers(0, 5, size=(T, E, A))
    lut = no.coverage_penalty_lut(5, no.coverage_fieldview(5, A))
    pos = starts.copy()

    def step_fn(t):
        nonlocal pos
        pos, r, c, _ = no.coverage_discrete_step(pos, actions[t], 5, lut, [1.0, 2.0, 3.0])
        return r, c
    want = no.rollout(step_fn, T, 0.999, [0.2] * A)
    lam_want = no.lambda_update([0.2] * A, want["C"].mean(0), [10.0] * A, 0.05)
    for rank, glob, lam in got:
        assert np.array_equal(glob[:A], want["C"].sum(0)) and glob[-1] == E
        np.testing.assert_allclose(glob[2 * A:3 * A], want["R"].sum(0), rtol=1e-5)
        np.testing.assert_allclose(lam, lam_want, rtol=1e-14)
    assert np.array_equal(got[0][2], got[1][2])                   # bit-identical lambda on both ranks
