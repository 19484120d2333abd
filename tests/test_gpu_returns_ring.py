"""smarl_rollout_returns against a float64 torch reference, at the edges of returns_kernel's shared-memory ring:
horizons around its depth (including T shorter than the ring), ragged tail chunks, every cost dtype and g_mode,
with and without a penalty row and stats.  Every buffer sits in a guarded arena, so a bulk copy or store past the
end of a row shows up as an overrun."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_gpu_bounds import Arena

pytestmark = pytest.mark.gpu
RTOL = 1e-5
STAGES = 6          # kReturnsStages in csrc/returns.cu
GAMMA = 0.99
COST = {"u8": (0, torch.uint8), "i32": (1, torch.int32), "f32": (2, torch.float32)}


def close(got, want, scale):
    np.testing.assert_allclose(np.asarray(got, np.float64), want, rtol=RTOL, atol=RTOL * scale + 1e-30)


def _cases():
    """Every horizon meets every tail chunk once (T x E), the other axes on independent indices."""
    Ts = [1, STAGES - 1, STAGES, STAGES + 1, 50, 300]
    Es = [1, 5, 37, 511, 513, 1001]
    AKs = [(1, 1), (3, 2), (16, 16), (32, 5)]
    dts = ["u8", "i32", "f32"]
    out = []
    for i, (T, E) in enumerate((T, E) for T in Ts for E in Es):
        A, K = AKs[(i + i // 6) % 4]
        out.append((T, E, A, K, dts[(i // 2 + i // 6) % 3], (i // 3) % 2 == 0, (i + i // 4) % 4, (i // 5) % 2 == 0,
                    i % 7 != 3))
    return out


def reference(rew, cost, pen, n_act, g_mode, T):
    """rew [T][A][E], cost [T][K][E], pen [T][E] or None (float64, on the GPU); returns R, modR, C, G."""
    m = rew - (pen[:, None, :] if pen is not None else 0.0)
    disc = GAMMA ** torch.arange(T, dtype=torch.float64, device=rew.device)[:, None, None]
    R = (disc * rew).sum(0)
    Cs = cost.sum(0)
    rtg = torch.zeros_like(m)
    run = torch.zeros_like(m[0])
    for t in range(T - 1, -1, -1):
        run = m[t] + GAMMA * run
        rtg[t] = run
    M = rtg[0]
    if g_mode == 1:
        G = rtg
    elif g_mode == 2:
        G = disc * m
    elif g_mode == 3:
        n = n_act.clamp(0, T).to(torch.float64)                                   # [E]
        mask = torch.arange(T, device=rew.device)[:, None, None] < n[None, None, :]
        s = (rtg * mask).sum(0)
        sq = (rtg * rtg * mask).sum(0)
        mean = s / n
        var = (sq - n * mean * mean) / (n - 1.0)
        inv = 1.0 / (var.clamp(min=0.0).sqrt() + 1e-7)
        inv = torch.where(n < 2, torch.full_like(inv, float("nan")), inv)
        G = torch.where(mask, (rtg - mean) * inv, torch.zeros_like(rtg))
    else:
        G = None
    return R, M, Cs, G


@pytest.mark.parametrize("T,E,A,K,cdt,with_pen,g_mode,with_stats,with_n_active", _cases())
def test_rollout_returns_ring(T, E, A, K, cdt, with_pen, g_mode, with_stats, with_n_active):
    from safe_multiagent_rl_b200 import _lib
    lib = _lib.load()
    P = _lib.ptr
    st = torch.cuda.current_stream().cuda_stream
    ld = (E + 15) // 16 * 16
    code, cdtype = COST[cdt]
    g = torch.Generator(device="cuda"); g.manual_seed(T * 1000 + E)
    f32, f64, i32 = torch.float32, torch.float64, torch.int32
    ar = Arena()
    rew = ar.make(T * A, ld, f32, torch.randn(T * A, ld, generator=g, device="cuda"))
    cost = ar.make(T * K, ld, cdtype, torch.randint(0, 3, (T * K, ld), generator=g, device="cuda").to(cdtype))
    pen = ar.make(T, ld, f32, torch.rand(T, ld, generator=g, device="cuda")) if with_pen else None
    n_act = None
    if g_mode == 3 and with_n_active:
        n_act = ar.make(1, ld, i32, torch.randint(0, T + 2, (1, ld), generator=g, device="cuda", dtype=i32))
    R, M, Cs = ar.make(A, ld, f32), ar.make(A, ld, f32), ar.make(K, ld, i32)
    G = ar.make(T * A, ld, f32) if g_mode else None
    thr_val = 1.0 * T
    thr = ar.make(1, K, f64, torch.full((1, K), thr_val, device="cuda", dtype=f64))
    stats = scratch = None
    if with_stats:
        stats = ar.make(1, lib.smarl_stats_len(A, K), f64)
        scratch = ar.make(1, lib.smarl_stats_scratch_len(A, K, E), f64)
    acc = _lib.Accounting(GAMMA, T, g_mode, P(thr))
    _lib.check(lib.smarl_rollout_returns(C.byref(acc), P(rew), P(cost), code, P(pen), P(n_act), P(R), P(M), P(Cs),
                                         P(G), P(stats), P(scratch), A, K, E, ld, st))
    torch.cuda.synchronize()
    ar.check()

    rw = rew.view(T, A, ld)[:, :, :E].to(f64)
    cw = cost.view(T, K, ld)[:, :, :E].to(f64)
    pw = pen[:, :E].to(f64) if with_pen else None
    na = n_act[0, :E].to(torch.int64) if n_act is not None else torch.full((E,), T, device="cuda")
    wR, wM, wC, wG = reference(rw, cw, pw, na, g_mode, T)
    scale = float(rw.abs().max()) * T + 1.0
    close(R[:, :E].cpu(), wR.cpu().numpy(), scale)
    close(M[:, :E].cpu(), wM.cpu().numpy(), scale)
    got_C = Cs[:, :E]
    if cdt == "f32":
        got_C = got_C.view(f32)
    assert torch.equal(got_C.to(f64), wC), "C differs"
    if g_mode:
        gG = G.view(T, A, ld)[:, :, :E].cpu().numpy().astype(np.float64)
        want = wG.cpu().numpy()
        assert np.array_equal(np.isnan(gG), np.isnan(want))
        ok = ~np.isnan(want)
        close(gG[ok], want[ok], float(np.abs(want[ok]).max(initial=0.0)) + 1.0)
    if with_stats:
        s = stats[0].cpu().numpy()
        assert np.array_equal(s[:K], wC.sum(1).cpu().numpy())
        assert np.array_equal(s[K:2 * K], (wC > thr_val).sum(1).to(f64).cpu().numpy())
        assert s[2 * K + 2 * A] == E
        close(s[2 * K:2 * K + A], wR.sum(1).cpu().numpy(), scale * E)
        close(s[2 * K + A:2 * K + 2 * A], wM.sum(1).cpu().numpy(), scale * E)
