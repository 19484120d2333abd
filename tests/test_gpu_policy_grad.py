"""smarl_policy_grad_discrete / policy_gradient_loss: the REINFORCE loss of the DiscretePolicy (agent.py:23-47, loss
agent.py:134-157) and its fc1 / fc2 gradients in one kernel, against a float64 autograd of the same loss on the same
records and psi.  A result g is accepted when max|g - g64| <= max(4 max|g_torch32 - g64|, 1e-6 max|g64|) for every
parameter tensor (g_torch32: the PyTorch path, log_prob per step and autograd), and the loss when it is within
1e-5 mean|psi log pi| of the float64 loss."""
import ctypes as C
import importlib.util
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUARD = 4096


def make(kind, A, E, seed=0):
    """An on-policy env of `kind` and its fused policy, with logits wide enough that every action has real mass."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy, FusedDiscretizedPolicy
    if kind == "coverage":
        env = s.BatchedCoverageDiscrete(5, A, n_envs=E, shuffle=True, seed=seed)
        cls = FusedDiscretePolicy
    elif kind == "congestion":
        env = s.BatchedCongestionOnPolicy(3, A, n_envs=E, noise=0.1, shuffle=True, seed=seed)
        cls = FusedDiscretePolicy
    else:
        env = s.BatchedCoverageDiscretizedOnPolicy(5, A, n_envs=E, coarseness=6, shuffle=True, seed=seed)
        cls = FusedDiscretizedPolicy
    torch.manual_seed(seed)
    pol = cls(env, seed=99 + seed)
    with torch.no_grad():
        pol.fc1.weight.mul_(0.5)
        pol.fc2.weight.mul_(4.0)
    return env, pol


def records(kind, A, E, T, seed=0):
    env, pol = make(kind, A, E, seed)
    out = env.policy_rollout(pol, T)
    g = torch.Generator(device="cuda").manual_seed(seed)
    psi = torch.randn(T, A, E, generator=g, device="cuda")           # mixed signs
    return env, pol, out, psi


def synthetic(A, NA, E, T, seed=0):
    """Records of the right layout for agent counts the one-launch rollouts do not run (A >= 9): uniform positions in
    the grid and uniform actions."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy, FusedDiscretizedPolicy
    if NA == 5:
        env = s.BatchedCoverageDiscrete(5, A, n_envs=E)
        pol = FusedDiscretePolicy(env)
    else:
        env = s.BatchedCoverageDiscretized(5, A, n_envs=E, coarseness=6)
        pol = FusedDiscretizedPolicy(env)
    torch.manual_seed(seed)
    with torch.no_grad():
        for p in pol.parameters():
            p.copy_(torch.randn_like(p) * 0.5)
    g = torch.Generator(device="cuda").manual_seed(seed)
    ld = env.ld
    obs_ = torch.zeros(T, 2 * A, ld, device="cuda")
    obs_[:, :, :E] = torch.randint(0, 6, (T, 2 * A, E), generator=g, device="cuda").float()
    act_ = torch.zeros(T, A, ld, dtype=torch.uint8, device="cuda")
    act_[:, :, :E] = torch.randint(0, NA, (T, A, E), generator=g, device="cuda", dtype=torch.uint8)
    out = {"obs_": obs_, "actions_": act_, "obs": obs_[:, :, :E].permute(0, 2, 1), "actions": act_[:, :, :E]}
    psi = torch.randn(T, A, E, generator=g, device="cuda")
    return env, pol, out, psi


def reference(pol, out, psi, scale, dtype):
    """Loss and gradients of -scale sum psi log pi(a|s) through the policy in `dtype` (autograd), step chunks summed."""
    params = [p.detach().to(dtype).requires_grad_() for p in (pol.fc1.weight, pol.fc1.bias, pol.fc2.weight,
                                                                pol.fc2.bias)]
    T = psi.shape[0]
    grads = [torch.zeros_like(p) for p in params]
    loss, mag = 0.0, 0.0
    step = max(1, (1 << 22) // (psi.shape[1] * psi.shape[2]))
    for t0 in range(0, T, step):
        obs = out["obs"][t0:t0 + step].to(dtype)                          # [t, E, S]
        act = out["actions"][t0:t0 + step].long()                         # [t, A, E]
        h = F.relu(torch.matmul(obs[:, None], params[0]) + params[1])     # [t, A, E, 16]
        lp = F.log_softmax(torch.matmul(h, params[2]) + params[3], -1).gather(-1, act[..., None]).squeeze(-1)
        term = psi[t0:t0 + step].to(dtype) * lp
        chunk = -scale * term.sum()
        for g, d in zip(grads, torch.autograd.grad(chunk, params)):
            g += d
        loss += float(chunk)
        mag += float(term.abs().sum())
    return [g.float() if dtype == torch.float32 else g for g in grads], loss, mag / psi.numel()


def torch32(pol, out, psi):
    """The PyTorch path the kernel replaces: log_prob per step, the loss and autograd, in f32."""
    T = psi.shape[0]
    pol.zero_grad()
    logp = torch.stack([pol.log_prob(out["obs"][t], out["actions"][t].long()) for t in range(T)])
    (-(logp * psi).mean()).backward()
    return [p.grad.clone() for p in (pol.fc1.weight, pol.fc1.bias, pol.fc2.weight, pol.fc2.bias)]


def fused(pol, out, psi, scale=None):
    pol.zero_grad()
    loss = pol.policy_gradient_loss(out, psi, scale)
    loss.backward()
    return [p.grad.clone() for p in (pol.fc1.weight, pol.fc1.bias, pol.fc2.weight, pol.fc2.bias)], float(loss.detach())


def check(pol, out, psi):
    T, A, E = psi.shape
    got, loss = fused(pol, out, psi)
    g64, l64, mag = reference(pol, out, psi, 1.0 / (T * A * E), torch.float64)
    g32 = torch32(pol, out, psi)
    for name, g, want, base in zip(("w1", "b1", "w2", "b2"), got, g64, g32):
        err = float((g.double() - want).abs().max())
        tol = max(4 * float((base.double() - want).abs().max()), 1e-6 * float(want.abs().max()))
        assert err <= tol, (name, err, tol)
    assert abs(loss - l64) <= 1e-5 * mag, (loss, l64, mag)
    return got


CASES = [(1, 1, 1), (3, 50, 50), (5, 4099, 300), (8, 65536, 50), (3, 65536, 300), (8, 50, 1), (1, 4099, 50)]


@pytest.mark.parametrize("kind", ["coverage", "congestion", "discretized"])
@pytest.mark.parametrize("A,E,T", CASES)
def test_rollout_records_match_float64(kind, A, E, T):
    if kind == "coverage":
        T = min(T, 255)                          # CoverageDiscrete's one launch keeps byte cost counters
    env, pol, out, psi = records(kind, A, E, T, seed=A + E + T)
    if E * T >= 65536 * 50:                      # every action value occurs
        na = pol.n_actions
        assert int(torch.bincount(out["actions"].flatten().long(), minlength=na).min()) > 0
    check(pol, out, psi)


@pytest.mark.parametrize("NA", [5, 9])
@pytest.mark.parametrize("A,E,T", [(9, 300, 7), (16, 1000, 20), (32, 4099, 5), (32, 17, 50)])
def test_synthetic_records_match_float64(A, NA, E, T):
    env, pol, out, psi = synthetic(A, NA, E, T, seed=A * NA)
    check(pol, out, psi)


@pytest.mark.parametrize("NA", [5, 9])
def test_zero_psi_gives_exact_zeros(NA):
    env, pol, out, psi = synthetic(3, NA, 1000, 10)
    got, loss = fused(pol, out, torch.zeros_like(psi))
    assert loss == 0.0 and all(bool((g == 0).all()) for g in got)


@pytest.mark.parametrize("kind", ["coverage", "discretized"])
def test_dead_unit_gets_zero_fc1_gradient(kind):
    env, pol, out, psi = records(kind, 3, 4099, 20)
    with torch.no_grad():
        pol.fc1.weight[:, :, 5] = 0.0
        pol.fc1.bias[:, :, 5] = 0.0                 # h == 0 for every sample
    got = check(pol, out, psi)
    assert bool((got[0][:, :, 5] == 0).all()) and bool((got[1][:, :, 5] == 0).all())
    assert bool((got[2][:, 5, :] == 0).all())        # r == 0 too


def c_call(pol, obs_, act_, psi_, T, E, scale, outs=None):
    """The C ABI on preallocated outputs: (dw1, db1, dw2, db2, loss, scratch)."""
    from safe_multiagent_rl_b200 import _lib
    A, NA, ld = pol.fc1.weight.shape[0], pol.n_actions, obs_.shape[2]
    if outs is None:
        n = pol.lib.smarl_policy_grad_scratch_len(A, NA, T, E)
        outs = [torch.empty_like(p) for p in (pol.fc1.weight, pol.fc1.bias, pol.fc2.weight, pol.fc2.bias)]
        outs += [torch.empty((), dtype=torch.float64, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")]
    p = pol.c_params(pol.env)
    _lib.check(pol.lib.smarl_policy_grad_discrete(C.byref(p), _lib.ptr(obs_), _lib.ptr(act_), _lib.ptr(psi_), T, scale,
                                                  *[_lib.ptr(o) for o in outs], E, ld, _lib.stream_ptr()))
    return outs


def slab(psi, ld, fill=0.0):
    T, A, E = psi.shape
    s = torch.full((T, A, ld), fill, device="cuda")
    s[:, :, :E] = psi
    return s


@pytest.mark.parametrize("kind", ["congestion", "discretized"])
def test_padding_columns_are_never_read(kind):
    env, pol, out, psi = records(kind, 3, 4099, 30)
    T, A, E = psi.shape
    clean = [o.clone() for o in c_call(pol, out["obs_"], out["actions_"], slab(psi, env.ld), T, E, 0.01)[:5]]
    obs_, act_ = out["obs_"].clone(), out["actions_"].clone()
    obs_[:, :, E:] = float("nan")
    act_[:, :, E:] = 255
    dirty = c_call(pol, obs_, act_, slab(psi, env.ld, float("nan")), T, E, 0.01)[:5]
    for a, b in zip(clean, dirty):
        assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a.view(torch.int64),
                           b.view(torch.int32) if b.dtype == torch.float32 else b.view(torch.int64))


def test_repeatable_and_graph_replay():
    env, pol, out, psi = records("coverage", 3, 65536, 50)
    T, A, E = psi.shape
    ps = slab(psi, env.ld)
    first = [o.clone() for o in c_call(pol, out["obs_"], out["actions_"], ps, T, E, 1.0 / (T * A * E))[:5]]
    outs = c_call(pol, out["obs_"], out["actions_"], ps, T, E, 1.0 / (T * A * E))
    for a, b in zip(first, outs[:5]):
        assert torch.equal(a, b)
    for o in outs[:5]:
        o.fill_(7.0)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
        c_call(pol, out["obs_"], out["actions_"], ps, T, E, 1.0 / (T * A * E), outs)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        for o in outs[:5]:
            o.fill_(7.0)
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(first, outs[:5]):
            assert torch.equal(a, b)


def test_half_shards_sum_to_the_whole():
    env, pol, out, psi = records("congestion", 3, 8192, 40)
    T, A, E = psi.shape
    scale = 1.0 / (T * A * E)
    whole = c_call(pol, out["obs_"], out["actions_"], slab(psi, env.ld), T, E, scale)
    h = E // 2
    parts = []
    for lo in (0, h):
        o = c_call(pol, out["obs_"][:, :, lo:lo + h].contiguous(), out["actions_"][:, :, lo:lo + h].contiguous(),
                   psi[:, :, lo:lo + h].contiguous(), T, h, scale)
        parts.append([x.clone() for x in o[:5]])
    g64, l64, mag = reference(pol, out, psi, scale, torch.float64)
    g32 = torch32(pol, out, psi)
    for i, (want, base) in enumerate(zip(g64, g32)):
        tol = max(4 * float((base.double() - want).abs().max()), 1e-6 * float(want.abs().max()))
        assert float(((parts[0][i] + parts[1][i]).double() - want).abs().max()) <= tol
        assert float((whole[i].double() - want).abs().max()) <= tol
    assert abs(float(parts[0][4] + parts[1][4]) - l64) <= 1e-5 * mag


def test_backward_fills_and_accumulates_grad():
    env, pol, out, psi = records("discretized", 3, 4099, 20)
    T, A, E = psi.shape
    want = c_call(pol, out["obs_"], out["actions_"], slab(psi, env.ld), T, E, 1.0 / (T * A * E))
    params = [pol.fc1.weight, pol.fc1.bias, pol.fc2.weight, pol.fc2.bias]
    pol.zero_grad()
    loss = pol.policy_gradient_loss(out, psi)
    assert loss.dim() == 0 and loss.dtype == torch.float32 and loss.requires_grad
    assert float(loss.detach()) == float(want[4].float())
    loss.backward()
    for p, w in zip(params, want):
        assert torch.equal(p.grad, w)
    pol.zero_grad()
    (2 * pol.policy_gradient_loss(out, psi)).backward()
    for p, w in zip(params, want):
        assert torch.equal(p.grad, 2 * w)
    pol.zero_grad()
    pol.policy_gradient_loss(out, psi).backward()
    pol.policy_gradient_loss(out, psi).backward()
    for p, w in zip(params, want):
        assert torch.equal(p.grad, w + w)
    pol.zero_grad()                                  # psi as the [:, :, :E] view of a slab is read in place
    pol.policy_gradient_loss(out, slab(psi, env.ld, float("nan"))[:, :, :E]).backward()
    for p, w in zip(params, want):
        assert torch.equal(p.grad, w)


def test_value_errors():
    env, pol, out, psi = records("coverage", 3, 100, 10)
    with pytest.raises(ValueError, match="shape"):
        pol.policy_gradient_loss(out, psi[:, :, :50])
    with pytest.raises(ValueError, match="shape"):
        pol.policy_gradient_loss(out, psi.double())
    with pytest.raises(ValueError, match="requires grad"):
        pol.policy_gradient_loss(out, psi.clone().requires_grad_())
    env2, pol2, out2, _ = records("coverage", 3, 200, 10)
    with pytest.raises(ValueError, match="not those of this env"):
        pol.policy_gradient_loss(out2, psi)
    with pytest.raises(ValueError, match="record=True"):
        pol.policy_gradient_loss(env.policy_rollout(pol, 10, record=False), psi)
    env4, pol4, out4, psi4 = records("coverage", 4, 100, 10)
    with pytest.raises(ValueError, match="not those of this env"):
        pol.policy_gradient_loss(out4, psi)


class Arena:
    def __init__(self):
        self.bufs = []

    def make(self, shape, dtype, fill=None):
        n = 1
        for d in shape:
            n *= d
        item = torch.empty((), dtype=dtype).element_size()
        raw = torch.full((n * item + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        view = raw[GUARD:GUARD + n * item].view(dtype).view(*shape)
        if fill is not None:
            view.copy_(fill)
        self.bufs.append(raw)
        return view

    def check(self):
        for i, raw in enumerate(self.bufs):
            assert bool((raw[:GUARD] == 0xA5).all()) and bool((raw[-GUARD:] == 0xA5).all()), f"buffer {i} overrun"


@pytest.mark.parametrize("NA", [5, 9])
@pytest.mark.parametrize("A,E", [(1, 1), (3, 37), (16, 1001), (32, 5)])
def test_buffers_stay_in_bounds(A, NA, E):
    from safe_multiagent_rl_b200 import _lib
    lib = _lib.load()
    T, ld = 9, (E + 15) // 16 * 16
    g = torch.Generator(device="cuda").manual_seed(A + E)
    ar = Arena()
    f32 = torch.float32
    obs_ = ar.make((T, 2 * A, ld), f32, torch.rand(T, 2 * A, ld, generator=g, device="cuda") * 5)
    act_ = ar.make((T, A, ld), torch.uint8, torch.randint(0, 256, (T, A, ld), generator=g, device="cuda",
                                                           dtype=torch.uint8))   # bytes >= NA too
    psi = ar.make((T, A, ld), f32, torch.randn(T, A, ld, generator=g, device="cuda"))
    w = [ar.make(s, f32, torch.randn(*s, generator=g, device="cuda")) for s in
         ((A, 2 * A, 16), (A, 16), (A, 16, NA), (A, NA))]
    outs = [ar.make(s, f32) for s in ((A, 2 * A, 16), (A, 16), (A, 16, NA), (A, NA))]
    loss = ar.make((1,), torch.float64)
    scratch = ar.make((lib.smarl_policy_grad_scratch_len(A, NA, T, E),), torch.float64)
    p = _lib.DiscretePolicyParams(A, 16, NA, 0, *[_lib.ptr(x) for x in w], 0, 0, None)
    _lib.check(lib.smarl_policy_grad_discrete(C.byref(p), _lib.ptr(obs_), _lib.ptr(act_), _lib.ptr(psi), T, 0.01,
                                              *[_lib.ptr(o) for o in outs], _lib.ptr(loss), _lib.ptr(scratch), E, ld,
                                              _lib.stream_ptr()))
    torch.cuda.synchronize()
    ar.check()


def test_example_agent_cycle_matches_the_pytorch_loss():
    spec = importlib.util.spec_from_file_location("train_coverage", os.path.join(ROOT, "examples", "train_coverage.py"))
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    argv = ["--fused", "--n_envs", "4096", "--meta_cycles", "1", "--agent_cycles", "1"]
    a = ex.parse_args(argv)
    base = [p.detach().clone() for p in ex.train(a).parameters()]
    new = [p.detach().clone() for p in ex.train(ex.parse_args(argv + ["--fused_grad"])).parameters()]
    for b, n in zip(base, new):                 # Adam's first step moves every weight by about actor_lr
        assert float((b - n).abs().max()) <= 1e-3 * a.actor_lr
