"""GPU: SAC seed populations (rlrep_b200.SACPopulation) -- member m of a population computes bit for bit what a lone
SACAgent seeded with seeds[m] computes, through the eager call, the graph capture and replays."""
import numpy as np
import pytest
import torch

from parity_util import Space, worst_info_error, worst_param_error

from oracle import rl_oracle as O

pytestmark = pytest.mark.gpu

S, A, H, B = 17, 6, 96, 128


def _buffers(n, rows=3000):
    from rlrep_b200 import ReplayBuffer
    out = []
    for m in range(n):
        ring = O.synthetic_ring(S, A, rows, seed=100 + m)
        b = ReplayBuffer(S, A, max_size=rows)
        b.load(ring.state, ring.action, ring.next_state, ring.reward, ring.done)
        out.append(b)
    return out


def _lone_run(seed, buf, steps, kw, after=None):
    """What a lone process seeded with `seed` does: build a SACAgent, train it `steps` times."""
    from rlrep_b200 import SACAgent
    np.random.seed(seed)
    torch.manual_seed(seed)
    agent = SACAgent(S, A, Space(A), hidden_dim=H, **kw)
    init = agent.state_dict()
    infos = [agent.train(buf, B) for _ in range(steps)]
    return agent, init, infos


def _full_state(sd, opt):
    out = {k: v for k, v in sd.items()}
    out.update({k: v for k, v in opt.items() if k != "control"})
    return out, opt["control"]


def _assert_member_equals(pop, m, agent):
    ps, pc = _full_state(pop.state_dict(m), pop.optimizer_state_dict(m))
    ls, lc = _full_state(agent.state_dict(), agent.optimizer_state_dict())
    assert set(ps) == set(ls)
    for k in ls:
        assert torch.equal(ps[k], ls[k]), (m, k)
    assert pc == lc, (m, pc, lc)


@pytest.mark.parametrize("members", [3, 8])
@pytest.mark.parametrize("precision", ["tf32", "fp32"])
def test_members_are_bit_identical_to_lone_agents(members, precision):
    from rlrep_b200 import SACPopulation
    seeds = [7 + 11 * m for m in range(members)]
    bufs = _buffers(members)
    kw = dict(precision=precision)
    pop = SACPopulation(seeds, S, A, Space(A), hidden_dim=H, **kw)
    pop_infos = [pop.train(bufs, B) for _ in range(4)]  # eager, capture, two replays
    for m, s in enumerate(seeds):
        agent, init, infos = _lone_run(s, bufs[m], 4, kw)
        assert [pi[m] for pi in pop_infos] == infos, m
        assert all(type(v) is type(infos[0][k]) for k, v in pop_infos[0][m].items())
        _assert_member_equals(pop, m, agent)
        agent._h.close()
    if members == 8:
        from rlrep_b200 import SACAgent
        lone = SACAgent(S, A, Space(A), hidden_dim=H, **kw)
        for _ in range(3):
            lone.train(bufs[0], B)
        assert pop.gpu_launches_last_train == lone.gpu_launches_last_train > 0


def test_seeded_population_equals_seeded_lone_runs():
    """Initial weights, the info dicts of four calls and the final state of SACPopulation(seeds=[s0, s1, s2])."""
    from rlrep_b200 import SACPopulation
    seeds = [3, 1000, 99]
    bufs = _buffers(3)
    pop = SACPopulation(seeds, S, A, Space(A), hidden_dim=H)
    init = [pop.state_dict(m) for m in range(3)]
    infos = [pop.train(bufs, B) for _ in range(4)]
    for m, s in enumerate(seeds):
        agent, linit, linfos = _lone_run(s, bufs[m], 4, {})
        for k in linit:
            assert torch.equal(init[m][k], linit[k]), (m, k)
        assert [i[m] for i in infos] == linfos
        _assert_member_equals(pop, m, agent)


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_member_meets_the_oracle_bar(precision):
    from rlrep_b200 import ReplayBuffer, SACPopulation
    bar = {"fp32": 1e-5, "tf32": 1e-3}[precision]
    kw = dict(hidden_dim=256)
    seeds = [5, 6, 7]
    init = O.init_state("sac", S, A, kw, seed=0)
    oracle = O.ORACLES["sac"](S, A, init, discount=0.99, tau=0.005, **kw)
    oring = O.synthetic_ring(S, A, 5000, seed=0)
    pop = SACPopulation(seeds, S, A, Space(A), discount=0.99, tau=0.005, precision=precision, **kw)
    bufs = _buffers(3, rows=5000)
    bufs[2] = ReplayBuffer(S, A, max_size=5000)
    bufs[2].load(oring.state, oring.action, oring.next_state, oring.reward, oring.done)
    pop.train(bufs, 256)  # builds the handle; member 2 is then reset to the oracle's weights and generators
    pop.load_state_dict(2, init)
    pop.load_optimizer_state_dict(2, {k: torch.zeros_like(v) for k, v in pop.optimizer_state_dict(2).items()
                                      if k != "control"} | {"control": dict(
        steps=0, t_feature=0, t_critic=0, t_actor=0, t_alpha=0, log_alpha=float(np.log(0.1)), log_alpha_m=0.0,
        log_alpha_v=0.0, agent_steps=0)})
    pop._rs[2].seed(seeds[2])
    pop._cpu_gen[2].manual_seed(seeds[2])
    ci = [pop.train(bufs, 256)[2] for _ in range(4)]
    np.random.seed(seeds[2])
    torch.manual_seed(seeds[2])
    oi = [oracle.train(oring, 256) for _ in range(4)]

    class Member:
        def state_dict(self):
            return pop.state_dict(2)

    wi, where_i = worst_info_error(ci, oi, atol=1e-5)
    wp, where_p, _ = worst_param_error(Member(), oracle)
    assert wi < bar, where_i
    assert wp < bar, where_p


def test_select_actions_equal_lone_select_action():
    from rlrep_b200 import SACAgent, SACPopulation
    seeds = [21, 22, 23, 24]
    pop = SACPopulation(seeds, S, A, Space(A), hidden_dim=H)
    states = np.random.RandomState(0).randn(4, S).astype(np.float32)
    got = [pop.select_actions(states, explore=e) for e in (False, True, True)]
    for m, s in enumerate(seeds):
        torch.manual_seed(s)
        agent = SACAgent(S, A, Space(A), hidden_dim=H)
        want = [agent.select_action(states[m], explore=e) for e in (False, True, True)]
        for g, w in zip(got, want):
            assert np.array_equal(g[m], w), m


def test_checkpoint_of_a_member_resumes_in_a_lone_agent(tmp_path):
    from rlrep_b200 import SACAgent, SACPopulation
    seeds = [1, 2, 3]
    bufs = _buffers(3)
    pop = SACPopulation(seeds, S, A, Space(A), hidden_dim=H)
    for _ in range(3):
        pop.train(bufs, B)
    m = 1
    pop.save_member(m, tmp_path / "m1.pt")
    agent = SACAgent(S, A, Space(A), hidden_dim=H)
    agent.load(tmp_path / "m1.pt")
    # the lone agent continues on member 1's generators from here
    np.random.set_state(pop._rs[m].get_state())
    torch.set_rng_state(pop._cpu_gen[m].get_state())
    li = [agent.train(bufs[m], B) for _ in range(3)]
    pi = [pop.train(bufs, B)[m] for _ in range(3)]
    assert li == pi
    _assert_member_equals(pop, m, agent)
    # and a member loads a lone checkpoint back
    agent.save(tmp_path / "lone.pt")
    pop.load_member(0, tmp_path / "lone.pt")
    _assert_member_equals(pop, 0, agent)


def test_cuda_noise_equals_cpu_noise_fed_the_same_tensors(monkeypatch):
    from rlrep_b200 import SACPopulation
    seeds = [4, 5, 6]
    bufs = _buffers(3)
    cpu = SACPopulation(seeds, S, A, Space(A), hidden_dim=H, noise_device="cpu")
    dev = SACPopulation(seeds, S, A, Space(A), hidden_dim=H, noise_device="cuda")
    drawn = []
    real = cpu._randn

    def record(m, rows, cols):
        t = real(m, rows, cols)
        drawn.append(t)
        return t
    monkeypatch.setattr(cpu, "_randn", record)
    replay = iter(drawn)
    monkeypatch.setattr(dev, "_randn", lambda m, rows, cols: next(replay).cuda())
    for _ in range(4):
        a = cpu.train(bufs, B)
        b = dev.train(bufs, B)
        assert a == b
    for m in range(3):
        for k, v in cpu.state_dict(m).items():
            assert torch.equal(v, dev.state_dict(m)[k]), (m, k)


def test_refusals():
    from rlrep_b200 import ReplayBuffer, RlrepError, SACPopulation
    from rlrep_b200 import _lib
    import ctypes as C
    bufs = _buffers(3)
    pop = SACPopulation([1, 2, 3], S, A, Space(A), hidden_dim=H)
    pop.train(bufs, B)
    with pytest.raises(ValueError):
        pop.train(bufs[:2], B)
    other = ReplayBuffer(S + 1, A, max_size=100)
    other.load(*(lambda r: (r.state, r.action, r.next_state, r.reward, r.done))(O.synthetic_ring(S + 1, A, 100, seed=1)))
    with pytest.raises(RlrepError, match="ring shape"):
        pop.train([bufs[0], other, bufs[2]], B)
    h = pop._h
    idx = np.zeros(3 * B, dtype=np.int64)
    idx[2 * B + 5] = 10 ** 6
    eps = np.zeros(3 * 2 * B * A, dtype=np.float32)
    with pytest.raises(RlrepError, match=r"out of range \(member 2\)"):
        h.train(bufs, idx, eps)
    with pytest.raises(RlrepError, match="wrong number"):
        h.train(bufs, idx[:-1], eps)
    lib = _lib.load()
    cfg = pop._shells[0]._config(B)
    out = C.c_void_p()
    assert lib.rlrep_sacpop_create(C.byref(cfg), 0, None, C.byref(out)) != 0
    assert b"at least one member" in lib.rlrep_last_error()
    cfg.alg = _lib.ALG["ctrlsac"]
    assert lib.rlrep_sacpop_create(C.byref(cfg), 2, None, C.byref(out)) != 0
    assert b"implemented for sac" in lib.rlrep_last_error()
