"""GPU: checkpoints of the three pixel agents (DrQ-v2, μLV-Rep, latent Diff-SR).  `save` / `load` carry the parameters,
the Polyak targets, the Adam moments and the step counters, so a resumed run continues bit-identically; the exported
moments are torch.optim's exp_avg / exp_avg_sq of the same parameter (checked against the CPU oracles' optimisers); the
weights-only load, the refusals, and `state_dict()` keeping its old contents.  Small shapes of the agents' own GPU tests
(tests/test_gpu_drq.py, test_gpu_mulv.py, test_gpu_ldiffsr.py), weights and batches from oracle/*_oracle.py."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

AGENTS = ("drqv2", "mulvdrq", "ldiffsr")
LDIFF_DIMS = (4, 64, 32, 32, 32, 2, 32, 4, 64)  # Dims(A, L, feat, bn, psi_h, psi_d, zeta_h, zeta_d, H)


class Box:
    def __init__(self, shape):
        self.shape = shape


def _make(alg, precision, seed=0, update_every=2, action_dim=4):
    """(agent, initial weights from the oracle's init_state(seed), batch(seed) -> a synthetic replay batch, batch size)."""
    if alg == "drqv2":
        from oracle import drq_oracle as O
        from rlrep_b200.pixel import DrQv2
        C_, bn, H, B = 9, 50, 256, 8
        args = types.SimpleNamespace(tau=0.01, update_every=update_every, critic_loss="mse",
                                     stddev_schedule="linear(1.0,0.1,500000)", stddev_clip=0.3, bn_dim=bn,
                                     actor_hidden_dim=H, critic_hidden_dim=H, encoder_lr=1e-4, actor_lr=1e-4,
                                     critic_lr=1e-4)
        agent = DrQv2(Box((C_, 84, 84)), Box((action_dim,)), args, precision=precision)
        init = O.init_state(C_, action_dim, bn, H, seed=seed)
        return agent, init, lambda s: O.synthetic_pixel_batch(B, C_, 84, action_dim, seed=s), B
    if alg == "mulvdrq":
        from oracle import mulv_oracle as O
        from rlrep_b200.pixel import MuLVDrQv2
        C_, F, H, B = 9, 100, 64, 4
        cfg = dict(aug=True, pre_aug=False, back_q2feat=True, tanh=True, both_q=False, q_activ="relu", q_loss="huber",
                   q_up_n=1, l2_norm=0.0, c_targ_tau=0.01, up_every=update_every,
                   stddev_schedule="linear(1.0,0.1,500000)", stddev_clip=0.3, feat_dim=F, hid_dim=H, lr=1e-4, vae_w=0.5,
                   mse_w=1.0, c_noise=0.1)
        agent = MuLVDrQv2((C_, 84, 84), (action_dim,), cfg, precision=precision)
        init = O.init_state(C_, action_dim, F, H, seed=seed)
        return agent, init, lambda s: O.synthetic_pixel_batch(B, C_, 84, action_dim, seed=s), B
    from oracle import ldiffsr_oracle as O
    from rlrep_b200.pixel import LatentDiffSRDrQv2
    d = O.Dims(action_dim, *LDIFF_DIMS[1:])
    B = 4
    args = types.SimpleNamespace(use_repr_target=True, back_critic_grad=True, critic_loss="mse", reg_coef=0.0,
                                 grad_norm=None, extra_repr_step=1, do_scale=False, repr_coef=1.0, ae_num_layers=4,
                                 ae_num_filters=32, noise_schedule="linear", ae_lr=3e-4, score_lr=3e-4, actor_lr=1e-4,
                                 critic_lr=1e-4, bn_dim=d.bn, update_every=update_every,
                                 stddev_schedule="linear(1.0,0.1,500000)", stddev_clip=0.3, latent_dim=d.L,
                                 feature_dim=d.feat, psi_hidden_dim=d.psi_h, psi_hidden_depth=d.psi_d,
                                 zeta_hidden_dim=d.zeta_h, zeta_hidden_depth=d.zeta_d, actor_hidden_dim=d.H,
                                 critic_hidden_dim=d.H, noise_param1=1e-4, noise_param2=0.02, num_noises=1000, tau=0.01,
                                 kl_coef=1.0, ae_coef=1.0)
    agent = LatentDiffSRDrQv2(Box((9, 84, 84)), Box((action_dim,)), args, precision=precision)
    return agent, O.init_state(d, seed=seed), lambda s: O.synthetic_pixel_batch(B, 9, 84, action_dim, seed=s), B


def _oracle(alg, init):
    """The CPU oracle of `alg` on `init`, updating on every call."""
    if alg == "drqv2":
        from oracle import drq_oracle as O
        return O.OracleDrQv2(4, init, update_every=1)
    if alg == "mulvdrq":
        from oracle import mulv_oracle as O
        return O.OracleMuLVDrQ(4, init, up_every=1)
    from oracle import ldiffsr_oracle as O
    return O.OracleLatentDiffSR(O.Dims(*LDIFF_DIMS), init, update_every=1)


def _call(alg, agent, batch, step):
    """One call of the reference's training entry point (it updates or not, as update_every / up_every says)."""
    if alg == "mulvdrq":
        return agent.update(iter([tuple(batch)]), step)
    return agent.train_step(iter([tuple(batch)]), step)


def _oracle_call(alg, oracle, batch, step):
    return oracle.update(batch, step) if alg == "mulvdrq" else oracle.train_step(batch, step)


def _act(alg, agent, obs):
    if alg == "drqv2":
        return agent.select_actions(obs, 250000, deterministic=False)
    return agent.act_batch(obs, 250000, eval_mode=False)


def _assert_same_tensors(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert torch.equal(a[k], b[k]), k


def _rel(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()


@pytest.mark.parametrize("precision", ["tf32", "fp32"])
@pytest.mark.parametrize("alg", AGENTS)
def test_resume_is_bit_identical(alg, precision, tmp_path):
    """Three calls (update_every = 2: the period is half way through), save, four more calls; a second agent built from
    other initial weights loads the file and makes the same four calls from the same generator state.  Every metric, every
    parameter, target and moment, the counters and the actions then agree bit for bit."""
    a1, init, batch, _ = _make(alg, precision, seed=0)
    a1.load_state_dict(init)
    n, k = 3, 4
    batches = [batch(100 + i) for i in range(n + k)]
    torch.manual_seed(1)
    np.random.seed(1)
    for i in range(n):
        _call(alg, a1, batches[i], i)
    path = tmp_path / f"{alg}.pt"
    a1.save(path, step=n)
    rng, np_rng = torch.get_rng_state(), np.random.get_state()
    m1 = [_call(alg, a1, batches[i], i) for i in range(n, n + k)]
    assert [bool(m) for m in m1] == [False, True, False, True]

    a2, init2, _, _ = _make(alg, precision, seed=5)
    a2.load_state_dict(init2)
    a2.load(path)
    torch.set_rng_state(rng)
    np.random.set_state(np_rng)
    m2 = [_call(alg, a2, batches[i], i) for i in range(n, n + k)]
    assert m1 == m2
    _assert_same_tensors(a1.state_dict(), a2.state_dict())
    o1, o2 = a1.optimizer_state_dict(step=n + k), a2.optimizer_state_dict(step=n + k)
    assert o1.pop("control") == o2.pop("control")
    _assert_same_tensors(o1, o2)
    if alg != "ldiffsr":  # latent Diff-SR has no act path
        obs = torch.from_numpy(batch(7).img)
        acts = []
        for a in (a1, a2):
            torch.manual_seed(9)
            acts.append(_act(alg, a, obs))
        assert np.array_equal(acts[0], acts[1])
    a1.close()
    a2.close()


# Bars on the moments after one update from identical weights: exp_avg = 0.1 g, so its error is the gradient's, and the
# gradient bars are those of the agents' own fp32 gradient tests (tests/test_gpu_drq.py per group: critic 2e-5, actor
# 2e-3 after the critic's Adam step, encoder 5e-3 behind four ReLU conv layers whose masks flip at rounding distance from
# zero; tests/test_gpu_mulv.py 5e-3 for every group; the conv / deconv realistic-regime gradient bar 5e-3 for latent
# Diff-SR, whose own test compares parameters only).  exp_avg_sq = 0.001 g^2 doubles a relative error: twice the bar.
MOMENT_BARS = {"drqv2": {"critic": 2e-5, "actor": 2e-3, "encoder": 5e-3}, "mulvdrq": {}, "ldiffsr": {}}


@pytest.mark.parametrize("alg", AGENTS)
def test_moments_are_the_reference_optimisers_state(alg):
    """Every exported `optim.m/<name>` / `optim.v/<name>` is the oracle optimiser's exp_avg / exp_avg_sq of parameter
    <name> -- same names, same shapes (a moment in the internal conv layout or transposed fails here), norm-wise close --
    and the three step counters are the optimisers' `step`."""
    agent, init, batch, _ = _make(alg, "fp32", seed=0, update_every=1)
    agent.load_state_dict(init)
    oracle = _oracle(alg, init)
    b = batch(30)
    torch.manual_seed(1)
    _oracle_call(alg, oracle, b, 0)
    torch.manual_seed(1)
    _call(alg, agent, b, 0)
    got = agent.optimizer_state_dict(step=0)
    ctl = got.pop("control")
    name = {id(v): k for k, v in oracle.p.items()}
    ref, steps = {}, set()
    for opt in oracle.opt.values():
        for p, st in opt.state.items():
            ref["optim.m/" + name[id(p)]], ref["optim.v/" + name[id(p)]] = st["exp_avg"], st["exp_avg_sq"]
            steps.add(int(st["step"]))
    assert set(got) == set(ref), (sorted(set(got) - set(ref))[:8], sorted(set(ref) - set(got))[:8])
    worst = {}
    for k, r in ref.items():
        assert tuple(got[k].shape) == tuple(r.shape), (k, tuple(got[k].shape), tuple(r.shape))
        group = k.split("/", 1)[1].split(".")[0]
        bar = MOMENT_BARS[alg].get(group, 5e-3) * (2 if k.startswith("optim.v/") else 1)
        worst[k] = (_rel(got[k], r), bar)
    bad = {k: e for k, e in worst.items() if e[0] >= e[1]}
    print(f"\n{alg}: worst moment errors " + ", ".join(
        f"{k} {e:.1e}" for k, (e, _) in sorted(worst.items(), key=lambda kv: -kv[1][0] / kv[1][1])[:6]))
    assert not bad, bad
    assert steps == {1}
    assert (ctl["t_feature"], ctl["t_critic"], ctl["t_actor"]) == (1, 1, 1)
    agent.close()


@pytest.mark.parametrize("alg", AGENTS)
def test_moments_accumulate_like_torch_adam(alg):
    """Across updates the exported moments mix as torch.optim's do: torch.optim.Adam, given the moments and step count
    after update 2 and the gradients update 3 stepped with (read back as "grad/<name>"), lands on the moments the agent
    exports after update 3.  This pins the beta mixing and the counters independently of how closely the gradients
    themselves follow the oracle (the test above holds those to the gradient bars)."""
    agent, init, batch, _ = _make(alg, "fp32", seed=0, update_every=1)
    agent.load_state_dict(init)
    torch.manual_seed(1)
    for i in range(2):
        _call(alg, agent, batch(60 + i), i)
    before = agent.optimizer_state_dict(step=2)
    assert (before["control"]["t_feature"], before["control"]["t_critic"], before["control"]["t_actor"]) == (2, 2, 2)
    _call(alg, agent, batch(62), 2)
    after, g = agent.optimizer_state_dict(step=3), agent.grads()
    assert (after["control"]["t_feature"], after["control"]["t_critic"], after["control"]["t_actor"]) == (3, 3, 3)
    worst = (0.0, "")
    for k in (k for k in after if k.startswith("optim.m/")):
        name = k[len("optim.m/"):]
        p = torch.zeros_like(g[name], requires_grad=True)
        opt = torch.optim.Adam([p], lr=1e-4, foreach=False)
        opt.state[p] = {"step": torch.tensor(2.0), "exp_avg": before[k].clone(),
                        "exp_avg_sq": before["optim.v/" + name].clone()}
        p.grad = g[name].clone()
        opt.step()
        for got, want in ((after[k], opt.state[p]["exp_avg"]), (after["optim.v/" + name], opt.state[p]["exp_avg_sq"])):
            assert got.shape == want.shape
            e = _rel(got, want)
            worst = max(worst, (e, name))
            assert e < 1e-6, (name, e)
    print(f"\n{alg}: worst relative difference to torch.optim.Adam's accumulated moments {worst[0]:.1e} ({worst[1]})")
    agent.close()


@pytest.mark.parametrize("alg", AGENTS)
def test_counters_round_trip(alg):
    """Each step counter goes to its own slot of the control block and comes back from it, and the next update advances
    each by one."""
    agent, init, batch, B = _make(alg, "tf32", seed=0, update_every=1)
    agent.load_state_dict(init)
    agent.prepare(B)
    sd = agent.optimizer_state_dict(step=0)
    sd["control"].update(t_feature=3, t_critic=5, t_actor=7)
    agent.load_optimizer_state_dict(sd)
    ctl = agent.optimizer_state_dict()["control"]
    assert (ctl["t_feature"], ctl["t_critic"], ctl["t_actor"]) == (3, 5, 7)
    torch.manual_seed(1)
    _call(alg, agent, batch(70), 0)
    ctl = agent.optimizer_state_dict()["control"]
    assert (ctl["t_feature"], ctl["t_critic"], ctl["t_actor"]) == (4, 6, 8)
    agent.close()


@pytest.mark.parametrize("alg", AGENTS)
def test_weights_only_load(alg, tmp_path):
    """load(path, load_optimizer=False) restores the saved parameters with their saved (not re-synchronised) targets and
    leaves the moments and counters as a fresh handle has them."""
    a1, init, batch, B = _make(alg, "tf32", seed=0, update_every=1)
    a1.load_state_dict(init)
    torch.manual_seed(1)
    _call(alg, a1, batch(40), 0)
    path = tmp_path / f"{alg}.pt"
    a1.save(path)
    a2, init2, _, _ = _make(alg, "tf32", seed=5, update_every=1)
    a2.load_state_dict(init2)
    a2.load(path, load_optimizer=False)
    _assert_same_tensors(a2.state_dict(), a1.state_dict())
    fresh, _, _, _ = _make(alg, "tf32", seed=5, update_every=1)
    fresh.prepare(B)
    o2, of = a2.optimizer_state_dict(), fresh.optimizer_state_dict()
    assert o2.pop("control") == of.pop("control")
    _assert_same_tensors(o2, of)
    for a in (a1, a2, fresh):
        a.close()


@pytest.mark.parametrize("alg", AGENTS)
def test_refusals(alg, tmp_path):
    from rlrep_b200 import _lib
    from rlrep_b200._lib import RlrepError
    agent, init, batch, B = _make(alg, "tf32", seed=0)
    path = tmp_path / f"{alg}.pt"
    with pytest.raises(RlrepError):  # no handle yet, so no moments to save
        agent.save(path)
    agent.load_state_dict(init)
    agent.prepare(B)
    agent.save(path)

    other = _make(AGENTS[(AGENTS.index(alg) + 1) % 3], "tf32")[0]
    with pytest.raises(RlrepError):  # a checkpoint of another agent
        other.load(path)
    wrong_a = _make(alg, "tf32", action_dim=6)[0]
    with pytest.raises(RlrepError):
        wrong_a.load(path)
    wrong_b = _make(alg, "tf32")[0]
    wrong_b.prepare(2 * B)
    with pytest.raises(RlrepError):  # the batch size is fixed per handle
        wrong_b.load(path)

    for field in ("steps", "t_alpha", "log_alpha"):  # the pixel agents have no steps gate and no temperature
        st = _lib.OptimState(**{field: 1})
        assert agent._fn("set_optim_state")(agent._h, C.byref(st)) != 0
        assert b"must be 0" in agent.lib.rlrep_last_error()
    assert agent.optimizer_state_dict()["control"]["t_critic"] == 0
    for a in (agent, wrong_b):
        a.close()


@pytest.mark.parametrize("alg", AGENTS)
def test_state_dict_keeps_its_contents(alg):
    """The moments are reached through optimizer_state_dict only: state_dict() still holds parameters and targets."""
    agent, init, _, B = _make(alg, "tf32", seed=0)
    agent.load_state_dict(init)
    agent.prepare(B)
    sd = agent.state_dict()
    assert not [k for k in sd if k.startswith(("optim.", "grad/"))]
    assert set(init) <= set(sd)
    assert set(k for k in agent._index if k.startswith("optim.")) == set(agent.optimizer_state_dict()) - {"control"}
    agent.close()
