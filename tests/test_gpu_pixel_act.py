"""The pixel agents' small-batch act path (csrc/pixel_act.cu): DrQv2.select_actions / MuLVDrQv2.act_batch against the
CPU oracle's per-observation select_action / act, independence of each action from the batch it is acted on with, the
generator contract, and that acting neither disturbs training nor misses the latest weights.  Handles are prepared at the
shipped batch of 256; N = 100 crosses the 64-row chunk boundary."""
import types

import numpy as np
import pytest
import torch

from oracle import drq_oracle as D
from oracle import mulv_oracle as M


class Box:
    def __init__(self, shape):
        self.shape = shape


def _drq_args(bn, H, update_every=2):
    return types.SimpleNamespace(tau=0.01, update_every=update_every, critic_loss="mse",
                                 stddev_schedule="linear(1.0,0.1,500000)", stddev_clip=0.3, bn_dim=bn, actor_hidden_dim=H,
                                 critic_hidden_dim=H, encoder_lr=1e-4, actor_lr=1e-4, critic_lr=1e-4)


def _mulv_cfg(F, H):
    return dict(aug=True, pre_aug=False, back_q2feat=True, tanh=True, both_q=False, q_activ="relu", q_loss="huber",
                q_up_n=1, l2_norm=0.0, c_targ_tau=0.01, up_every=2, stddev_schedule="linear(1.0,0.1,500000)",
                stddev_clip=0.3, feat_dim=F, hid_dim=H, lr=1e-4, vae_w=0.5, mse_w=1.0, c_noise=0.1)


# (agent, C, A): DrQ-v2 at bn 50 / H 1024, muLV-Rep at feat 100 / H 1024 (the shipped widths)
AGENTS = [("drq", 9, 4), ("drq", 3, 6), ("mulv", 9, 4)]
B = 256
STEP = 250000  # past muLV-Rep's exploration phase


def _make(kind, C, A, precision, seed=0, B=B):
    """(agent, oracle, batched act, single act of the agent, single act of the oracle)."""
    from rlrep_b200.pixel import DrQv2, MuLVDrQv2
    if kind == "drq":
        init = D.init_state(C, A, 50, 1024, seed=seed)
        oracle = D.OracleDrQv2(A, init)
        agent = DrQv2(Box((C, 84, 84)), Box((A,)), _drq_args(50, 1024), precision=precision)
        batched = lambda obs, step, det: agent.select_actions(obs, step, det)
        single = lambda obs, step, det: agent.select_action(obs, step, det)
        ref = lambda obs, step, det: oracle.select_action(obs, step, det)
    else:
        init = M.init_state(C, A, 100, 1024, seed=seed)
        oracle = M.OracleMuLVDrQ(A, init)
        agent = MuLVDrQv2((C, 84, 84), (A,), _mulv_cfg(100, 1024), precision=precision)
        batched = lambda obs, step, det: agent.act_batch(obs, step, det)
        single = lambda obs, step, det: agent.act(obs, step, det)
        ref = lambda obs, step, det: oracle.act(obs, step, det)
    agent.load_state_dict(init)
    agent.prepare(B)
    return agent, oracle, batched, single, ref


def _frames(n, C, seed=3):
    return D.synthetic_pixel_batch(n, C, 84, 1, seed=seed).img


@pytest.mark.gpu
@pytest.mark.parametrize("kind,C,A", AGENTS)
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_act_batch_matches_oracle(kind, C, A, precision):
    agent, _, batched, _, ref = _make(kind, C, A, precision)
    obs = _frames(100, C)
    worst = 0.0
    for n in (1, 3, 64, 100):
        for det in (True, False):
            torch.manual_seed(5)
            got = batched(obs[:n], STEP, det)
            torch.manual_seed(5)
            want = np.stack([ref(obs[i], STEP, det) for i in range(n)])
            assert got.shape == want.shape == (n, A)
            worst = max(worst, float(np.abs(got - want).max()))
            assert np.allclose(got, want, atol=2e-5), (n, det, np.abs(got - want).max())
    print(f"{kind} C={C} A={A} {precision}: worst |action - oracle| {worst:.2e}")
    agent.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,C,A", AGENTS)
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_action_does_not_depend_on_the_batch(kind, C, A, precision):
    agent, _, batched, single, _ = _make(kind, C, A, precision)
    obs = _frames(100, C, seed=7)
    for det in (True, False):
        torch.manual_seed(9)
        singles = [torch.from_numpy(np.asarray(single(obs[i], STEP, det))) for i in range(100)]
        for n in (1, 7, 64, 100):
            torch.manual_seed(9)
            got = torch.from_numpy(batched(obs[:n], STEP, det))
            for i in range(n):
                assert torch.equal(got[i], singles[i]), (det, n, i, got[i], singles[i])
    agent.close()


def test_act_noise_consumes_the_generator_like_sequential_acts():
    """CPU only: the host draws of a batched act equal those of N sequential oracle acts, in order and in generator
    state; in muLV-Rep's exploration phase the uniform draws are the oracle's actions bit for bit."""
    from rlrep_b200.pixel import _act_noise
    C, A, n = 3, 6, 5
    obs = _frames(n, C)
    od = D.OracleDrQv2(A, D.init_state(C, A, 16, 32, seed=0))
    om = M.OracleMuLVDrQ(A, M.init_state(C, A, 16, 32, seed=0))
    torch.manual_seed(3)
    for i in range(n):
        od.select_action(obs[i], 1000)
    want = torch.get_rng_state()
    torch.manual_seed(3)
    eps, uni = _act_noise(n, A, sample=True)
    assert uni is None and eps.shape == (n, A) and torch.equal(torch.get_rng_state(), want)
    want = torch.manual_seed(3).get_state()
    assert _act_noise(n, A, sample=False) == (None, None)  # deterministic: no draws at all
    assert torch.equal(torch.get_rng_state(), want)
    for step, explore in ((100, True), (250000, False)):
        torch.manual_seed(4)
        acts = np.stack([om.act(obs[i], step, False) for i in range(n)])
        want = torch.get_rng_state()
        torch.manual_seed(4)
        eps, uni = _act_noise(n, A, sample=True, explore=explore)
        assert torch.equal(torch.get_rng_state(), want), step
        if explore:
            assert np.array_equal(uni, acts)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["drq", "mulv"])
def test_acting_between_updates_does_not_change_training(kind):
    """update, act on 64 frames, update == update, update.  Between the two, one more update runs on the batch the first
    one left in the device buffers (`*_update_resident`), so an act that wrote any update buffer (frames, latents,
    activations) would change what it computes."""
    import ctypes as C
    from rlrep_b200.pixel import DrQv2, MuLVDrQv2
    Cc, A, Bu = 9, 4, 64
    obs = _frames(64, Cc, seed=11)

    def run(act_between):
        if kind == "drq":
            init = D.init_state(Cc, A, 50, 256, seed=0)
            agent = DrQv2(Box((Cc, 84, 84)), Box((A,)), _drq_args(50, 256, update_every=1), precision="tf32")
            batches = [D.synthetic_pixel_batch(Bu, Cc, 84, A, seed=20 + i) for i in range(2)]
            update = lambda b, step: agent.train_step(iter([tuple(b)]), step)
            act = lambda: agent.select_actions(obs, STEP)
            resident = lambda: agent.lib.rlrep_drq_update_resident
        else:
            init = M.init_state(Cc, A, 100, 256, seed=0)
            agent = MuLVDrQv2((Cc, 84, 84), (A,), _mulv_cfg(100, 256), precision="tf32")
            batches = [M.synthetic_pixel_batch(Bu, Cc, 84, A, seed=20 + i) for i in range(2)]
            update = lambda b, step: agent.update(iter([tuple(b)]), step)
            act = lambda: agent.act_batch(obs, STEP, False)
            resident = lambda: agent.lib.rlrep_mulv_update_resident
        agent.load_state_dict(init)
        torch.manual_seed(1)
        m = [update(batches[0], 2)]
        if act_between:
            act()
        ms = C.c_float()
        assert resident()(agent._h, 1, 0.5, C.byref(ms)) == 0
        after_resident = agent.state_dict()
        torch.manual_seed(2)
        m.append(update(batches[1], 4))
        sd = agent.state_dict()
        agent.close()
        return m, after_resident, sd

    m0, r0, sd0 = run(False)
    m1, r1, sd1 = run(True)
    assert all(m0) and m0 == m1, (m0, m1)
    for a, b in ((r0, r1), (sd0, sd1)):
        assert set(a) == set(b)
        for k in a:
            assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["drq", "mulv"])
def test_wide_trunk_handle_updates_and_acts(kind):
    """A trunk wider than 128 (bn_dim / feat_dim 256): the handle is created and updated as before, and acting on it
    matches the oracle on the weights the update left."""
    from rlrep_b200.pixel import DrQv2, MuLVDrQv2
    Cc, A, W, H, Bu = 3, 4, 256, 64, 8
    obs = _frames(3, Cc, seed=13)
    if kind == "drq":
        agent = DrQv2(Box((Cc, 84, 84)), Box((A,)), _drq_args(W, H, update_every=1), precision="fp32")
        agent.load_state_dict(D.init_state(Cc, A, W, H, seed=0))
        torch.manual_seed(1)
        m = agent.train_step(iter([tuple(D.synthetic_pixel_batch(Bu, Cc, 84, A, seed=5))]), 2)
        oracle = D.OracleDrQv2(A, agent.state_dict())
        got, want = agent.select_actions(obs, STEP, True), [oracle.select_action(o, STEP, True) for o in obs]
    else:
        agent = MuLVDrQv2((Cc, 84, 84), (A,), _mulv_cfg(W, H), precision="fp32")
        agent.load_state_dict(M.init_state(Cc, A, W, H, seed=0))
        torch.manual_seed(1)
        m = agent.update(iter([tuple(M.synthetic_pixel_batch(Bu, Cc, 84, A, seed=5))]), 2)
        oracle = M.OracleMuLVDrQ(A, agent.state_dict())
        got, want = agent.act_batch(obs, STEP, True), [oracle.act(o, STEP, True) for o in obs]
    assert m and all(np.isfinite(v) for v in m.values()), m
    assert np.allclose(got, np.stack(want), atol=2e-5), np.abs(got - np.stack(want)).max()
    agent.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["drq", "mulv"])
def test_act_sees_loaded_weights(kind):
    C, A = 9, 4
    agent, _, batched, _, _ = _make(kind, C, A, "fp32")
    obs = _frames(5, C)
    before = batched(obs, STEP, True)
    if kind == "drq":
        init = D.init_state(C, A, 50, 1024, seed=1)
        oracle = D.OracleDrQv2(A, init)
        ref = lambda o: oracle.select_action(o, STEP, True)
    else:
        init = M.init_state(C, A, 100, 1024, seed=1)
        oracle = M.OracleMuLVDrQ(A, init)
        ref = lambda o: oracle.act(o, STEP, True)
    agent.load_state_dict(init)
    got = batched(obs, STEP, True)
    want = np.stack([ref(o) for o in obs])
    assert not np.allclose(before, want, atol=1e-3)
    assert np.allclose(got, want, atol=2e-5), np.abs(got - want).max()
    agent.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["drq", "mulv"])
def test_act_input_checks_and_cuda_frames(kind):
    C, A = 9, 4
    agent, _, batched, _, _ = _make(kind, C, A, "fp32", B=8)
    obs = _frames(6, C)
    for bad in (obs.astype(np.float32), obs[:, :3], obs[0], obs[:0], obs.astype(np.int64)):
        with pytest.raises(ValueError):
            batched(bad, STEP, True)
    with pytest.raises(ValueError):
        batched(torch.from_numpy(obs).cuda().float(), STEP, True)
    host = batched(obs, STEP, True)
    assert np.array_equal(batched(torch.from_numpy(obs), STEP, True), host)
    assert np.array_equal(batched(torch.from_numpy(obs).cuda(), STEP, True), host)
    agent.close()
