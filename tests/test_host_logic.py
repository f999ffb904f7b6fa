"""CPU: host-side logic of the agent shims that does not need a device -- RNG consumption order, config mapping,
initial-weight tables, info-dict keys."""
import numpy as np
import pytest
import torch

from oracle import rl_oracle as O
from rlrep_b200 import _lib
from rlrep_b200.agents import AGENTS, CTRLSACAgent, SACAgent


class Space:
    def __init__(self, A):
        self.low, self.high = -np.ones(A, np.float32), np.ones(A, np.float32)


class FakeBuffer:
    size = 5000


CASES = {
    "sac": (dict(hidden_dim=32), 64),
    "ctrlsac": (dict(hidden_dim=32, feature_dim=64, extra_feature_steps=3), 32),
    "vlsac": (dict(hidden_dim=32, feature_dim=64, extra_feature_steps=3), 32),
    "spedersac": (dict(feature_dim=64, extra_feature_steps=2, phi_and_mu_lr=1e-5, phi_hidden_dim=64, phi_hidden_depth=1,
                       mu_hidden_dim=64, mu_hidden_depth=0, critic_and_actor_lr=3e-4, critic_and_actor_hidden_dim=32), 32),
    "diffsrsac": (dict(hidden_dim=32, feature_dim=32, phi_hidden_dim=32, nabla_mu_hidden_dim=64, extra_feature_steps=2), 32),
}


@pytest.mark.parametrize("alg", list(CASES))
def test_draw_consumes_the_global_rngs_exactly_like_the_reference(alg):
    """After one train(), numpy's legacy RNG and torch's CPU generator must be in the same state on both sides,
    and the drawn indices / noise must be the ones the oracle (== reference) consumed (SURVEY.md A.5)."""
    kw, B = CASES[alg]
    S, A = 17, 6
    init = O.init_state(alg, S, A, kw)
    okw = dict(critic_noise=torch.zeros(20, kw["feature_dim"])) if alg == "vlsac" else {}
    oracle = O.ORACLES[alg](S, A, init, discount=0.99, tau=0.005, **kw, **okw)
    ring = O.synthetic_ring(S, A, FakeBuffer.size, seed=0)
    drawn = []
    orig_take = ring.take
    ring.take = lambda ind: (drawn.append(np.array(ind)), orig_take(ind))[1]
    np.random.seed(11)
    torch.manual_seed(11)
    oracle.train(ring, B)
    np_state, torch_state = np.random.get_state()[1].copy(), torch.get_rng_state().clone()

    agent = AGENTS[alg](S, A, Space(A), **kw)
    np.random.seed(11)
    torch.manual_seed(11)
    idx, eps = agent._draw(FakeBuffer(), B)
    assert np.array_equal(np.random.get_state()[1], np_state)
    assert torch.equal(torch.get_rng_state(), torch_state)
    K = kw.get("extra_feature_steps", 0) + 1
    if alg == "diffsrsac":  # per feature iteration: B replay rows, then B noise levels (torch.randint, CPU generator)
        idx = idx.reshape(K, 2, B)
        assert idx[:, 1].min() >= 0 and idx[:, 1].max() < 1000
        idx = idx[:, 0].reshape(-1)
    assert np.array_equal(idx, np.concatenate(drawn))
    n_feat_eps = {"vlsac": K * B * kw.get("feature_dim", 0), "diffsrsac": K * B * S}.get(alg, 0)
    assert eps.shape == (n_feat_eps + 2 * B * A,)


def test_config_mapping_follows_reference_constructors():
    a = CTRLSACAgent(17, 6, Space(6), discount="0.99", tau="0.005", hidden_dim=1024, feature_dim=2048,
                     extra_feature_steps=3)  # main.py passes --discount/--tau as strings (SURVEY A.1)
    c = a._config(256)
    assert c.alg == _lib.ALG["ctrlsac"] and c.feature_steps == 4 and c.actor_hidden_dim == 256
    assert c.lr_feature == pytest.approx(1e-4) and c.lr_actor == pytest.approx(1e-4 / 3)  # ctrlsac_agent.py:195-197
    assert c.discount == pytest.approx(0.99) and c.feature_tau == pytest.approx(0.005)
    s = SACAgent(17, 6, Space(6), hidden_dim=256)
    c = s._config(256)
    assert c.lr_critic == pytest.approx(3e-4) and c.feature_steps == 0 and c.target_update_period == 2


@pytest.mark.parametrize("alg", list(CASES))
def test_initial_state_covers_the_oracle_parameter_table(alg):
    kw, _ = CASES[alg]
    agent = AGENTS[alg](17, 6, Space(6), **kw)
    want = O.init_state(alg, 17, 6, kw)
    have = agent.state_dict()
    assert set(want) <= set(have)
    for k, v in want.items():
        assert tuple(have[k].shape) == tuple(v.shape), k
    # actor: orthogonal rows / zero bias (utils/util.py:61-66)
    w = have["actor.trunk.2.weight"]
    assert torch.allclose(w @ w.t(), torch.eye(w.shape[0]), atol=1e-4)
    assert float(have["actor.trunk.0.bias"].abs().max()) == 0.0


def test_epilogue_struct_matches_header_layout():
    assert _lib.Epilogue.scale.offset == 60 and __import__("ctypes").sizeof(_lib.Epilogue) == 64


def test_drqv2_draw_consumes_the_generator_like_the_reference():
    """One updating train_step of the plain DrQ-v2 pixel agent: two RandomShiftsAug integer draws (float dtype, like
    network_arch/drqv2.py:43-47) and two _standard_normal([B, A]) draws, in that order; non-updating calls draw
    nothing.  Checked against the oracle, which is bit-identical to the real reference class (tests/golden/drqv2_*)."""
    import types
    from oracle import drq_oracle as D
    from rlrep_b200.pixel import DrQv2
    C_, A, bn, H, B = 3, 4, 16, 32, 4

    class Box:
        def __init__(self, shape):
            self.shape = shape
    args = types.SimpleNamespace(tau=0.01, update_every=2, critic_loss="mse", stddev_schedule="linear(1.0,0.1,500000)",
                                 stddev_clip=0.3, bn_dim=bn, actor_hidden_dim=H, critic_hidden_dim=H, encoder_lr=1e-4,
                                 actor_lr=1e-4, critic_lr=1e-4)
    agent = DrQv2(Box((C_, 84, 84)), Box((A,)), args)  # lazy: no device needed until the first update
    oracle = D.OracleDrQv2(A, D.init_state(C_, A, bn, H, seed=0))
    batch = D.synthetic_pixel_batch(B, C_, 84, A, seed=0)
    torch.manual_seed(7)
    assert oracle.train_step(batch, 0) != {}  # _step 1 -> 2: updates
    state_after_update = torch.get_rng_state().clone()
    assert oracle.train_step(batch, 0) == {}  # _step 3: no update, no draws
    assert torch.equal(torch.get_rng_state(), state_after_update)
    torch.manual_seed(7)
    shifts, eps = agent._draw(B)
    assert torch.equal(torch.get_rng_state(), state_after_update)
    assert shifts.shape == (2, B, 2) and shifts.dtype == np.int32 and shifts.min() >= 0 and shifts.max() <= 8
    assert eps.shape == (2, B, A)
    torch.manual_seed(7)
    want = torch.stack([D.draw_shift(B).reshape(B, 2) for _ in range(2)]).to(torch.int32).numpy()
    assert np.array_equal(shifts, want)
    assert agent.stddev_schedule(250000) == pytest.approx(0.55)


def test_mulvdrq_host_logic():
    """muLV-Rep DrQ-v2 shim without a device: RNG consumption of one update equals the oracle's (which is pinned to the
    real reference class, tests/golden/mulvdrq_b4.npz), `up_every` gating draws nothing, unsupported configuration
    switches raise, weight layouts round-trip through the pending state_dict, and the first device call raises without
    CUDA (no CPU fallback)."""
    from oracle import mulv_oracle as M
    from rlrep_b200 import RlrepError
    from rlrep_b200.pixel import MuLVDrQv2
    C_, A, F, H, B = 3, 4, 20, 32, 2
    cfg = dict(feat_dim=F, hid_dim=H, up_every=2)
    agent = MuLVDrQv2((C_, 84, 84), (A,), cfg)  # lazy: no device needed until the first update
    oracle = M.OracleMuLVDrQ(A, M.init_state(C_, A, F, H, seed=0))
    batch = M.synthetic_pixel_batch(B, C_, 84, A, seed=0)
    torch.manual_seed(7)
    assert oracle.update(batch, 0) != {}
    after = torch.get_rng_state().clone()
    assert oracle.update(batch, 1) == {} and torch.equal(torch.get_rng_state(), after)
    torch.manual_seed(7)
    shifts, eps_z, eps_act, noise = agent._draw(B)
    assert torch.equal(torch.get_rng_state(), after)
    assert shifts.shape == (2, B, 2) and eps_z.shape == (B, F) and eps_act.shape == (2, B, A) and noise.shape == (3, 20, F)
    assert agent.update(iter([]), step=1) == {}  # odd step: returns before touching the iterator or the device
    with pytest.raises(NotImplementedError):
        MuLVDrQv2((C_, 84, 84), (A,), dict(cfg, q_loss="mse"))
    with pytest.raises(NotImplementedError):
        MuLVDrQv2((C_, 84, 84), (A,), dict(cfg, pre_aug=True))
    sd = M.init_state(C_, A, F, H, seed=1)
    agent.load_state_dict(sd)  # kept pending until the handle exists
    assert set(agent.state_dict()) == set(sd)
    assert agent._kind("decoder.deconvnet.2.weight") == "deconv" and agent._kind("decoder.deconvnet.8.weight") == "outconv"
    assert agent._kind("feat_f_target.log_std_linear.1.weight") == "vec" and agent._kind("critic.l1.weight") == "mat"
    assert agent._ref_shape("predict_encoder.convnet.0.weight", 32, 27) == (32, 3, 3, 3)
    if not torch.cuda.is_available():
        with pytest.raises(RlrepError):
            agent.update(iter([tuple(batch)]), step=0)


def _shifted_row_gemm(A, Wk, conv_w):
    """CPU model of GemmArgs::conv_w (gemm.cuh): C[m, n] = sum_{t < 9, c < 32} A[m + (t // 3) * conv_w + t % 3, c] *
    Wk[n, t * 32 + c], rows past the end of A read as zero -- what the TMA producer's shifted row coordinate computes."""
    M = A.shape[0]
    Apad = torch.cat([A, torch.zeros(2 * conv_w + 2, A.shape[1], dtype=A.dtype)])
    out = torch.zeros(M, Wk.shape[0], dtype=A.dtype)
    for t in range(9):
        s = (t // 3) * conv_w + t % 3
        out += Apad[s:s + M] @ Wk[:, t * 32:(t + 1) * 32].T
    return out


def test_implicit_convolution_algebra():
    """The index algebra behind conv_implicit.cu, checked in float64 against torch's own operators:
    (1) valid 3x3 convolution = shifted-row GEMM on the input's own grid + compaction of the top-left (H-2)^2 block;
    (2) full correlation (the data gradient of that convolution, and a stride-1 ConvTranspose2d forward) = the same
        GEMM on a grid zero-padded by 2 with the taps flipped (t -> 8 - t) + compaction of the top-left (H+2)^2 block,
        for both weight layouts the kernels repack from (FC_CONV_DGRAD, FC_DECONV_FWD)."""
    import torch.nn.functional as F
    torch.manual_seed(0)
    B, H = 2, 7
    x = torch.randn(B, 32, H, H, dtype=torch.float64)
    w = torch.randn(32, 32, 3, 3, dtype=torch.float64)  # conv weight [co, ci, ky, kx]
    nhwc = lambda t: t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])  # [B*H*W, C]
    # (1) stored conv weight [co, (ky, kx, ci)]
    wk = w.permute(0, 2, 3, 1).reshape(32, 288)
    grid = _shifted_row_gemm(nhwc(x), wk, H).reshape(B, H, H, 32)[:, :H - 2, :H - 2]
    assert torch.allclose(grid.permute(0, 3, 1, 2), F.conv2d(x, w), atol=1e-10)
    # (2a) data gradient of the convolution: dX = full correlation of dY with W; repack [ci, (8 - t) -> t, co]
    dy = torch.randn(B, 32, H, H, dtype=torch.float64)
    want = F.conv_transpose2d(dy, w)  # == conv2d's input gradient for stride 1, no padding
    Wp = H + 4
    padded = F.pad(dy, (2, 2, 2, 2))
    flip = torch.empty(32, 288, dtype=torch.float64)
    for t in range(9):
        tap = 8 - t
        flip[:, t * 32:(t + 1) * 32] = wk[:, tap * 32:(tap + 1) * 32].T  # w_flip[ci, t*32 + co] = W[co, tap*32 + ci]
    grid = _shifted_row_gemm(nhwc(padded), flip, Wp).reshape(B, Wp, Wp, 32)[:, :H + 2, :H + 2]
    assert torch.allclose(grid.permute(0, 3, 1, 2), want, atol=1e-10)
    # (2b) ConvTranspose2d forward with the decoder's stored layout Wd[(ky, kx, co), ci] = W_ref[ci, co, ky, kx]
    wt = torch.randn(32, 32, 3, 3, dtype=torch.float64)  # reference layout [ci, co, ky, kx]
    wd = wt.permute(2, 3, 1, 0).reshape(288, 32)
    flip2 = torch.empty(32, 288, dtype=torch.float64)
    for t in range(9):
        tap = 8 - t
        flip2[:, t * 32:(t + 1) * 32] = wd[tap * 32:(tap + 1) * 32, :]  # w_flip[co, t*32 + ci] = Wd[tap*32 + co, ci]
    grid = _shifted_row_gemm(nhwc(F.pad(x, (2, 2, 2, 2))), flip2, Wp).reshape(B, Wp, Wp, 32)[:, :H + 2, :H + 2]
    assert torch.allclose(grid.permute(0, 3, 1, 2), F.conv_transpose2d(x, wt), atol=1e-10)


def test_latent_diffsr_draw_consumes_the_generator_like_the_reference():
    """Latent Diff-SR DrQ-v2 shim: the host-side randomness of one updating train_step -- shifts, posterior
    noise, diffusion levels / noise, the dropout masks of the online score network (drawn as Bernoulli(0.9) tensors, which
    is what F.dropout consumes), the action normals -- leaves the CPU generator exactly where the oracle (bit-identical
    to the reference class, tests/golden/ldiffsr_b4.npz) leaves it, and the masks are the ones the oracle applied."""
    import types
    import torch.nn.functional as F
    from oracle import ldiffsr_oracle as O
    from rlrep_b200.pixel import LatentDiffSRDrQv2
    d = O.Dims(4, 16, 32, 24, 32, 2, 32, 4, 64)

    class Box:
        def __init__(self, shape):
            self.shape = shape
    args = types.SimpleNamespace(use_repr_target=True, back_critic_grad=True, critic_loss="mse", reg_coef=0.0, grad_norm=None,
                                 extra_repr_step=1, do_scale=False, repr_coef=1.0, ae_num_layers=4, ae_num_filters=32,
                                 noise_schedule="linear", ae_lr=3e-4, score_lr=3e-4, actor_lr=1e-4, critic_lr=1e-4, bn_dim=d.bn,
                                 update_every=2, stddev_schedule="linear(1.0,0.1,500000)", stddev_clip=0.3, latent_dim=d.L,
                                 feature_dim=d.feat, psi_hidden_dim=d.psi_h, psi_hidden_depth=d.psi_d, zeta_hidden_dim=d.zeta_h,
                                 zeta_hidden_depth=d.zeta_d, actor_hidden_dim=d.H, critic_hidden_dim=d.H, noise_param1=1e-4,
                                 noise_param2=0.02, num_noises=1000, tau=0.01, kl_coef=1.0, ae_coef=1.0)
    agent = LatentDiffSRDrQv2(Box((9, 84, 84)), Box((d.A,)), args)
    oracle = O.OracleLatentDiffSR(d, O.init_state(d, seed=0))
    B = 3
    batch = O.synthetic_pixel_batch(B, 9, 84, d.A, seed=0)
    torch.manual_seed(11)
    assert oracle.train_step(batch, 0) != {}
    after = torch.get_rng_state().clone()
    torch.manual_seed(11)
    draws = agent._draw(B)
    assert torch.equal(torch.get_rng_state(), after)
    assert draws["psi_masks"].shape == (d.psi_d, 2 * B, d.psi_h) and draws["zeta_masks"].shape == (d.zeta_d, B, d.zeta_h)
    assert draws["eps_post"].shape == (4 * B, d.L) and draws["temb"].shape == (B, d.L // 2)
    assert set(np.unique(draws["psi_masks"])) <= {0.0, 1.0}
    torch.manual_seed(5)
    y = F.dropout(torch.ones(6, 10), 0.1, True)
    torch.manual_seed(5)
    assert torch.equal((y > 0).float(), torch.empty(6, 10).bernoulli_(0.9))
    with pytest.raises(NotImplementedError):
        LatentDiffSRDrQv2(Box((9, 84, 84)), Box((d.A,)), types.SimpleNamespace(**{**vars(args), "grad_norm": 1.0}))
