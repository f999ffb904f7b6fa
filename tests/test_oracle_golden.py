"""CPU: the oracle (oracle/rl_oracle.py) against the committed golden fixtures, which were produced by running the
REAL reference agents in the build container (oracle/make_golden.py).  This is what pins the oracle."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import rl_oracle as O

GOLDEN = Path(__file__).resolve().parent / "golden"
# Intra-op threads of the machine the fixtures were recorded on.  CPU kernels split their reductions by thread count, and
# Adam's first step turns the last-bit differences of another split into +-lr moves (ldiffsr_b4 then misses its bar by up
# to 2.8x at 1, 3 or 16 threads), so the oracle runs with the recording's thread count wherever the suite runs.
GOLDEN_THREADS = 8


@pytest.fixture(autouse=True)
def golden_threads():
    before = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(before)


CASES = sorted(p.stem for p in GOLDEN.glob("*.npz") if not p.stem.startswith(("drqv2", "mulvdrq", "ldiffsr", "pixreplay")))
DRQ_CASES = sorted(p.stem for p in GOLDEN.glob("drqv2*.npz"))
MULV_CASES = sorted(p.stem for p in GOLDEN.glob("mulvdrq*.npz"))
LDIFFSR_CASES = sorted(p.stem for p in GOLDEN.glob("ldiffsr*.npz"))


def test_fixtures_present():
    assert {"sac_hc_b256", "ctrlsac_small", "ctrlsac_hc_b256", "vlsac_hc_b64", "vlsac_hum_b128", "spedersac_hc_b64",
            "diffsrsac_hc_b64"} <= set(CASES)
    assert {"drqv2_b8", "drqv2_b16_c3"} <= set(DRQ_CASES)
    assert {"mulvdrq_b4"} <= set(MULV_CASES)
    assert {"ldiffsr_b4"} <= set(LDIFFSR_CASES)


@pytest.mark.parametrize("name", CASES)
def test_oracle_reproduces_reference(name):
    z = np.load(GOLDEN / f"{name}.npz")
    meta = json.loads(bytes(z["meta_json"]).decode())
    infos = json.loads(bytes(z["infos_json"]).decode())
    alg, S, A, kw, B, rows, n = (meta[k] for k in ("alg", "S", "A", "kwargs", "batch", "rows", "n"))
    extra = {}
    if "extra/critic_noise" in z:
        extra["critic_noise"] = torch.from_numpy(z["extra/critic_noise"])
    init = O.init_state(alg, S, A, kw, seed=0)
    oracle = O.ORACLES[alg](S, A, init, discount=0.99, tau=0.005, **kw, **extra)
    ring = O.synthetic_ring(S, A, rows, seed=0)
    np.random.seed(1)
    torch.manual_seed(1)
    got = [oracle.train(ring, B) for _ in range(n)]
    for step, (g, w) in enumerate(zip(got, infos)):
        assert set(g) == set(w)
        for k in w:
            # fp32 scalars produced by the same op sequence: identical up to thread-count dependent summation order
            assert abs(g[k] - w[k]) <= 2e-6 + 2e-5 * abs(w[k]), (step, k, g[k], w[k])
    sd = oracle.state_dict()
    for k in meta["keys"]:
        t = sd[k].detach().double().flatten()
        stats, sample = z["stats/" + k], z["sample/" + k]
        stride = max(1, t.numel() // 256)
        got_sample = t[::stride][:256].numpy()
        # norm-wise (Adam amplifies 1-ulp gradient noise to 2*lr on isolated elements, SURVEY 7.2 #1)
        assert abs(t.norm().item() - stats[1]) <= 1e-5 * max(stats[1], 1e-6), k
        assert np.linalg.norm(got_sample - sample) <= 2e-5 * max(np.linalg.norm(sample), 1e-6) + 1e-7, k


def test_host_ring_follows_reference_semantics():
    """add() wrap-around, size saturation and fp64 -> fp32 cast at sample time (utils/buffer.py:28-48)."""
    ring = O.HostRing(3, 2, max_size=5)
    for i in range(7):
        ring.add(np.full(3, i + 0.1), np.full(2, -i), np.full(3, i + 0.5), i * 1.5, float(i == 6))
    assert ring.size == 5 and ring.ptr == 2
    b = ring.take(np.array([0, 1, 2]))
    assert b.state.dtype == torch.float32
    assert torch.equal(b.state[:, 0], torch.tensor([5.1, 6.1, 2.1], dtype=torch.float64).float())
    assert b.done[1].item() == 1.0 and b.reward.shape == (3, 1)
    np.random.seed(0)
    i1 = np.random.randint(0, 5, size=4)
    np.random.seed(0)
    assert torch.equal(ring.sample(4).state, ring.take(i1).state)


@pytest.mark.parametrize("name", DRQ_CASES)
def test_drq_oracle_reproduces_reference(name):
    """Plain DrQ-v2 pixel update (agent/diffsrdrq/drqv2.py:93-148): oracle/drq_oracle.py against fixtures produced by
    the real reference class (oracle/make_golden_drq.py)."""
    from oracle import drq_oracle as D
    z = np.load(GOLDEN / f"{name}.npz")
    meta = json.loads(bytes(z["meta_json"]).decode())
    infos = json.loads(bytes(z["infos_json"]).decode())
    C, A, bn, H, B, n = (meta[k] for k in ("C", "A", "bn_dim", "hidden_dim", "batch", "n"))
    oracle = D.OracleDrQv2(A, D.init_state(C, A, bn, H, seed=0))
    batches = [D.synthetic_pixel_batch(B, C, 84, A, seed=10 + i) for i in range(n)]
    torch.manual_seed(1)
    got = [oracle.train_step(b, step=1000 * i) for i, b in enumerate(batches)]
    assert [bool(g) for g in got] == [bool(w) for w in infos]  # update_every = 2: every other call is a no-op
    for step, (g, w) in enumerate(zip(got, infos)):
        assert set(g) == set(w)
        for k in w:
            assert abs(g[k] - w[k]) <= 2e-6 + 2e-5 * abs(w[k]), (step, k, g[k], w[k])
    sd = oracle.state_dict()
    for k in meta["keys"]:
        t = sd[k].detach().double().flatten()
        stats, sample = z["stats/" + k], z["sample/" + k]
        stride = max(1, t.numel() // 256)
        assert abs(t.norm().item() - stats[1]) <= 1e-5 * max(stats[1], 1e-6), k
        assert np.linalg.norm(t[::stride][:256].numpy() - sample) <= 2e-5 * max(np.linalg.norm(sample), 1e-6) + 1e-7, k


@pytest.mark.parametrize("name", MULV_CASES)
def test_mulvdrq_oracle_reproduces_reference(name):
    """muLV-Rep DrQ-v2 pixel update (agent/mulvdrq/drqv2.py:313-461): oracle/mulv_oracle.py against fixtures produced by
    the real reference class (oracle/make_golden_mulv.py).  Groundwork for SURVEY 8a row a16 (no CUDA path yet)."""
    from oracle import mulv_oracle as M
    z = np.load(GOLDEN / f"{name}.npz")
    meta = json.loads(bytes(z["meta_json"]).decode())
    infos = json.loads(bytes(z["infos_json"]).decode())
    C, A, Fd, H, B, n = (meta[k] for k in ("C", "A", "feat_dim", "hid_dim", "batch", "n"))
    oracle = M.OracleMuLVDrQ(A, M.init_state(C, A, Fd, H, seed=0))
    batches = [M.synthetic_pixel_batch(B, C, 84, A, seed=20 + i) for i in range(n)]
    torch.manual_seed(1)
    got = [oracle.update(b, step=2 * i) for i, b in enumerate(batches)]
    for step, (g, w) in enumerate(zip(got, infos)):
        assert set(g) == set(w)
        for k in w:
            assert abs(g[k] - w[k]) <= 2e-6 + 2e-5 * abs(w[k]), (step, k, g[k], w[k])
    assert oracle.update(batches[0], step=1) == {}  # up_every = 2: odd steps are no-ops and draw nothing
    sd = oracle.state_dict()
    for k in meta["keys"]:
        t = sd[k].detach().double().flatten()
        stats, sample = z["stats/" + k], z["sample/" + k]
        stride = max(1, t.numel() // 256)
        assert abs(t.norm().item() - stats[1]) <= 1e-5 * max(stats[1], 1e-6), k
        assert np.linalg.norm(t[::stride][:256].numpy() - sample) <= 2e-5 * max(np.linalg.norm(sample), 1e-6) + 1e-7, k


@pytest.mark.parametrize("name", LDIFFSR_CASES)
def test_ldiffsr_oracle_reproduces_reference(name):
    """Latent Diff-SR DrQ-v2 pixel update (agent/diffsrdrq/latent_diff_sr.py:306-390): oracle/ldiffsr_oracle.py against
    the fixture produced by the real reference class (oracle/make_golden_ldiffsr.py; bit-identical at generation time,
    dropout masks included).  Groundwork for SURVEY 8a row a17, second half (no CUDA path yet)."""
    from oracle import ldiffsr_oracle as O
    z = np.load(GOLDEN / f"{name}.npz")
    meta = json.loads(bytes(z["meta_json"]).decode())
    infos = json.loads(bytes(z["infos_json"]).decode())
    d, B, n = O.Dims(*meta["dims"]), meta["batch"], meta["n"]
    oracle = O.OracleLatentDiffSR(d, O.init_state(d, seed=0))
    batches = [O.synthetic_pixel_batch(B, 9, 84, d.A, seed=40 + i) for i in range(n)]
    torch.manual_seed(1)
    got = [oracle.train_step(b, step=1000 * i) for i, b in enumerate(batches)]
    assert [bool(g) for g in got] == [bool(w) for w in infos] == [True, False, True, False]
    for step, (g, w) in enumerate(zip(got, infos)):
        assert set(g) == set(w)
        for k in w:
            assert abs(g[k] - w[k]) <= 2e-6 + 2e-5 * abs(w[k]), (step, k, g[k], w[k])
    sd = oracle.state_dict()
    for k in meta["keys"]:
        t = sd[k].detach().double().flatten()
        stats, sample = z["stats/" + k], z["sample/" + k]
        stride = max(1, t.numel() // 256)
        assert abs(t.norm().item() - stats[1]) <= 1e-5 * max(stats[1], 1e-6), k
        assert np.linalg.norm(t[::stride][:256].numpy() - sample) <= 2e-5 * max(np.linalg.norm(sample), 1e-6) + 1e-7, k


def test_pixel_replay_oracle_matches_reference_fixture():
    """oracle/pixel_replay_oracle.py vs outputs of the real EfficientReplayBuffer (efficient_buffer.py:35-149) recorded by
    oracle/make_golden_pixreplay.py: valid mask, length and all six gathered arrays, bit for bit, across two ring wraps."""
    import numpy as np
    from pathlib import Path
    from oracle.pixel_replay_oracle import OraclePixelReplay, synthetic_stream
    g = np.load(Path(__file__).parent / "golden" / "pixreplay.npz")
    ora = OraclePixelReplay(61, 24, 3, 0.99, 3)
    for t, ts in enumerate(synthetic_stream(150, frame_stack=3, seed=5)):
        ora.add(ts)
        if f"idx_{t}" in g:
            assert np.array_equal(ora.valid, g[f"valid_{t}"]) and len(ora) == int(g[f"len_{t}"])
            got = ora.gather(g[f"idx_{t}"])
            for name, a in zip(("obs", "act", "rew", "dis", "nobs", "sobs"), got):
                assert a.dtype == g[f"{name}_{t}"].dtype and np.array_equal(a, g[f"{name}_{t}"]), (t, name)
