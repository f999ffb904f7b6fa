"""Programmatic dependent launch (PDL) in the state agents' updates.

Every kernel of the chained CTRL-SAC update is launched with programmatic stream serialization, so in the captured graph
each kernel-to-kernel edge is programmatic: a kernel's CTAs start, and run the prologue that touches no data, while the
kernel before it finishes.  A kernel that read or wrote before its griddepcontrol.wait would race with its predecessor,
so these tests run many updates and require bit-identical results between fresh handles and between graph replay and
eager launches, at the benchmark's shapes."""
import numpy as np
import pytest
import torch

import bench
from oracle import rl_oracle as O

pytestmark = pytest.mark.gpu

N_UPDATES = 30
ROWS = 20_000

# The chained CTRL-SAC update at B = 256 is one stream of 38 kernels: tick, 4 x (gather, forward chain, contrastive
# head, backward chain, column reductions, Adam) -- the critic step's actor trunks run inside the last forward chain --
# then actor_sample (both samples), critic chain, TD head, column reductions, critic weight-gradient GEMM, Adam, critic
# hidden-layer GEMM, actor head, actor dgrad chain, actor_sample_bwd, actor backward chain, column reductions, Adam.
CTRLSAC_KERNELS = 38


def _run(name, use_graph, seed=5):
    from rlrep_b200 import ReplayBuffer
    from rlrep_b200.agents import AGENTS
    w = bench.WORKLOADS[name]
    S, A, kw = w["S"], w["A"], w["kw"]
    torch.manual_seed(seed)  # VLSAC draws its critic's fixed noise from the global generator at construction
    agent = AGENTS[w["alg"]](S, A, bench.Space(A), discount=0.99, tau=0.005, use_cuda_graph=use_graph, **kw)
    agent.load_state_dict(O.init_state(w["alg"], S, A, kw, seed=0))
    ring = O.synthetic_ring(S, A, ROWS, seed=0)
    buf = ReplayBuffer(S, A, max_size=ROWS)
    buf.load(ring.state, ring.action, ring.next_state, ring.reward, ring.done)
    np.random.seed(seed)
    torch.manual_seed(seed)
    infos = [agent.train(buf, w["B"]) for _ in range(N_UPDATES)]
    torch.cuda.synchronize()
    return agent, infos, agent.state_dict()


def _assert_identical(a, b):
    (_, infos_a, sd_a), (_, infos_b, sd_b) = a, b
    assert infos_a == infos_b
    assert sd_a.keys() == sd_b.keys()
    for k in sd_a:
        assert torch.equal(sd_a[k], sd_b[k]), k


def test_ctrlsac_graph_edges_are_programmatic():
    agent, _, _ = _run("ctrlsac_hc_b256", True)
    kernels, programmatic = agent._h.graph_stats
    assert agent.gpu_launches_last_train == CTRLSAC_KERNELS
    assert kernels == CTRLSAC_KERNELS
    # one stream, so kernels - 1 kernel-to-kernel edges, and the runtime refused none of them
    assert programmatic == CTRLSAC_KERNELS - 1


@pytest.mark.parametrize("name", ["ctrlsac_hc_b256", "sac_hc_b256", "spedersac_hc_b256", "diffsrsac_hc_b256",
                                  "vlsac_hum_b1024"])
def test_repeatable_and_replay_equals_eager(name):
    graph1 = _run(name, True)
    graph2 = _run(name, True)
    eager = _run(name, False)
    kernels, programmatic = graph1[0]._h.graph_stats
    print(f"{name}: {kernels} kernel nodes, {programmatic} programmatic edges, "
          f"{graph1[0].gpu_launches_last_train} launches per update")
    assert 0 < programmatic < kernels
    _assert_identical(graph1, graph2)
    _assert_identical(graph1, eager)
