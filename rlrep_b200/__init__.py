"""rlrep_b200: B200-native (sm_100a) implementation of the rl-rep representation-learning update step.

Public surface mirrors the reference (haotiansun14/rl-rep): `ReplayBuffer`, `SACAgent`, `CTRLSACAgent`, ... with
the reference's constructor / `train` / `select_action` signatures.  All compute lives in librlrep_b200.so
(C ABI in include/rlrep_b200.h); build it with `python -m rlrep_b200.build`.
"""
from ._lib import RlrepError, load  # noqa: F401


def __getattr__(name):  # lazy: importing the package must not require torch.cuda
    if name in ("ReplayBuffer", "Batch"):
        from . import buffer
        return getattr(buffer, name)
    if name in ("SACAgent", "CTRLSACAgent", "VLSACAgent", "SPEDERSACAgent", "DIFFSRSACAgent", "ShardedCTRLSACAgent",
                "AGENTS"):
        from . import agents
        return getattr(agents, name)
    if name in ("ConvEncoder", "ConvDecoder", "DrQv2", "MuLVDrQv2", "LatentDiffSRDrQv2"):
        from . import pixel
        return getattr(pixel, name)
    if name == "PixelReplayBuffer":
        from . import pixel_replay
        return pixel_replay.PixelReplayBuffer
    if name == "SACPopulation":
        from . import sac_population
        return sac_population.SACPopulation
    if name == "Population":
        from . import population
        return population.Population
    raise AttributeError(name)
