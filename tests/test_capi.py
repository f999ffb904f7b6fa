"""CPU: the C-ABI library loads without a GPU, exports every symbol include/rlrep_b200.h declares, and its compute
entry points fail loudly (error code + message) when there is no CUDA device -- there is no CPU fallback."""
import ctypes as C
import re
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]


def declared_symbols():
    text = (ROOT / "include" / "rlrep_b200.h").read_text()
    return sorted(set(re.findall(r"RLREP_EXPORT[^;]*?\b(rlrep_[a-z0-9_]+)\s*\(", text, flags=re.S)))


def test_header_declares_the_expected_surface():
    names = declared_symbols()
    for must in ("rlrep_gemm", "rlrep_ring_create", "rlrep_ring_gather", "rlrep_agent_create", "rlrep_agent_train",
                 "rlrep_agent_act", "rlrep_last_error"):
        assert must in names


def test_library_exports_every_declared_symbol(lib):
    missing = [n for n in declared_symbols() if not hasattr(lib, n)]
    assert not missing, missing
    assert lib.rlrep_abi_version() == 3


def test_python_binding_declares_every_symbol_it_uses(lib):
    from rlrep_b200 import _lib
    for n in declared_symbols():
        fn = getattr(_lib.load(), n)
        if n not in ("rlrep_abi_version", "rlrep_last_error"):
            assert fn.argtypes is not None, f"{n} has no ctypes signature in rlrep_b200/_lib.py"


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback(lib):
    h = C.c_void_p()
    rc = lib.rlrep_ring_create(17, 6, 1000, C.byref(h))
    assert rc != 0 and lib.rlrep_last_error()
    from rlrep_b200 import ReplayBuffer, RlrepError
    from rlrep_b200.agents import SACAgent
    import numpy as np
    with pytest.raises(RlrepError):
        ReplayBuffer(17, 6)

    class Sp:
        low, high = -np.ones(6), np.ones(6)
    agent = SACAgent(17, 6, Sp(), hidden_dim=32)  # construction is lazy; the first call that needs the device raises
    with pytest.raises(RlrepError):
        agent.select_action(np.zeros(17))


def _handle_entry_points():
    pixel = [n for n in declared_symbols() if re.match(r"rlrep_(drq|mulv|ldiff)_", n) and not n.endswith("_create")]
    return pixel + ["rlrep_agent_num_tensors", "rlrep_agent_tensor_info", "rlrep_agent_tensor_read",
                    "rlrep_agent_tensor_write"]


@pytest.mark.parametrize("name", _handle_entry_points())
def test_null_handle_is_an_error_not_a_crash(lib, name):
    """Every entry point that takes a pixel-agent handle, and the state agents' tensor accessors, reject a NULL handle
    with an error code and message before touching the device; destroying NULL is a no-op."""
    from rlrep_b200 import _lib
    fn = getattr(_lib.load(), name)
    args = [0.0 if t in (C.c_float, C.c_double) else 0 if t in (C.c_int, C.c_longlong) else None for t in fn.argtypes]
    # leave a different message behind first, so the one checked below is this call's
    assert lib.rlrep_agent_create_sharded(None, None, None, None) != 0
    if name.endswith("_destroy"):
        assert fn(*args) == 0
    else:
        assert fn(*args) != 0
        assert b"null argument" in lib.rlrep_last_error()
