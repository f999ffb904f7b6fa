"""CPU: the SAC population entry points (rlrep_sacpop_*) are exported, bound in Python, and reject NULL handles and
buffers with an error code and message before touching the device."""
import ctypes as C
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def _sacpop_symbols():
    text = (ROOT / "include" / "rlrep_b200.h").read_text()
    return sorted(set(re.findall(r"RLREP_EXPORT[^;]*?\b(rlrep_sacpop_[a-z0-9_]+)\s*\(", text, flags=re.S)))


def test_population_surface_is_declared_and_exported(lib):
    names = _sacpop_symbols()
    for must in ("rlrep_sacpop_create", "rlrep_sacpop_train", "rlrep_sacpop_act", "rlrep_sacpop_train_resident",
                 "rlrep_sacpop_get_optim_state", "rlrep_sacpop_set_optim_state", "rlrep_sacpop_tensor_read",
                 "rlrep_sacpop_last_launches"):
        assert must in names
    assert all(hasattr(lib, n) for n in names)


@pytest.mark.parametrize("name", [n for n in _sacpop_symbols() if n != "rlrep_sacpop_metric_name"])
def test_null_population_handle_is_an_error_not_a_crash(lib, name):
    from rlrep_b200 import _lib
    fn = getattr(_lib.load(), name)
    args = [0.0 if t in (C.c_float, C.c_double) else 0 if t in (C.c_int, C.c_longlong) else None for t in fn.argtypes]
    assert lib.rlrep_agent_create_sharded(None, None, None, None) != 0  # a different message first
    if name.endswith("_destroy"):
        assert fn(*args) == 0
    else:
        assert fn(*args) != 0
        assert b"null argument" in lib.rlrep_last_error()


def test_null_population_metric_name(lib):
    from rlrep_b200 import _lib
    assert _lib.load().rlrep_sacpop_metric_name(None, 0) is None
    assert b"null argument" in lib.rlrep_last_error()


def test_population_class_is_exported_lazily():
    import rlrep_b200
    from rlrep_b200.sac_population import SACPopulation
    assert rlrep_b200.SACPopulation is SACPopulation
