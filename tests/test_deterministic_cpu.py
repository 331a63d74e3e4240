"""The deterministic-mode switch of the C ABI, without a GPU."""
from reactranker_b200 import _lib


def test_deterministic_switch_round_trips():
    L = _lib.lib()
    try:
        assert L.rr_get_deterministic() == 0
        assert L.rr_set_deterministic(1) == 0 and L.rr_get_deterministic() == 1
        assert L.rr_set_deterministic(0) == 0 and L.rr_get_deterministic() == 0
        assert L.rr_set_deterministic(2) == -1          # RR_ERR_INVALID
        assert L.rr_get_deterministic() == 0
    finally:
        L.rr_set_deterministic(0)
