"""sc_set_eval_cache / sc_eval_cache_stats reject a NULL engine before touching the device (no GPU needed)."""
import ctypes as C

import scb200

SC_E_INVAL = -1


def test_null_engine_is_rejected():
    L = scb200.load_library()
    assert L.sc_set_eval_cache(None, 16) == SC_E_INVAL
    assert "sc_set_eval_cache" in scb200.last_error()
    counts = scb200.EvalCacheCounts()
    assert L.sc_eval_cache_stats(None, C.byref(counts)) == SC_E_INVAL
    assert "sc_eval_cache_stats" in scb200.last_error()
