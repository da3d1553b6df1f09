"""CPU suite: the library's option table (csrc/gd_options.cuh) holds exactly the switches tests and tools set; the names of
retired tuning switches are unknown to gd_set_option (no compute calls: the table is host state)."""
import pytest

from gnn_decode_b200 import _cabi, options

KEPT = ["GD_NO_LEAN", "GD_FORCE_STREAMED", "GD_FORCE_LIGHT", "GD_NO_CTAB", "GD_NO_VTAB", "GD_NO_VSKIP", "GD_LEAN_PARTS",
        "GD_LEAN_R", "GD_LEAN_G"]

# tuning experiments whose measured winner is now the only value (DESIGN.md keeps the numbers)
RETIRED = ["GD_CPS", "GD_NO_PWL", "GD_NO_RTAB", "GD_RTAB_N", "GD_CTAB_N", "GD_VTAB_N", "GD_VTAB_K", "GD_TILE", "GD_R", "GD_EB",
           "GD_NPOLY", "GD_NO_DIRECT", "GD_NO_LIGHT", "GD_LTILE", "GD_LR", "GD_GATE_CHUNKS", "GD_GATE_COPIES_FIRST", "GD_STILE",
           "GD_STHREADS", "GD_STREAM_LEGACY", "GD_SROWS", "GD_SSTAGES", "GD_SWARPS", "GD_NO_BWD_CTAB", "GD_LEAN_VTAB_N",
           "GD_LEAN_CTAB_N", "GD_LEAN_RTAB_N", "GD_NO_PDL",
           # switches of gd_decode_host's gated single launch, which is gone (the call runs on gd_pipeline)
           "GD_NO_GATED_HOST", "GD_LAUNCH_BLOCKING"]


@pytest.mark.parametrize("name", KEPT)
def test_kept_option_is_accepted(name):
    lib = _cabi.lib()
    assert lib.gd_set_option(name.encode(), 1, 0) == _cabi.GD_OK
    assert lib.gd_set_option(name.encode(), 0, 1) == _cabi.GD_OK


@pytest.mark.parametrize("name", RETIRED)
def test_retired_option_is_unknown(name):
    lib = _cabi.lib()
    assert lib.gd_set_option(name.encode(), 1, 0) == _cabi.GD_ERR_INVALID
    assert "unknown option" in lib.gd_last_error().decode()
    with pytest.raises(ValueError):
        options.set_option(name)
