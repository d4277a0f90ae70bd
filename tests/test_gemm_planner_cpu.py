"""Host-side tile planner of the GEMM (csrc/gemm.cu: plan_tiles / wide_plan_cycles / plan_splits) -- pure host arithmetic behind the
C ABI, so it is checked without a GPU (148 SMs assumed when no device is visible).  `aoz_gemm_describe_plan` returns
bn + 1000*pair + 10000*tail_splits + 1000000*tail_tiles + 100000000*splits."""
import ctypes

import pytest

from aozora_sdxl_training_b200 import _lib


def plan(M, N, K, b_mn=0, splits=1):
    code = _lib.query("aoz_gemm_describe_plan", M, N, K, b_mn, splits)
    return dict(bn=code % 1000, pair=(code // 1000) % 10, tail_splits=(code // 10000) % 100, tail_tiles=(code // 1000000) % 100,
                splits=code // 100000000)


_FAKE_SCRATCH = ctypes.create_string_buffer(64)          # the planner only asks whether a scratch exists and how large it is


@pytest.fixture(autouse=True)
def _defaults():
    _lib.call("aoz_gemm_set_scratch", ctypes.addressof(_FAKE_SCRATCH), 24 << 20)
    yield
    from aozora_sdxl_training_b200 import ops
    if ops._gemm_scratch:                                       # same process as GPU tests: hand the real scratch back
        buf = next(iter(ops._gemm_scratch.values()))
        _lib.call("aoz_gemm_set_scratch", buf.data_ptr(), buf.numel())
    else:
        _lib.call("aoz_gemm_set_scratch", 0, 0)
    _lib.call("aoz_gemm_set_wide_mode", 1)
    _lib.call("aoz_gemm_set_wide_max_rounds", 2)
    _lib.call("aoz_gemm_set_tail_mode", 1)
    _lib.call("aoz_gemm_set_pair_mode", 1)


@pytest.mark.parametrize("K,b_mn", [(1280, 0), (1280, 1), (5120, 0), (3840, 1), (10240, 1)])
def test_projection_outputs_take_the_one_wave_wide_plan(K, b_mn):
    """4096 x 1280 outputs: 16 x 4 tiles of 256 x 320 on 74 SM pairs instead of 80 tiles of 256 x 256 (two rounds)."""
    p = plan(4096, 1280, K, b_mn)
    assert (p["bn"], p["pair"], p["tail_tiles"], p["splits"]) == (320, 1, 0, 1)


def test_wide_plan_needs_whole_320_column_tiles_and_few_rounds():
    assert plan(4096, 1024, 1280)["bn"] != 320                  # N is not a multiple of 320
    assert plan(128, 1280, 1280)["bn"] != 320                   # a single 128-row tile cannot form a CTA pair
    assert plan(65536, 320, 2880)["bn"] != 320                  # 256 tiles = 4 rounds of single-accumulator tiles
    assert plan(16384, 640, 5120, 1)["bn"] == 320               # 128 tiles = two rounds, no padded third column tile
    _lib.call("aoz_gemm_set_wide_max_rounds", 1)
    assert plan(16384, 640, 5120, 1)["bn"] != 320
    assert plan(4096, 1280, 1280)["bn"] == 320


def test_wide_plan_switches():
    _lib.call("aoz_gemm_set_wide_mode", 0)
    p = plan(4096, 1280, 1280)
    assert p["bn"] != 320 and p["bn"] <= 256
    _lib.call("aoz_gemm_set_wide_mode", 1)
    _lib.call("aoz_gemm_set_pair_mode", 0)                      # single-CTA tiles only: no pairs, no wide plan
    assert plan(4096, 1280, 1280)["pair"] == 0
    _lib.call("aoz_gemm_set_pair_mode", 1)
    _lib.call("aoz_gemm_set_tail_mode", 2)                      # a forced tail split keeps its plan (tests / experiments)
    p = plan(4096, 1280, 5120)
    assert p["bn"] != 320 and p["tail_tiles"] > 0 and p["tail_splits"] >= 2


def test_tail_split_covers_the_ragged_last_wave():
    """80 pair tiles on 74 SM pairs: the 6 tiles of the last wave are cut along K over the idle pairs (wide plan off)."""
    _lib.call("aoz_gemm_set_wide_mode", 0)
    p = plan(4096, 1280, 10240, 1)
    assert p["pair"] == 1 and p["bn"] == 256 and p["tail_tiles"] == 6 and 2 <= p["tail_splits"] <= 12
    assert p["tail_tiles"] * p["tail_splits"] <= 74


def test_auto_split_k_only_where_one_wave_is_mostly_empty():
    assert _lib.query("aoz_gemm_auto_splits", 4096, 1280, 1280, 0) == 1
    assert _lib.query("aoz_gemm_auto_splits", 4096, 10240, 1280, 0) == 1
    assert _lib.query("aoz_gemm_auto_splits", 640, 640, 16384, 1) > 1          # 25 tiles of a weight gradient with a long K
