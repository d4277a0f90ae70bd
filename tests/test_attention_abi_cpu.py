"""CPU test of the attention entry points' argument checks: the backward form switch accepts exactly its two forms."""
import pytest

from aozora_sdxl_training_b200 import _lib


def test_attention_bwd_mode_accepts_only_its_two_forms():
    try:
        for bad in (1, 3, -1):
            with pytest.raises(_lib.AozoraError) as e:
                _lib.call("aoz_attn_set_bwd_mode", bad)
            assert "aoz_attn_set_bwd_mode" in str(e.value)
        for good in (0, 2):
            _lib.call("aoz_attn_set_bwd_mode", good)
    finally:
        _lib.call("aoz_attn_set_bwd_mode", 2)
