"""xfm_attention_fwd_parts: the host-side query that sizes the forward's key-block scratch.  It needs no device, so it is
checked here with aligned placeholder addresses (nothing is dereferenced)."""
import ctypes as C
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


@pytest.fixture(scope="module")
def parts():
    from xfm_b200 import lib
    if not os.path.exists(lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    l = lib.load()

    def query(Lq, Lk, cross=False, **over):
        H, B = 12, 4
        p = lib.AttnParams()
        p.q = p.k = p.v = p.out = p.lse = 0x10000
        p.q_stride = p.k_stride = p.v_stride = p.o_stride = 3 * H * 64
        p.B, p.H, p.Lq, p.Lk, p.head_dim, p.Bkv, p.scale = B, H, Lq, Lk, 64, (2 if cross else B), 0.125
        p.allow_tc = 1
        if cross:
            p.kv_index = p.kv_offsets = p.kv_samples = 0x20000
        else:
            ws = int(round((Lk - 1) ** 0.5))
            p.rel_table, p.rel_window = 0x30000, ws
        for k, v in over.items():
            setattr(p, k, v)
        return l.xfm_attention_fwd_parts(C.byref(p))
    return query


@pytest.mark.parametrize("L,nb", [(197, 0), (577, 3), (901, 5)])
def test_key_block_count(parts, L, nb):
    assert parts(L, L) == nb                 # ViT self-attention with the closed-form table
    assert parts(L, L, rel_table=0) == nb    # ... and without a bias (VQ-KD tokenizer)
    assert parts(40, L, cross=True) == nb    # 40 text tokens attending to L image tokens


def test_paths_without_key_blocks(parts):
    assert parts(901, 901, allow_tc=0) == 0                    # mma.sync kernel requested
    assert parts(901, 901, kmask=0x40000) == 0                 # masked: streaming mma.sync fallback
    assert parts(901, 901, dropout_p=0.1) == 0
    assert parts(12, 901, cross=True) == 0                     # Lq != 40: streaming fallback
    assert parts(1025, 1025) == 0                              # W = 32: no tcgen05 instantiation
    assert parts(40, 901, cross=True, kmask=0x40000) == 0
