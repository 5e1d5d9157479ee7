"""CPU: the C-ABI library loads and exports every symbol include/f5tts_b200.h declares; host-side guards raise."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "f5tts_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(f5_[a-z_0-9]+)\s*\(", src)))


def test_header_symbols_exported():
    from f5_tts_b200 import _lib

    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built (run __graft_entry__.build())")
    lib = _lib.lib()
    names = _declared()
    assert set(names) == set(_lib.EXPORTED_SYMBOLS), (names, _lib.EXPORTED_SYMBOLS)
    for n in names:
        assert hasattr(lib, n), n
    assert lib.f5_version() >= 100


def test_no_cpu_fallback():
    import f5_tts_b200 as F5
    from f5_tts_b200 import _lib, ops

    with pytest.raises(_lib.F5LibraryError):
        F5.MelSpec()(torch.zeros(1, 8000))
    with pytest.raises(_lib.F5LibraryError):
        ops.row_norm(torch.zeros(8, 128), 0, torch.zeros(128), torch.zeros(128))
    m = F5.DiT(dim=1024, depth=1, heads=16, ff_mult=2, text_dim=512, conv_layers=1, text_num_embeds=10)
    with pytest.raises(_lib.F5LibraryError):
        m.engine()  # parameters on CPU


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "f5_tts_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "import oracle" not in txt and "from oracle" not in txt, os.path.join(dirpath, f)


def test_state_dict_layout_matches_released_checkpoints():
    import f5_tts_b200 as F5
    from oracle import f5_oracle as O

    for cfg, cls in ((O.f5tts_base(), F5.DiT), (O.e2tts_base(), F5.UNetT)):
        m = F5.CFM(transformer=cls(dim=cfg.dim, depth=2 if cls is F5.DiT else 4, heads=cfg.heads, ff_mult=cfg.ff_mult,
                                   text_dim=cfg.text_dim, conv_layers=cfg.conv_layers, text_num_embeds=2545, mel_dim=100))
        cfg.depth = 2 if cls is F5.DiT else 4
        want = {k: tuple(s) for k, s, _ in O.state_dict_spec(cfg)}
        got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        assert got == want


def test_text_helpers():
    from f5_tts_b200 import infer

    assert infer.chunk_text("A b. C d! E", 5) == ["A b.", "C d!", "E"]
    toks = infer.convert_char_to_pinyin(["Hi there; ok"])[0]
    assert "".join(toks) == "Hi there, ok"


def test_gemm_tile_planner():
    """bn = 0 leaves the tile shape to the planner; the query entry point reports what f5_gemm will run (host logic only)."""
    from f5_tts_b200 import _lib, ops
    from f5_tts_b200.ops import ACT_GELU_ERF, ACT_NONE, EPI_F16, EPI_F32, EPI_QKV_ROPE, EPI_RESID

    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built (run __graft_entry__.build())")
    for M, N, K, epi, act in ((1876, 3072, 1024, EPI_QKV_ROPE, ACT_NONE), (1876, 1024, 2048, EPI_RESID, ACT_NONE),
                              (15008, 3072, 1024, EPI_QKV_ROPE, ACT_NONE), (300, 100, 1024, EPI_F32, ACT_NONE),
                              (700, 1024, 512, EPI_F16, ACT_GELU_ERF)):
        bn, pair = ops.gemm_tile(M, N, K, epi, act)
        assert bn in (64, 128, 192, 256) and pair in (0, 1)
        assert not (pair and epi == EPI_F32)
        if act == ACT_GELU_ERF:
            assert bn != 192 and not pair  # only instantiated shapes are ever chosen
    assert ops.gemm_tile(1876, 1024, 1024, EPI_RESID, ACT_NONE, bn=64) == (64, 0)  # explicit request is kept
    assert ops.gemm_tile(15008, 3072, 1024, EPI_QKV_ROPE, ACT_NONE) == (256, 1)  # large batch: cta_group::2 pairs


_FAKE_A, _FAKE_W, _FAKE_OUT, _FAKE_OUT2 = 0x7f0000000000, 0x7f0000100000, 0x7f0000200000, 0x7f0000300000


@pytest.mark.parametrize("case,want", [
    ("out16b_odd_ldo", "out16b"),      # F32 + out16b, ldo = n_out = 101: the fp16 copy's pair stores need ldo % 8 == 0
    ("f32_out_misaligned", "aligned out"),  # F32 full chunks are float4 stores
    ("f16_ldo", "ldo % 8"),            # fp16 TMA store rows must be 16-byte aligned
    ("resid_null", "resid != NULL"),
    ("qkv_no_tables", "rope tables"),
    ("lda_lt_k", "lda"),
])
def test_gemm_rejects_bad_layout_before_driver(case, want):
    """gemm_plan validates every argument before it encodes a tensor map, so a bad layout is reported as itself (never as
    a driver error, and identically with or without a GPU).  The pointers are fake: rejected calls never dereference them."""
    import ctypes as C

    from f5_tts_b200 import _lib
    from f5_tts_b200.ops import EPI_F16, EPI_F32, EPI_QKV_ROPE, EPI_RESID

    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built (run __graft_entry__.build())")
    g = _lib.GemmArgs()
    g.rows, g.batches, g.n_out, g.k, g.lda, g.ldw, g.bn, g.epi = 256, 1, 256, 128, 128, 128, 128, EPI_F16
    g.out, g.ldo = _FAKE_OUT, 256
    if case == "out16b_odd_ldo":
        g.epi, g.n_out, g.ldo, g.out16b = EPI_F32, 101, 101, _FAKE_OUT2
    elif case == "f32_out_misaligned":
        g.epi, g.out = EPI_F32, _FAKE_OUT + 4
    elif case == "f16_ldo":
        g.n_out, g.ldo = 100, 100
    elif case == "resid_null":
        g.epi, g.out = EPI_RESID, None
    elif case == "qkv_no_tables":
        g.epi, g.n_out, g.ldo, g.inner, g.seq = EPI_QKV_ROPE, 384, 384, 128, 128
    elif case == "lda_lt_k":
        g.lda = 64
    lib = _lib.lib()
    rc = lib.f5_gemm(_FAKE_A, _FAKE_W, C.byref(g), None)
    msg = lib.f5_last_error().decode()
    assert rc < 0 and want in msg and "cuTensorMap" not in msg, (rc, msg)
