"""GPU: the kernel-level contracts the engine builds on that the end-to-end parity tests cannot resolve.

Variable-length execution (engine.cu build_step_plans / run_prologue) relies on the GEMM skipping tiles that hold only
padding, masking the padded rows of the tiles it computes, indexing gates by the device step counter, and on the
attention kernel masking keys past kv_len exactly.  A fault confined to the rows next to a sample's end or to one tile
shape barely moves an utterance-level rel-L2, so every case here compares one kernel call against a float64 torch
reference computed from the same fp16-rounded operands, at the tile / chunk boundaries where kernels go wrong.

Tolerances are those of test_gpu_kernels.py: fp32 rel-L2 <= 2e-4; fp16 rel-L2 <= 1.5e-3 and max-abs <= 4e-3 * max|ref|;
attention rel-L2 <= 3e-3.  Outputs are pre-filled with a finite sentinel and every output buffer has spare rows past M and
spare columns past n_out; whatever the code guarantees bit for bit is asserted with torch.equal.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

from f5_tts_b200 import ops  # noqa: E402
from f5_tts_b200.ops import (ACT_GELU_ERF, ACT_GELU_TANH, ACT_NONE, EPI_F16, EPI_F32, EPI_QKV_ROPE,  # noqa: E402
                             EPI_RESID)

DEV = "cuda:0"
S16, S32 = -1234.0, -12345.0  # sentinels: finite, and no kernel output of these tests comes near them
SPARE_ROWS = 3


def gen(shape, seed, scale=1.0, dtype=torch.float16):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dtype).to(DEV)


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300))


def check_f16(got, ref, what):
    d = float((got.double() - ref).abs().max())
    r = rel(got, ref)
    print(f"[{what}] rel-L2 {r:.3e} max|d| {d:.3e} max|ref| {float(ref.abs().max()):.3e}")
    assert r <= 1.5e-3, what
    assert d <= 4e-3 * float(ref.abs().max()), what


def check_f32(got, ref, what):
    r = rel(got, ref)
    print(f"[{what}] rel-L2 {r:.3e}")
    assert r <= 2e-4, what


def canvas(rows, cols, dtype, ldo=None):
    """Sentinel-filled [rows + SPARE_ROWS, ldo] buffer and its [rows, cols] output view (row stride ldo)."""
    ldo = ldo if ldo is not None else cols + 8 + (-cols) % 8
    full = torch.full((rows + SPARE_ROWS, ldo), S16 if dtype == torch.float16 else S32, dtype=dtype, device=DEV)
    return full, full[:rows, :cols]


def untouched(full, rows, cols):
    """The spare rows past M and the gap columns past n_out still hold the sentinel."""
    s = S16 if full.dtype == torch.float16 else S32
    assert bool((full[rows:] == s).all()), "write past the last row"
    assert bool((full[:, cols:] == s).all()), "write past n_out"


def strided(t, seed):
    """t [R, K] copied into a wider row-strided buffer (ld > K) whose gap columns hold +-6e4: a GEMM that read the gap
    instead of taking the K tail from TMA zero fill would be off by orders of magnitude."""
    R, K = t.shape
    ld = K + 24 + (-K) % 8
    g = torch.Generator().manual_seed(seed)
    full = (torch.randint(0, 2, (R, ld), generator=g) * 1.2e5 - 6e4).half().to(DEV)
    full[:, :K] = t
    return full[:, :K]


def ref_linear(a, w, bias, act=ACT_NONE):
    y = a.double() @ w.double().t()
    if bias is not None:
        y = y + bias.double()
    if act == ACT_GELU_TANH:
        y = F.gelu(y, approximate="tanh")
    elif act == ACT_GELU_ERF:
        y = F.gelu(y)
    return y


def ref_rope(y, seq, inner, pe_heads, cs, sn):
    """RoPE of the q and k sections of the first pe_heads heads (EPI_QKV_ROPE, interleaved pairs, position = row % seq)."""
    M = y.shape[0]
    y = y.view(M // seq, seq, 3, inner // 64, 32, 2)
    c, s = cs.double().view(1, seq, 1, 1, 32), sn.double().view(1, seq, 1, 1, 32)
    rot = torch.stack((y[..., 0] * c - y[..., 1] * s, y[..., 1] * c + y[..., 0] * s), dim=-1)
    out = y.clone()
    out[:, :, :2, :pe_heads] = rot[:, :, :2, :pe_heads]
    return out.reshape(M, 3 * inner)


def row_classes(M, seq, lens, tm):
    """(valid, skipped, padded) row masks of a plain GEMM with row_len: valid = position < row_len of its sample; skipped =
    rows of a tm-row tile that lies inside one sample and starts at or past its row_len (gemm.cuh tile_is_padding);
    padded = the remaining rows past row_len, computed and masked."""
    r = torch.arange(M)
    valid = (r % seq) < torch.tensor(lens)[r // seq]
    skipped = torch.zeros(M, dtype=torch.bool)
    for m0 in range(0, M, tm):
        last = min(m0 + tm, M) - 1
        b0 = m0 // seq
        if b0 == last // seq and m0 - b0 * seq >= lens[b0]:
            skipped[m0:last + 1] = True
    return valid.to(DEV), skipped.to(DEV), (~valid & ~skipped).to(DEV)


# ------------------------------------------------------------------------------------------------------------------
# GEMM: padded-tile skipping
# ------------------------------------------------------------------------------------------------------------------

# engine call site -> (epi, act, pe_heads); tile widths instantiated in gemm.cu configure_kernels (single CTA, CTA pair)
_SITES = {
    "f16": (EPI_F16, ACT_NONE, 0, (64, 128, 192, 256), (128, 192, 256)),
    "ff1_gelu_tanh": (EPI_F16, ACT_GELU_TANH, 0, (64, 128, 192, 256), (128, 192, 256)),
    "f16_gelu_erf": (EPI_F16, ACT_GELU_ERF, 0, (64, 128, 256), ()),
    "oproj_ff2_resid_gate": (EPI_RESID, ACT_NONE, 0, (64, 128, 192, 256), (128, 192, 256)),
    "qkv_rope_pe1": (EPI_QKV_ROPE, ACT_NONE, 1, (128, 192, 256), (128, 192, 256)),
    "qkv_rope_pe_all": (EPI_QKV_ROPE, ACT_NONE, 4, (128, 192, 256), (128, 192, 256)),
    "input_proj_f32_out16b": (EPI_F32, ACT_NONE, 0, (64, 128, 256), ()),
}
_SKIP_CASES = [pytest.param(site, bn, pair, id=f"{site}-bn{bn}{'-pair' if pair else ''}")
               for site, (_, _, _, single, pairs) in _SITES.items()
               for bn, pair in [(b, 0) for b in single] + [(b, 1) for b in pairs]]
# (seq, per-sample row_len): seq not a multiple of 128; lengths = full sample, 128, 129, 256, 257 and 1
_LAYOUTS = [(300, [300, 128, 129, 1]), (700, [256, 257, 700, 1])]


@pytest.mark.parametrize("site,bn,pair", _SKIP_CASES)
def test_gemm_skip_padded_tiles(site, bn, pair):
    """engine.cu build_step_plans with skip_padded_tiles (input projection, QKV, out-proj, FF1, FF2) and
    gemm.cuh tile_is_padding.  engine.cu run_prologue clears h0h / c1 / qkv once per call and relies on exactly this:
    tiles wholly past row_len are never written (sentinel survives in out, out16b and resid), padded rows of computed
    tiles are masked (fp16 0, residual unchanged, out16b 0; the F32 output itself is unmasked)."""
    epi, act, pe_heads, _, _ = _SITES[site]
    K, inner = 256, 256
    N = 3 * inner if epi == EPI_QKV_ROPE else 512
    for li, (seq, lens) in enumerate(_LAYOUTS):
        Be = len(lens)
        M = Be * seq
        what = f"{site} bn{bn} pair{pair} seq{seq}"
        a, w = gen((M, K), 100 + li), gen((N, K), 110 + li, 1 / math.sqrt(K))
        bias = gen((N,), 120 + li, 0.5, torch.float32)
        assert ops.gemm_tile(M, N, K, epi, act, bn, pair) == (bn, pair)
        valid, skipped, padded = row_classes(M, seq, lens, 256 if pair else 128)
        assert bool(skipped.any()) and bool(padded.any())  # the layout reaches all three row classes
        kw = dict(epi=epi, act=act, bn=bn, pair=pair, row_len=torch.tensor(lens, dtype=torch.int32, device=DEV), seq=seq,
                  skip_padded=True, static_w=True)
        y = ref_linear(a, w, bias, act)
        if epi == EPI_RESID:
            gate = gen((N,), 130 + li, 0.5, torch.float32)
            full, x = canvas(M, N, torch.float32)
            x0 = gen((M, N), 140 + li, 1.0, torch.float32)
            x.copy_(x0)
            ops.linear(a, w, bias, resid=x, gate=gate, **kw)
            check_f32(x[valid], x0[valid] + gate.double() * y[valid], what)
            # skipped rows: never touched; padded rows of computed tiles: reduce-add of an exact 0
            assert torch.equal(x[~valid], x0[~valid]), what
            untouched(full, M, N)
        elif epi == EPI_F32:
            full, o = canvas(M, N, torch.float32)
            full16, o16 = canvas(M, N, torch.float16, ldo=full.shape[1])
            ops.linear(a, w, bias, out=o, out16b=o16, **kw)
            check_f32(o[~skipped], y[~skipped], what)
            assert bool((o[skipped] == S32).all()) and bool((o16[skipped] == S16).all()), what
            # one __float2half_rn of the same fp32 value, the same rounding as Tensor.half()
            assert torch.equal(o16[valid], o[valid].half()), what
            assert bool((o16[padded] == 0).all()), what
            untouched(full, M, N)
            untouched(full16, M, N)
        else:
            if epi == EPI_QKV_ROPE:
                cs, sn = ops.rope_tables(seq, DEV)
                kw.update(rope=(cs, sn), inner=inner, pe_heads=pe_heads)
                y = ref_rope(y, seq, inner, pe_heads, cs, sn)
            full, o = canvas(M, N, torch.float16)
            ops.linear(a, w, bias, out=o, **kw)
            check_f16(o[valid], y[valid], what)
            assert bool((o[skipped] == S16).all()), what
            assert bool((o[padded] == 0).all()), what
            untouched(full, M, N)


@pytest.mark.parametrize("resid", [False, True], ids=["conv1_f16", "conv2_resid"])
def test_conv_skip_padded_tiles(resid):
    """engine.cu conv position embedding (conv1 F16 -> c1, conv2 RESID into h0) with skip_padded_tiles over batches > 1:
    gemm.cuh tile_is_padding<CONV> skips a 128-row tile when m0 >= row_len[b]."""
    B, N, D = 4, 700, 256
    lens = [700, 257, 128, 1]
    pos = torch.arange(N, device=DEV)[None, :]
    lt = torch.tensor(lens, dtype=torch.int32, device=DEV)
    valid = pos < lt[:, None].long()
    skipped = (pos // 128 * 128) >= lt[:, None].long()
    padded = ~valid & ~skipped
    assert bool(skipped.any()) and bool(padded.any())
    x = gen((B, N, D), 150)
    x = torch.where(valid[..., None], x, torch.zeros_like(x)).contiguous()  # the engine's cleared h0h
    w = gen((D, 64, 31), 151, 1 / math.sqrt(64 * 31))
    bias = gen((D,), 152, 0.1, torch.float32)
    wp = w.permute(2, 0, 1).contiguous()
    y = F.conv1d(x.double().cpu().transpose(1, 2), w.double().cpu(), bias.double().cpu(), padding=15,
                 groups=D // 64).transpose(1, 2).to(DEV)
    ref = y * torch.tanh(F.softplus(y))  # Mish
    if resid:
        full = torch.full((B * N + SPARE_ROWS, D), S32, dtype=torch.float32, device=DEV)
        r = full[:B * N].view(B, N, D)
        r0 = gen((B, N, D), 153, 1.0, torch.float32)
        r.copy_(r0)
        ops.grouped_conv31(x, wp, bias, resid=r, row_len=lt, skip_padded=True)
        check_f32(r[valid], r0[valid] + ref[valid], "conv2 resid")
        assert torch.equal(r[~valid], r0[~valid])
    else:
        full = torch.full((B * N + SPARE_ROWS, D), S16, dtype=torch.float16, device=DEV)
        o = full[:B * N].view(B, N, D)
        ops.grouped_conv31(x, wp, bias, out=o, row_len=lt, skip_padded=True)
        check_f16(o[valid], ref[valid], "conv1 f16")
        assert bool((o[skipped] == S16).all()) and bool((o[padded] == 0).all())
    assert bool((full[B * N:] == (S32 if resid else S16)).all())


# ------------------------------------------------------------------------------------------------------------------
# GEMM: step-indexed gate, out16b, strides and tails, static-W prefetch
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("bn,pair", [(64, 0), (192, 0), (256, 1)])
def test_resid_gate_follows_device_step(bn, pair):
    """engine.cu out-proj / FF2 of a DiT layer: gate = L.mod + i*6D + {2,5}D read at row *step_ptr of the modulation
    table (stride modW > n_out), i.e. the gate follows the device step counter, not a value fixed at plan time."""
    M, N, K, S = 300, 512, 256, 5
    stride, off = 8 * N, 2 * N + 4
    a, w = gen((M, K), 160), gen((N, K), 161, 1 / math.sqrt(K))
    bias = gen((N,), 162, 0.5, torch.float32)
    table = gen((S, stride), 163, 0.5, torch.float32)
    x0 = gen((M, N), 164, 1.0, torch.float32)
    y = ref_linear(a, w, bias)
    step = torch.zeros(1, dtype=torch.int32, device=DEV)
    for s in (0, S - 1):
        step.fill_(s)
        x = x0.clone()
        ops.linear(a, w, bias, epi=EPI_RESID, bn=bn, pair=pair, resid=x, gate=table.view(-1)[off:], step_ptr=step,
                   gate_stride=stride)
        check_f32(x, x0 + table[s, off:off + N].double() * y, f"step gate s={s}")


@pytest.mark.parametrize("bn", [64, 128, 256])
def test_f32_out16b_odd_n_out(bn):
    """gemm.cuh F32 epilogue with out16b (the input projection's masked fp16 copy) at an odd n_out = 101, ldo = 104:
    the tail stores of the fp16 copy stop at column n_out - 1 (the gap columns keep the sentinel)."""
    M, N, K, seq = 300, 101, 192, 150
    lens = [150, 77]
    a, w = gen((M, K), 170), gen((N, K), 171, 1 / math.sqrt(K))
    bias = gen((N,), 172, 0.5, torch.float32)
    full, o = canvas(M, N, torch.float32, ldo=104)
    full16, o16 = canvas(M, N, torch.float16, ldo=104)
    ops.linear(a, w, bias, epi=EPI_F32, bn=bn, out=o, out16b=o16, row_len=torch.tensor(lens, dtype=torch.int32,
                                                                                       device=DEV), seq=seq)
    valid = row_classes(M, seq, lens, 128)[0]
    check_f32(o, ref_linear(a, w, bias), f"f32 n101 bn{bn}")
    assert torch.equal(o16[valid], o[valid].half())
    assert bool((o16[~valid] == 0).all())
    untouched(full, M, N)
    untouched(full16, M, N)


# (site, bn, pair, n_out, k, bias): K tails 100 / 712 / 1000 read through lda, ldw > k; ldo > n_out; M = 300 clips the
# last 128-row tile and, for pairs, leaves every row of the second CTA of the last pair tile past M
_TAIL_CASES = [
    ("f16", 64, 0, 200, 100, False), ("f16", 128, 0, 264, 712, True), ("f16", 192, 0, 1000, 1000, True),
    ("f16", 256, 0, 264, 100, True), ("f16", 128, 1, 264, 1000, True), ("f16", 192, 1, 264, 712, False),
    ("f16", 256, 1, 1000, 100, True),
    ("resid", 64, 0, 264, 1000, True), ("resid", 128, 0, 1000, 100, False), ("resid", 192, 0, 200, 712, True),
    ("resid", 256, 0, 1000, 712, True), ("resid", 128, 1, 264, 100, True), ("resid", 192, 1, 264, 1000, True),
    ("resid", 256, 1, 1000, 712, False),
    ("qkv", 128, 0, 384, 100, True), ("qkv", 192, 0, 384, 712, True), ("qkv", 128, 1, 384, 712, False),
    ("qkv", 256, 1, 384, 1000, True),
]


@pytest.mark.parametrize("site,bn,pair,n_out,k,with_bias", [
    pytest.param(*c, id=f"{c[0]}-bn{c[1]}{'-pair' if c[2] else ''}-n{c[3]}-k{c[4]}{'' if c[5] else '-nobias'}")
    for c in _TAIL_CASES])
def test_gemm_strides_and_tails(site, bn, pair, n_out, k, with_bias):
    """gemm.cu tensor maps: A / W read with lda, ldw > k (the K tail is TMA zero fill, never the gap), the staged TMA
    epilogues clip columns at n_out with ldo > n_out and rows at M, bias == NULL."""
    M, seq = 300, 150
    a = strided(gen((M, k), 180), 181)
    w = strided(gen((n_out, k), 182, 1 / math.sqrt(k)), 183)
    assert a.stride(0) > k and w.stride(0) > k
    bias = gen((n_out,), 184, 0.5, torch.float32) if with_bias else None
    y = ref_linear(a, w, bias)
    what = f"{site} bn{bn} pair{pair} n{n_out} k{k}"
    if site == "resid":
        gate = gen((n_out,), 185, 0.5, torch.float32)
        full, x = canvas(M, n_out, torch.float32)
        x0 = gen((M, n_out), 186, 1.0, torch.float32)
        x.copy_(x0)
        ops.linear(a, w, bias, epi=EPI_RESID, bn=bn, pair=pair, resid=x, gate=gate)
        check_f32(x, x0 + gate.double() * y, what)
    else:
        full, o = canvas(M, n_out, torch.float16)
        kw = {}
        if site == "qkv":
            inner = n_out // 3
            cs, sn = ops.rope_tables(seq, DEV)
            kw = dict(epi=EPI_QKV_ROPE, seq=seq, rope=(cs, sn), inner=inner, pe_heads=1)
            y = ref_rope(y, seq, inner, 1, cs, sn)
        ops.linear(a, w, bias, bn=bn, pair=pair, out=o, **kw)
        check_f16(o, y, what)
    untouched(full, M, n_out)


@pytest.mark.parametrize("bn,pair,k", [(64, 0, 64), (64, 0, 192), (64, 0, 448), (64, 0, 512), (256, 0, 64),
                                       (256, 0, 192), (256, 0, 448), (256, 1, 192), (256, 1, 320), (256, 1, 448)])
def test_static_weight_prefetch(bn, pair, k):
    """gemm.cuh producer: with weights_static the first min(num_kb, STAGES) W tiles are issued before the programmatic-
    launch wait (STAGES = 7 at bn 64, 3 at bn 256, 5 on 256-wide pairs), then the ring continues over later tiles of the
    persistent CTA.  num_kb below, equal to and above STAGES; more tiles than SMs (pairs) so the ring wraps."""
    M, N = 4800, 1024
    a, w = gen((M, k), 190), gen((N, k), 191, 1 / math.sqrt(k))
    bias = gen((N,), 192, 0.5, torch.float32)
    out = ops.linear(a, w, bias, bn=bn, pair=pair)
    out_s = ops.linear(a, w, bias, bn=bn, pair=pair, static_w=True)
    assert torch.equal(out_s, out)  # the prefetch changes when W arrives, not what is computed
    check_f16(out_s, ref_linear(a, w, bias), f"prefetch bn{bn} pair{pair} k{k}")


# ------------------------------------------------------------------------------------------------------------------
# Attention
# ------------------------------------------------------------------------------------------------------------------

def attn_ref(qkv, Be, seq, H, kv, scale):
    """float64 softmax(q k^T * scale) v of every sample over its first kv[b] keys, [Be*seq, H*64]."""
    x = qkv.double().view(Be, seq, 3, H, 64)
    out = []
    for b in range(Be):
        L = seq if kv is None else kv[b]
        q, k, v = x[b, :, 0].transpose(0, 1), x[b, :L, 1].transpose(0, 1), x[b, :L, 2].transpose(0, 1)
        p = torch.softmax(q @ k.transpose(1, 2) * scale, dim=-1)
        out.append((p @ v).transpose(0, 1).reshape(seq, H * 64))
    return torch.cat(out)


def written_rows(Be, seq, kv):
    """Rows f5_attention writes: with kv_len, the 256-row query blocks starting before kv_len[b] (attn.cuh early exit)."""
    w = torch.zeros(Be, seq, dtype=torch.bool)
    for b in range(Be):
        for q0 in range(0, seq, 256):
            w[b, q0:q0 + 256] = kv is None or q0 < kv[b]
    return w.view(-1).to(DEV)


def run_attention(qkv, Be, seq, H, kv, scale=0.125):
    full = torch.full((Be * seq + SPARE_ROWS, H * 64), S16, dtype=torch.float16, device=DEV)
    kv_t = None if kv is None else torch.tensor(kv, dtype=torch.int32, device=DEV)
    out = ops.attention(qkv, Be, seq, H, kv_t, scale=scale, out=full[:Be * seq])
    assert bool((full[Be * seq:] == S16).all()), "write past the last sample"
    return out


def check_attention(out, qkv, Be, seq, H, kv, scale, what):
    wr = written_rows(Be, seq, kv)
    assert bool((out[~wr] == S16).all()), f"{what}: a query block at or past kv_len was written"
    ref = attn_ref(qkv, Be, seq, H, kv, scale)
    worst = 0.0
    for b in range(Be):
        rows = torch.zeros_like(wr)
        rows[b * seq:(b + 1) * seq] = True
        rows &= wr
        r = rel(out[rows], ref[rows])
        worst = max(worst, r)
        assert r <= 3e-3, f"{what}: sample {b} (kv_len {None if kv is None else kv[b]}) rel-L2 {r:.3e}"
    print(f"[{what}] worst per-sample rel-L2 {worst:.3e}")
    return wr


# kv_len = 256 + r: last-tile key counts on both sides of the 32 / 64 / 96 chunk boundaries and of the 16-key P.V steps
_SWEEP = [256 + r for r in (1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 95, 96, 97, 111, 112, 113, 127, 128)] + [1, 33, 97, 127]


def test_attention_key_length_sweep():
    """attn.cuh last key tile of a sample (kv_rem = kv_len - 128 j): mask_tail32 in chunk 0 / 1 / 2 / 3 including the
    kv_rem in [96, 128) branch and the exact 32 / 64 / 96 boundaries, P.V step counts nkk = 1..8, single-tile samples.
    Then the keys and values past kv_len are set to +-6e4: masked scores become -inf before the max and their P is an
    exact 0, so every written row is bit-identical."""
    seq, H = 384, 2
    Be = len(_SWEEP)
    qkv = gen((Be * seq, 3 * H * 64), 200)
    out = run_attention(qkv, Be, seq, H, _SWEEP)
    wr = check_attention(out, qkv, Be, seq, H, _SWEEP, 0.125, "kv sweep")
    g = torch.Generator().manual_seed(201)
    big = (torch.randint(0, 2, (Be, seq, 2, H * 64), generator=g) * 1.2e5 - 6e4).half().to(DEV)
    q2 = qkv.clone().view(Be, seq, 3, H * 64)
    for b, L in enumerate(_SWEEP):
        q2[b, L:, 1:] = big[b, L:]
    out2 = run_attention(q2.view(Be * seq, -1), Be, seq, H, _SWEEP)
    assert torch.equal(out2[wr], out[wr])


@pytest.mark.parametrize("seq", [1, 2, 31, 97, 127, 225, 353, 383])
def test_attention_no_kv_len(seq):
    """f5_attention without kv_len (the reference's unmasked mode): the last key tile of each sample is masked at seq and
    the 3-D tensor map zero-fills rows past seq, so nothing of the adjacent sample leaks in (Be = 3)."""
    Be, H = 3, 2
    qkv = gen((Be * seq, 3 * H * 64), 210 + seq)
    out = run_attention(qkv, Be, seq, H, None)
    check_attention(out, qkv, Be, seq, H, None, 0.125, f"no kv_len seq{seq}")


@pytest.mark.parametrize("scale", [0.125, 0.05, 0.3])
def test_attention_query_block_exit(scale):
    """attn.cuh early exit: with kv_len a 256-row query block starting at q0 is computed exactly when q0 < kv_len[b],
    other blocks are left unwritten (sentinel).  Also the softmax scale argument."""
    seq, H = 700, 2
    kv = [700, 256, 255, 257, 1, 513]
    Be = len(kv)
    qkv = gen((Be * seq, 3 * H * 64), 220)
    out = run_attention(qkv, Be, seq, H, kv, scale)
    check_attention(out, qkv, Be, seq, H, kv, scale, f"query blocks scale {scale}")


def test_attention_production_grid():
    """engine.cu attention in exact variable-length mode at the production grid: H = 16, Be = 8, seq = 1876, cfg3-like
    lengths between 469 and 1875."""
    seq, H = 1876, 16
    kv = [1875, 1603, 1331, 1059, 938, 787, 600, 469]
    Be = len(kv)
    qkv = gen((Be * seq, 3 * H * 64), 230)
    out = run_attention(qkv, Be, seq, H, kv)
    check_attention(out, qkv, Be, seq, H, kv, 0.125, "production grid")


# ------------------------------------------------------------------------------------------------------------------
# Row norm
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("rows", [1, 3, 1001])
@pytest.mark.parametrize("D", list(range(128, 1025, 128)))
def test_row_norm_shapes(D, rows):
    """elementwise.cuh row_norm_kernel: every D the kernel accepts, row counts that are not a multiple of the 4-row
    block, rows with an offset of 100 and a spread of 0.1 (the two-pass variance holds there; E[x^2] - E[x]^2 in fp32
    would not), and in mode 2 an all-zero row gives exact zeros."""
    x = 100.0 + gen((rows, D), 240 + D + rows, 0.1, torch.float32)
    zero = rows // 2 if rows > 1 else None
    if zero is not None:
        x[zero] = 0.0
    a, b = gen((D,), 241, 0.3, torch.float32), gen((D,), 242, 0.3, torch.float32)
    xd, ad, bd = x.double(), a.double(), b.double()
    mean = xd.mean(-1, keepdim=True)
    ln = (xd - mean) / torch.sqrt(((xd - mean) ** 2).mean(-1, keepdim=True) + 1e-6)
    rms = xd / xd.norm(dim=-1, keepdim=True).clamp_min(1e-12) * math.sqrt(D) * ad
    for mode, ref, bb in ((0, ln * (1 + ad) + bd, b), (1, ln * ad + bd, b), (2, rms, None)):
        out = ops.row_norm(x, mode, a, bb)
        check_f16(out, ref, f"row_norm D{D} rows{rows} mode{mode}")
        if mode == 2 and zero is not None:
            assert torch.equal(out[zero], torch.zeros_like(out[zero]))
