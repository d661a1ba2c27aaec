"""The DiT attention kernels and the fused pair epilogues of the fp16 tensor-core GEMM against float64 references.

Kernels under test:
  fa5_kernel (gemm_tc.cu)            tcgen05 flash attention, scores in base 2 (q pre-scaled by log2(e)/8)
  flash_attn_tc_kernel (nn_ops.cu)   mma.sync flash attention, scores in base e (q pre-scaled by 1/8)
  gemm_tc_kernel EPI_SWIGLU / EPI_WNGATE / EPI_ROPE, with the weight interleave of pack_half_interleaved and the table of
  rope_table_kernel
  attention_rope                     SIMT fp32 (strict) and fp16 split + mma.sync (tf32 tail) back ends

Every reference is float64 numpy computed from the exact fp16 values the kernel receives, so what remains is the
kernel's own arithmetic.  The bounds are derived from that arithmetic, not tuned:
  attention   P is rounded to fp16 for P V while l sums the fp32 p:  2^-10 * sum p|v| / sum p, plus T * 2^-25 * max|v| / l
              for p below the fp16 normal range, plus 2^-11 |ref| when the output is fp16;
  epilogues   fp16 output rounding (2^-11 |ref|, doubled for the fast exp / divide) plus 1e-5 * sum |a||w| of fp32
              accumulation, carried through the derivative of the activation;
  RoPE        additionally the table: the device powf may differ from the reference's by an ulp of each frequency
              (numpy and torch already differ by one), i.e. an angle error of t * 2 ulp(freq).
Each case prints its largest error and the largest ratio of error to bound.  (Measured on a B200: the attention and RoPE
ratios stay near 0.5, where fp16 rounding alone would put them; the SwiGLU and gate ratios reach ~1.0 at outputs on the fp16
underflow threshold, which round to zero with an error of exactly the 2^-25 term.)

The CPU tests at the end pin the numpy references to oracle.s2mel._rope and torch's scaled_dot_product_attention.
"""
import math

import numpy as np
import pytest

U10 = 2.0 ** -10
U11 = 2.0 ** -11
HALF_SUB = 2.0 ** -25           # half the smallest fp16 subnormal: rounding error of a tiny value
LOG2E = 1.4426950408889634
HD = 64
FA_TS = [1, 2, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1741, 2622]
PATTERNS = ["peaked", "phantom", "ramp", "first", "alternating"]


# ------------------------------------------------------------------------------------------------ references --
def rope_freqs32():
    """The frequencies of oracle.s2mel._rope, computed the same way (torch fp32)."""
    import torch
    return (1.0 / (10000 ** (torch.arange(0, HD, 2)[: HD // 2].float() / HD))).numpy()


def rope_angles32(T):
    """fp32 angles t * freq as the reference module forms them (torch.outer of fp32 tensors)."""
    return (np.arange(T, dtype=np.float32)[:, None] * rope_freqs32()[None, :]).astype(np.float32)


def rope_angle_err(T):
    """Bound on |device angle - reference angle|: 2 ulp of each fp32 frequency, times t."""
    f = rope_freqs32()
    return np.arange(T, dtype=np.float64)[:, None] * 2 * np.spacing(f).astype(np.float64)[None, :]


def rope_ref(x):
    """x [..., T, 64] float64, interleaved pairs rotated by the fp32 angles (cos / sin evaluated in float64)."""
    T = x.shape[-2]
    ang = rope_angles32(T).astype(np.float64)
    c, s = np.cos(ang), np.sin(ang)
    x0, x1 = x[..., 0::2], x[..., 1::2]
    out = np.empty_like(x)
    out[..., 0::2] = x0 * c - x1 * s
    out[..., 1::2] = x1 * c + x0 * s
    return out


def rope_pair_mag(x):
    """|x0| + |x1| of each pair, repeated on both members: what an angle or table error is multiplied by."""
    m = np.abs(x[..., 0::2]) + np.abs(x[..., 1::2])
    return np.repeat(m, 2, axis=-1)


def attention_ref(q, k, v, base, fp16_out=False, eq=None, ek=None, v_rel=0.0, p16=True):
    """Softmax attention per head in float64: q, k, v [BH][T][64] (scores = q k^T in the kernel's log domain).
    Returns (out, bound).  eq / ek: per-element bounds on the error of q and k before the kernel (composed paths);
    v_rel: relative error of v before the kernel; p16: P is rounded to fp16 for P V (else fp32 throughout, where the
    bound is the 1e-5 of sum p|v| / sum p expected of an fp32 kernel)."""
    BH, T, _ = q.shape
    c = math.log(base)
    out = np.empty((BH, T, HD))
    bnd = np.empty((BH, T, HD))
    for h in range(BH):
        S = q[h] @ k[h].T
        P = np.exp((S - S.max(1, keepdims=True)) * c)
        l = P.sum(1, keepdims=True)
        av = np.abs(v[h])
        o = P @ v[h] / l
        pv = P @ av / l
        b = (U10 * pv + T * HALF_SUB * av.max() / l if p16 else 1e-5 * pv) + v_rel * pv
        if eq is not None:
            dS = eq[h] @ np.abs(k[h]).T + np.abs(q[h]) @ ek[h].T
            D = P * dS * c
            b = b + (D @ av + np.abs(o) * D.sum(1, keepdims=True)) / l
        if fp16_out:
            b = b + U11 * np.abs(o) + HALF_SUB
        out[h], bnd[h] = o, b
    return out, bnd


def heads_to_rows(x, B, H):
    """[B*H][T][64] -> [B][T][H*64] (the attention output layout)."""
    T = x.shape[1]
    return x.reshape(B, H, T, HD).transpose(0, 2, 1, 3).reshape(B, T, H * HD)


def check(name, got, ref, bound):
    err = np.abs(got.astype(np.float64) - ref)
    ratio = (err / bound).max()
    print(f"{name}: max err {err.max():.3e}, max err/bound {ratio:.3f}")
    assert np.all(np.isfinite(got)), name
    assert np.all(err <= bound), (name, float(err.max()), float(ratio), np.unravel_index(np.argmax(err / bound), err.shape))


# ---------------------------------------------------------------------------------------- attention inputs --
def unit_rows(rng, n):
    u = rng.standard_normal((n, HD))
    return u / np.linalg.norm(u, axis=1, keepdims=True)


def along(u, target, a, rng, noise=0.02):
    """Keys whose score against q = a*u is target: (target / a) u plus noise orthogonal to u."""
    n = rng.standard_normal((target.shape[0], HD)) * noise
    n -= (n @ u)[:, None] * u[None, :]
    return (target / a)[:, None] * u[None, :] + n


def make_qkv(pattern, BH, T, seed):
    """fp16 Qr | Kr | Vb [3][BH][T][64] whose scores q.k (the kernel's log domain) follow a pattern:
      peaked       random, score std ~4;
      phantom      every real score ~ -30: a zero-filled key that escapes the mask scores 0 and takes all the mass;
      ramp         scores rise along the keys, so every key tile moves the row max and O is rescaled every time;
      first        the row max lies in keys 0..31 (first tile of both kernels): the rescale is never taken;
      alternating  even rows ramp up, odd rows ramp down: inside one warp some lanes rescale and some do not."""
    rng = np.random.default_rng(seed)
    q = np.empty((BH, T, HD))
    k = np.empty((BH, T, HD))
    v = rng.standard_normal((BH, T, HD)) + 0.5
    a = 4.0
    ramp = 0.02 * (np.arange(T) - T / 2)           # 2.56 per 128-key tile
    for h in range(BH):
        u = unit_rows(rng, 1)[0]
        if pattern == "peaked":
            q[h] = rng.standard_normal((T, HD)) * 0.5
            k[h] = rng.standard_normal((T, HD))
        elif pattern == "phantom":
            c = math.sqrt(30.0)
            q[h] = -c * u[None, :]
            k[h] = c * u[None, :] + rng.standard_normal((T, HD)) * 0.3
        elif pattern == "ramp":
            q[h] = a * u[None, :]
            k[h] = along(u, ramp, a, rng)
        elif pattern == "first":
            tgt = rng.uniform(-8.0, 2.0, T)
            tgt[:32] = rng.uniform(4.0, 6.0, min(T, 32))
            q[h] = a * u[None, :]
            k[h] = along(u, tgt, a, rng)
        elif pattern == "alternating":
            sign = np.where(np.arange(T) % 2 == 0, 1.0, -1.0)
            q[h] = sign[:, None] * a * u[None, :]
            k[h] = along(u, ramp, a, rng)
        else:
            raise ValueError(pattern)
    return np.stack([q, k, v]).astype(np.float16)


# ------------------------------------------------------------------------------------------- flash kernels --
@pytest.mark.gpu
@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("B,H", [(1, 1), (2, 8)])
@pytest.mark.parametrize("T", FA_TS)
def test_flash_attention_kernels(engine, T, B, H, pattern):
    """Both flash kernels on the same fp16 Qr | Kr | Vb: kernel 1 reads the scores in base e, kernel 2 in base 2."""
    qkv = make_qkv(pattern, B * H, T, seed=T * 131 + B * 17 + PATTERNS.index(pattern))
    q, k, v = (x.astype(np.float64) for x in qkv)
    for kernel, base in ((1, math.e), (2, 2.0)):
        ref, bnd = (heads_to_rows(x, B, H) for x in attention_ref(q, k, v, base))
        out, out16 = engine.debug_flash_attention(qkv, B, T, H, kernel)
        tag = f"kernel {kernel} T={T} B={B} H={H} {pattern}"
        check(tag + " fp32", out, ref, bnd)
        check(tag + " fp16", out16, ref, bnd + U11 * np.abs(ref) + HALF_SUB)
        assert np.array_equal(out16.view(np.uint16), out.astype(np.float16).view(np.uint16)), tag
        out_b, out16_b = engine.debug_flash_attention(qkv, B, T, H, kernel)
        assert np.array_equal(out.view(np.uint32), out_b.view(np.uint32)), tag + ": not deterministic"
        assert np.array_equal(out16.view(np.uint16), out16_b.view(np.uint16)), tag + ": not deterministic"
        only16 = engine.debug_flash_attention(qkv, B, T, H, kernel, want_out=False)[1]
        assert np.array_equal(only16.view(np.uint16), out16.view(np.uint16)), tag + ": fp16-only output differs"


# ------------------------------------------------------------------------------------------ pair epilogues --
def gemm_ref(A16, W16, taps, pad, M, bias):
    """sum_tap A[m + tap - pad] W[:, tap]^T (+ bias) in float64 from the fp16 operands, and sum |a||w|."""
    B, Tin, K = A16.shape
    N = W16.shape[0]
    A = A16.astype(np.float64)
    W = W16.astype(np.float64).reshape(N, taps, K)
    x = np.zeros((B, M, N))
    mag = np.zeros((B, M, N))
    for t in range(taps):
        rows = np.arange(M) + t - pad
        ok = (rows >= 0) & (rows < Tin)
        a = np.zeros((B, M, K))
        a[:, ok] = A[:, rows[ok]]
        x += a @ W[:, t].T
        mag += np.abs(a) @ np.abs(W[:, t]).T
    if bias is not None:
        x += bias.astype(np.float64)
    return x, mag


def spread_rows(rng, n, K, lo, hi):
    """n weight rows of K whose outputs on N(0,1) activations have std from lo to hi (pre-activations to ~25 hi)."""
    return rng.standard_normal((n, K)) / math.sqrt(K) * np.geomspace(lo, hi, n)[rng.permutation(n)][:, None]


def sigmoid(x):
    return 0.5 * (1.0 + np.tanh(0.5 * x))


@pytest.mark.gpu
@pytest.mark.parametrize("B,M,K,N", [(2, 1741, 512, 3072)] +                  # DiT FFN w1 | w3: BN 128
                         [(2, m, 96, n) for n in (32, 64, 96, 512) for m in (1, 127, 129)])   # BN 32 / 64
def test_swiglu_epilogue(engine, B, M, K, N):
    rng = np.random.default_rng(M * 7 + N + K)
    h = N // 2
    A = rng.standard_normal((B, M, K)).astype(np.float32)
    w = np.concatenate([spread_rows(rng, h, K, 0.05, 25.0), spread_rows(rng, h, K, 0.5, 2.0)]).astype(np.float32)
    bias = (rng.standard_normal(N) * 0.5).astype(np.float32)
    got = engine.debug_gemm_pair_epilogue(A, w, 1, bias=bias)
    x, mag = gemm_ref(A.astype(np.float16), w.astype(np.float16), 1, 0, M, bias)
    x1, x3, m1, m3 = x[..., :h], x[..., h:], mag[..., :h], mag[..., h:]
    sg = sigmoid(x1)
    silu = x1 * sg
    dsilu = sg * (1 + x1 * (1 - sg))
    ref = silu * x3
    bound = U10 * np.abs(ref) + 1e-5 * (np.abs(dsilu * x3) * m1 + np.abs(silu) * m3) + HALF_SUB
    print(f"max |w1 x| {np.abs(x1).max():.1f}")
    check(f"SwiGLU B={B} M={M} K={K} N={N}", got, ref, bound)


@pytest.mark.gpu
@pytest.mark.parametrize("B,M,K,N,aux_stride", [
    (2, 1741, 512, 1024, 0),          # WaveNet in_layer as the DiT runs it: one g for both CFG halves
    (2, 129, 64, 64, 0),
    (1, 1, 64, 32, 0),
    (2, 129, 64, 64, 80),             # g [B][aux_stride]: a separate gate per batch entry
    (3, 127, 96, 96, 100),
])
def test_wn_gate_epilogue(engine, B, M, K, N, aux_stride):
    rng = np.random.default_rng(M + N + aux_stride)
    taps, h = 5, N // 2
    A = rng.standard_normal((B, M + taps - 1, K)).astype(np.float32)
    w = np.concatenate([spread_rows(rng, h, taps * K, 0.05, 25.0), spread_rows(rng, h, taps * K, 0.05, 25.0)]).astype(np.float32)
    bias = (rng.standard_normal(N) * 0.5).astype(np.float32)
    if aux_stride:
        g = (rng.standard_normal((B, aux_stride)) * 2).astype(np.float32)
        gb = g[:, None, :N].astype(np.float64)
    else:
        g = (rng.standard_normal(N) * 2).astype(np.float32)
        gb = g[None, None, :].astype(np.float64)
    got = engine.debug_gemm_pair_epilogue(A, w, 2, taps=taps, pad=0, M=M, bias=bias, aux=g, aux_stride=aux_stride)
    x, mag = gemm_ref(A.astype(np.float16), w.astype(np.float16), taps, 0, M, bias)
    za, zc = x[..., :h] + gb[..., :h], x[..., h:] + gb[..., h:]
    ta, sc = np.tanh(za), sigmoid(zc)
    ref = ta * sc
    bound = U10 * np.abs(ref) + 1e-5 * ((1 - ta * ta) * sc * mag[..., :h] + np.abs(ta) * sc * (1 - sc) * mag[..., h:]) + HALF_SUB
    print(f"max |pre-activation| {max(np.abs(za).max(), np.abs(zc).max()):.1f}")
    check(f"WN gate B={B} M={M} K={K} N={N} aux_stride={aux_stride}", got, ref, bound)


def rope_epilogue_ref(x, mag, B, T, H, scale):
    """x, mag [B][T][3*H*64] (GEMM result and sum |a||w|) -> reference and bound of Qr | Kr | Vb, each [B*H][T][64]."""
    def heads(y, s):
        return y[..., s * H * HD:(s + 1) * H * HD].reshape(B, T, H, HD).transpose(0, 2, 1, 3).reshape(B * H, T, HD)
    ang_err = np.repeat(rope_angle_err(T), 2, axis=-1)[None]
    refs, bnds = [], []
    for s, sc in ((0, scale), (1, 1.0)):
        xs, ms = heads(x, s), heads(mag, s)
        r = rope_ref(xs) * sc
        pm = rope_pair_mag(xs)
        refs.append(r)
        bnds.append(U10 * np.abs(r) + sc * (1e-5 * rope_pair_mag(ms) + (2.0 ** -22 + ang_err) * pm) + HALF_SUB)
    xv, mv = heads(x, 2), heads(mag, 2)
    refs.append(xv)
    bnds.append(U10 * np.abs(xv) + 1e-5 * mv + HALF_SUB)
    return np.stack(refs), np.stack(bnds)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [0.125, 0.125 * LOG2E], ids=["1/8", "log2e/8"])
@pytest.mark.parametrize("T", [1, 129, 1741])
@pytest.mark.parametrize("H", [1, 8])
def test_rope_epilogue(engine, H, T, scale):
    """q | k | v of the fused wqkv: q rotated and scaled, k rotated, v as is, written head-major Qr | Kr | Vb."""
    rng = np.random.default_rng(T * 3 + H)
    B, K, N = 2, 512, 3 * H * HD
    A = rng.standard_normal((B, T, K)).astype(np.float32)
    w = (rng.standard_normal((N, K)) / math.sqrt(K) * 1.5).astype(np.float32)
    bias = (rng.standard_normal(N) * 0.1).astype(np.float32) if H == 8 else None
    got = engine.debug_gemm_pair_epilogue(A, w, 3, bias=bias, aux_stride=H, scale=scale)
    x, mag = gemm_ref(A.astype(np.float16), w.astype(np.float16), 1, 0, T, bias)
    ref, bnd = rope_epilogue_ref(x, mag, B, T, H, scale)
    for s, name in enumerate(("Qr", "Kr", "Vb")):
        check(f"RoPE {name} H={H} T={T} scale={scale:.4f}", got[s], ref[s], bnd[s])


@pytest.mark.gpu
def test_pair_epilogue_bad_arguments(engine):
    rng = np.random.default_rng(0)
    A = rng.standard_normal((1, 16, 64)).astype(np.float32)
    with pytest.raises(RuntimeError, match="fused-epilogue"):          # N % 32 != 0
        engine.debug_gemm_pair_epilogue(A, rng.standard_normal((48, 64)).astype(np.float32), 1)
    with pytest.raises(RuntimeError, match="gate"):                    # EPI_WNGATE without g
        engine.debug_gemm_pair_epilogue(A, rng.standard_normal((64, 64)).astype(np.float32), 2)
    with pytest.raises(RuntimeError, match="heads"):                   # EPI_ROPE with N != 192 H
        engine.debug_gemm_pair_epilogue(A, rng.standard_normal((192, 64)).astype(np.float32), 3, aux_stride=2)


# ---------------------------------------------------------------------------------- composed production path --
def composed_ref(x, mag, B, T, H, eq_extra=2.0 ** -19, fp16=True):
    """float64 attention with RoPE of the GEMM result x [B][T][3*H*64] (scale 1/8, base e), and the bound of a path that
    rotates q and k in fp32 (table angle error included) and, with fp16, rounds q / 8, k and v to fp16 before a flash
    kernel that rounds P to fp16; without fp16 the fp32 SIMT kernel's bound.  eq_extra: relative error charged to q and
    to k for the fp32 sum of the 64 products of a score (64 * 2^-24 = 2 * 2^-19)."""
    def heads(y, s):
        return y[..., s * H * HD:(s + 1) * H * HD].reshape(B, T, H, HD).transpose(0, 2, 1, 3).reshape(B * H, T, HD)
    ang_err = np.repeat(rope_angle_err(T), 2, axis=-1)[None]
    qs, ks, v = heads(x, 0), heads(x, 1), heads(x, 2)
    q, k = rope_ref(qs) * 0.125, rope_ref(ks)
    eq = 0.125 * (1e-5 * rope_pair_mag(heads(mag, 0)) + (2.0 ** -22 + ang_err) * rope_pair_mag(qs)) + eq_extra * np.abs(q)
    ek = 1e-5 * rope_pair_mag(heads(mag, 1)) + (2.0 ** -22 + ang_err) * rope_pair_mag(ks) + eq_extra * np.abs(k)
    if fp16:
        eq = eq + U11 * np.abs(q) + HALF_SUB
        ek = ek + U11 * np.abs(k) + HALF_SUB
    return attention_ref(q, k, v, math.e, eq=eq, ek=ek, v_rel=U11 if fp16 else 0.0, p16=fp16)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1741, 2622])
def test_rope_epilogue_into_tcgen05_flash(engine, T):
    """The production DiT attention: wqkv GEMM with EPI_ROPE (q scale log2(e)/8) feeding the tcgen05 flash kernel."""
    rng = np.random.default_rng(T)
    B, H, K = 2, 8, 512
    N = 3 * H * HD
    A = rng.standard_normal((B, T, K)).astype(np.float32)
    w = (rng.standard_normal((N, K)) / math.sqrt(K) * 1.5).astype(np.float32)
    qkv16 = engine.debug_gemm_pair_epilogue(A, w, 3, aux_stride=H, scale=0.125 * LOG2E)
    out, _ = engine.debug_flash_attention(qkv16, B, T, H, 2, want_out16=False)
    x, mag = gemm_ref(A.astype(np.float16), w.astype(np.float16), 1, 0, T, None)
    # q also carries log2(e): one more fp32 rounding of q (2^-24), far below the fp16 term
    ref, bnd = composed_ref(x, mag, B, T, H, eq_extra=2.0 ** -19 + 2.0 ** -24)
    check(f"EPI_ROPE -> fa5 B={B} H={H} T={T}", out, heads_to_rows(ref, B, H), heads_to_rows(bnd, B, H))


# ---------------------------------------------------------------------------------------------- attention_rope --
@pytest.mark.gpu
@pytest.mark.parametrize("T", FA_TS)
def test_attention_rope_backends(engine, T):
    """attention_rope from fp32 qkv: the SIMT fp32 kernel (strict path) within ~1e-5 of float64, and the fp16 rotate /
    split + mma.sync flash kernel (tf32 tail) within the bound of its fp16 roundings."""
    rng = np.random.default_rng(T + 99)
    B, H = 2, 8
    qkv = rng.standard_normal((B, T, 3 * H * HD)).astype(np.float32)
    x = qkv.astype(np.float64)
    zero = np.zeros_like(x)                  # no GEMM in front: q, k, v are exact
    ref, b32 = composed_ref(x, zero, B, T, H, fp16=False)
    _, b16 = composed_ref(x, zero, B, T, H)
    ref = heads_to_rows(ref, B, H)
    strict = engine.debug_attention_rope(qkv, H, 1)
    check(f"attention_rope SIMT fp32 T={T}", strict, ref, heads_to_rows(b32, B, H))
    tail = engine.debug_attention_rope(qkv, H, 0)
    check(f"attention_rope fp16 mma.sync T={T}", tail, ref, heads_to_rows(b16, B, H))


# --------------------------------------------------------------------------------- CPU pinning of the references --
@pytest.mark.parametrize("T", [1, 37, 300])
def test_rope_reference_matches_oracle(T):
    import torch
    from oracle.s2mel import _rope
    rng = np.random.default_rng(T)
    x = rng.standard_normal((2, T, 3, HD)).astype(np.float32).astype(np.float64)
    ora = _rope(torch.from_numpy(x), HD).double().numpy()                    # [B, T, H, 64], fp32 arithmetic
    mine = rope_ref(x.transpose(0, 2, 1, 3)).transpose(0, 2, 1, 3)          # float64 arithmetic, same fp32 angles
    # the oracle rotates in fp32: two products and a sum, each rounded
    assert np.all(np.abs(ora - mine) <= 2.0 ** -22 * rope_pair_mag(x) + 1e-30)
    assert not np.array_equal(ora, mine) or T == 1


@pytest.mark.parametrize("T", [1, 65, 200])
def test_attention_reference_matches_sdpa(T):
    import torch
    import torch.nn.functional as F
    from oracle.s2mel import _rope
    rng = np.random.default_rng(T + 1)
    B, H = 2, 3
    qs, ks, v = (rng.standard_normal((B, T, H, HD)) for _ in range(3))
    # the DiT's attention as the oracle states it (oracle/s2mel.py dit_forward): RoPE, then SDPA (scale 1/8)
    tq = _rope(torch.from_numpy(qs), HD).double().transpose(1, 2)
    tk = _rope(torch.from_numpy(ks), HD).double().transpose(1, 2)
    tv = torch.from_numpy(v).transpose(1, 2)
    sdpa = F.scaled_dot_product_attention(tq, tk, tv).transpose(1, 2).reshape(B, T, H * HD).numpy()
    # the same from the numpy references, fed the oracle's rotated q and k
    q = tq.reshape(B * H, T, HD).numpy() * 0.125
    k = tk.reshape(B * H, T, HD).numpy()
    mine, _ = attention_ref(q, k, tv.reshape(B * H, T, HD).numpy(), math.e)
    assert np.abs(heads_to_rows(mine, B, H) - sdpa).max() <= 1e-12
    # and both bases describe one softmax: scores in base 2 scaled by log2(e) give the same attention
    mine2, _ = attention_ref(q * LOG2E, k, tv.reshape(B * H, T, HD).numpy(), 2.0)
    assert np.abs(mine2 - mine).max() <= 1e-12
    # the full composition (numpy RoPE with fp32 angles) stays within the oracle's fp32 rotation error
    qkv = np.concatenate([y.reshape(B, T, H * HD) for y in (qs, ks, v)], axis=-1)     # q | k | v, as wqkv writes it
    full, _ = composed_ref(qkv, np.zeros_like(qkv), B, T, H)
    assert np.abs(heads_to_rows(full, B, H) - sdpa).max() <= 1e-5


@pytest.mark.parametrize("T", [65, 257, 1741])
def test_attention_patterns_do_what_they_claim(T):
    """The score patterns of the flash tests, after fp16 rounding, still exercise the code paths they are built for."""
    for pattern in PATTERNS:
        q, k, v = (x.astype(np.float64) for x in make_qkv(pattern, 2, T, seed=T))
        S = np.einsum("htd,hsd->hts", q, k)
        if pattern == "phantom":
            assert S.max() < -15 and S.min() > -50
        elif pattern == "peaked":
            assert 3 < S.std() < 5
        elif pattern == "first":
            assert np.all(S.argmax(2) < 32)
        else:
            tiles = [S[..., j:j + 64].max(2) for j in range(0, T, 64)]
            rows = slice(None) if pattern == "ramp" else slice(0, None, 2)
            for a, b in zip(tiles, tiles[1:]):                   # the row max rises at every tile of 64 keys
                assert np.all(b[:, rows] > a[:, rows])
            if pattern == "alternating":
                for a, b in zip(tiles, tiles[1:]):               # ... and never for the odd rows
                    assert np.all(b[:, 1::2] < a[:, 1::2])
