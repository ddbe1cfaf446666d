"""Codec-decoder kernels against float64 references, one launch at a time (q3tts_codec_*_probe).

The whole-decode tests (test_gpu_codec.py, test_gpu_fullsize.py) hold these kernels to a PCM SNR of 40 dB over ~100 launches; a
kernel wrong on a few rows (the last partial tile, the first rows of batch item 1, one strip boundary) passes that.  Here each
launch is compared element by element with a float64 restatement of the same operation that applies exactly the roundings the
kernel applies at its operand boundaries (fp16 operands, fp16 stores), so each bar sits near fp32 accumulation error:

  * fused residual unit (codec_unit_kernel) and its two-GEMM form, both against the SAME reference:
        v1 = conv7_dil(a16; w7_16) + b7            h = fp16(snake2(v1))
        x' = res16 + (h @ w1_16^T + b1)             outr = fp16(x'),  out = fp16(snake3(x'))   (snake3 of the UNROUNDED x')
    A kernel value with error e (bar below) may round to any fp16 value in [fp16(ref - e), fp16(ref + e)]; that interval is the
    assertion.  The intermediate h is where a rounding flip matters downstream: for every h element whose bar interval straddles
    an fp16 rounding boundary, |the other fp16 neighbour - h| * |w1| is added to the bar of x'.  Bars:
        fp32 accumulation  ACC_U * 2^-24 * sum|terms|  (+ one rounding of each add that follows),
        SnakeBeta          (1 + ieb * ea) * e_in + 2 * ieb * |sin| * (SIN_ABS + SIN_REL * |v * ea|)  (__sinf: absolute error
                           2^-21.4 on [-pi, pi], growing with the argument: its range reduction is one fp32 multiply).
  * attention: codec_attention_mma_kernel rounds q, k (after RoPE), v and P to fp16 and sums l over the unrounded p.  With w_j the
    exact softmax weights, rounding P costs at most 2^-11 * sum_j w_j |v_j| (p >= 2^-14) plus 2^-25 per key (fp16 subnormals)
    times max|V|; the reference uses the fp16-rounded q, k, v.  The SIMT kernels take fp32 operands: ATT_SIMT_REL * max|V|.  Both
    add 2 * (score error) * max|V| for the fp32 dot products (8 * 2^-24 * scale * sum|q k| per key) and the fp16 output interval.
  * RoPE: angle = fp32(t) * inv_freq (fp32 product), t = row % T; rotated values within ROPE_ULPS fp32 ulp of |a| + |b|; v heads
    bit-identical.
  * output conv: causal 7-tap dot product per batch item, clip(-1, 1), NaN -> 0; +-Inf inputs clip to +-1, NaN inputs give 0.
  * row ops (dwconv7, LayerNorm, RMSNorm, SnakeBeta, SiLU * up): a few fp32 roundings of their magnitudes.

The references are anchored on oracle/codec.py by the CPU tests at the top, so a wrong reference cannot agree with a wrong kernel.
"""
import types
import zlib

import numpy as np
import pytest

U = 2.0 ** -24  # fp32 unit roundoff
# Measured on a B200 (1000 W), all cases of this file; _report prints these ratios (worst error / bar) after a `-m gpu -s` run.
ACC_U = 32          # fp32 accumulation of the unit's two contractions; with the SnakeBeta terms below the worst x' uses 0.87 of its
SIN_ABS = 2.0 ** -20  # bar and the worst snake3(x') 0.75, in both forms (the large-argument cases included)
SIN_REL = 2.0 ** -21
ATT_SIMT_REL = 1e-6  # SIMT attention: worst 0.04 of the bar (at 2e-6); the mma.sync kernel uses 0.27 of its fp16-P bar
ROPE_ULPS = 4       # worst 2.45 fp32 ulp of |a| + |b|
OUT_ACC_U = 16      # output conv, worst: streaming kernel 0.9, SIMT fp32 / fp16 input 7.1 / 5.5, tcgen05 pcm epilogue 5.9 (x 2^-24 sum|terms|)
ROW_U = 16          # row ops, worst: dwconv7 4.3, LayerNorm 2.2, SnakeBeta 4.6 (x 2^-24 of their magnitudes)
STATS = {}


def _stat(key, ratio):
    STATS[key] = max(STATS.get(key, 0.0), float(ratio))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k, v in sorted(STATS.items()):
        print(f"[codec kernel probe] {k}: worst error uses {v:.3f} of its bar")


def _r16(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float64)


def _interval16(ref, e):
    """fp16 values a kernel whose pre-rounding value lies in [ref - e, ref + e] can store."""
    return (ref - e).astype(np.float16).astype(np.float64), (ref + e).astype(np.float16).astype(np.float64)


def _check_interval(got, ref, e, label, key):
    lo, hi = _interval16(ref, e)
    got = np.asarray(got, np.float64)
    ok = (got >= lo) & (got <= hi)
    if not ok.all():
        i = tuple(np.argwhere(~ok)[0])
        raise AssertionError(f"{label}: {int((~ok).sum())} of {ok.size} values off; first at {i}: got {got[i]:.7g}, want {ref[i]:.7g} "
                             f"(+- {e[i]:.3g})")
    err = np.abs(got - ref)
    _stat(key, (np.maximum(err - np.spacing(np.abs(ref).astype(np.float16)).astype(np.float64), 0) / np.maximum(e, 1e-30)).max())


def _check_abs(got, ref, e, label, key):
    got = np.asarray(got, np.float64)
    err = np.abs(got - ref)
    ok = err <= e  # NaN fails
    if not ok.all():
        i = tuple(np.argwhere(~ok)[0])
        raise AssertionError(f"{label}: {int((~ok).sum())} of {ok.size} values off; first at {i}: got {got[i]:.7g}, want {ref[i]:.7g} "
                             f"(bar {e[i]:.3g})")
    _stat(key, (err / np.maximum(e, 1e-300)).max())


# ------------------------------------------------------------------------------------------------ float64 references
def ref_snake(v, ea, ieb):
    s = np.sin(v * ea)
    return v + ieb * s * s, s


def snake_bar(v, s, ea, ieb, e_in):
    """error of the kernels' fp32 SnakeBeta (__sinf) of an input known to e_in"""
    arg = np.abs(v * ea)
    return (1 + ieb * ea) * e_in + 2 * ieb * np.abs(s) * (SIN_ABS + SIN_REL * arg) + 2 * U * (np.abs(v) + ieb * s * s)


def causal_taps(x, w, dil):
    """x [B, T, Cin], w [K, N, Cin] (tap k reads row t - (K-1-k)*dil of the same item) -> (sum, sum of |terms|), float64"""
    B, T, _ = x.shape
    K = w.shape[0]
    y = np.zeros((B, T, w.shape[1]))
    s = np.zeros_like(y)
    for k in range(K):
        sh = (K - 1 - k) * dil
        if sh >= T:
            continue
        xs = np.zeros_like(x)
        xs[:, sh:] = x[:, :T - sh]
        y += xs @ w[k].T
        s += np.abs(xs) @ np.abs(w[k]).T
    return y, s


def ref_unit(a, w7, b7, ea2, ieb2, w1, b1, res, ea3, ieb3, dil, round16=True):
    """The residual unit on the operands as the kernel holds them (a, w7, w1, res already fp16 values when round16).
    -> (x', snake3(x'), bar of x', bar of snake3(x') before the fp16 store), float64."""
    acc1, s1 = causal_taps(a, w7, dil)
    v1 = acc1 + (0.0 if b7 is None else b7)
    e_v1 = ACC_U * U * s1 + U * np.abs(v1)
    pre, s2 = ref_snake(v1, ea2, ieb2)
    if round16:
        e_pre = snake_bar(v1, s2, ea2, ieb2, e_v1)
        h = _r16(pre)
        lo, hi = _interval16(pre, e_pre)
        flip = np.maximum(np.abs(lo - h), np.abs(hi - h))  # the other fp16 neighbour, where the bar straddles a rounding boundary
    else:
        h, flip = pre, np.zeros_like(pre)
    acc2 = h @ w1.T
    s_acc2 = np.abs(h) @ np.abs(w1).T
    y = acc2 + (0.0 if b1 is None else b1)
    x = res + y
    e_x = ACC_U * U * s_acc2 + U * (np.abs(y) + np.abs(x)) + flip @ np.abs(w1).T
    out, s3 = ref_snake(x, ea3, ieb3)
    return x, out, e_x, snake_bar(x, s3, ea3, ieb3, e_x)


def ref_out_conv(x, w, bias):
    """x [B, T, C], w [7, C], bias scalar -> clip(bias + causal 7-tap dot, -1, 1) with NaN -> 0; and sum of |terms| + |bias|"""
    with np.errstate(invalid="ignore"):
        y, s = causal_taps(x, w[:, None, :], 1)
        y = y[..., 0] + bias
    s = s[..., 0] + abs(bias)
    y = np.where(np.isnan(y), 0.0, np.clip(y, -1.0, 1.0))
    return y, s


def ref_attention(qkv, nh, nkv, causal=True, f16=False):
    """qkv [B, T, (nh + 2 nkv) 64] -> out [B, T, nh*64], max|V| over visible keys, sum_j w_j |v_j|, max score error, float64"""
    x = np.asarray(qkv, np.float64)
    if f16:
        x = _r16(qkv)
    B, T, _ = x.shape
    G = nh // nkv
    scale = np.float64(np.float32(1.0) / np.sqrt(np.float32(64.0)))
    out = np.zeros((B, T, nh, 64))
    vmax = np.zeros((B, T, nh))
    wv = np.zeros((B, T, nh))
    ds = np.zeros((B, T, nh))
    mask = np.tril(np.ones((T, T), bool)) if causal else np.ones((T, T), bool)
    for b in range(B):
        for h in range(nh):
            kvh = h // G
            q = x[b, :, h * 64:(h + 1) * 64]
            k = x[b, :, (nh + kvh) * 64:(nh + kvh + 1) * 64]
            v = x[b, :, (nh + nkv + kvh) * 64:(nh + nkv + kvh + 1) * 64]
            sc = np.where(mask, q @ k.T * scale, -np.inf)
            p = np.exp(sc - sc.max(-1, keepdims=True))
            wgt = p / p.sum(-1, keepdims=True)
            out[b, :, h] = wgt @ v
            av = np.abs(v).max(-1)
            vmax[b, :, h] = np.where(mask, av[None, :], 0).max(-1)
            wv[b, :, h] = wgt @ av
            ds[b, :, h] = np.where(mask, 8 * U * scale * (np.abs(q) @ np.abs(k).T), 0).max(-1)
    return out.reshape(B, T, nh * 64), vmax, wv, ds


def ref_rope(qkv, nh, nkv, inv_freq):
    """-> roped qkv (q and k heads; v untouched), |a| + |b| per rotated element; positions restart per batch item"""
    x = np.asarray(qkv, np.float64).copy()
    B, T, _ = x.shape
    ang = (np.arange(T, dtype=np.float32)[:, None] * np.asarray(inv_freq, np.float32)[None, :]).astype(np.float64)  # fp32 products
    c, s = np.cos(ang)[None], np.sin(ang)[None]
    mag = np.zeros_like(x)
    for h in range(nh + nkv):
        a, bb = x[..., h * 64:h * 64 + 32].copy(), x[..., h * 64 + 32:(h + 1) * 64].copy()
        x[..., h * 64:h * 64 + 32] = a * c - bb * s
        x[..., h * 64 + 32:(h + 1) * 64] = bb * c + a * s
        mag[..., h * 64:(h + 1) * 64] = np.concatenate([np.abs(a) + np.abs(bb)] * 2, -1)
    return x, mag


def _inv_freq(theta=10000.0):
    return (np.float32(1.0) / np.power(np.float32(theta), np.arange(0, 64, 2, dtype=np.float32) / np.float32(64.0))).astype(np.float32)


# ------------------------------------------------------------------------------------------------ CPU: references vs the oracle
def test_unit_and_snake_references_match_the_oracle():
    """snake_beta, causal_conv1d (dilated) and decode()'s residual unit of oracle/codec.py against ref_snake / causal_taps / ref_unit
    (without the fp16 roundings), and the output conv (causal_conv1d + clamp) against ref_out_conv."""
    import torch

    from oracle import codec as oc

    rng = np.random.default_rng(0)
    B, T, C = 2, 70, 24
    t64 = lambda a: torch.from_numpy(np.asarray(a, np.float64))
    alpha = rng.uniform(-1, 1.5, (3, C))
    beta = rng.uniform(-1, 1, (3, C))
    ea, ieb = np.exp(alpha), 1.0 / (np.exp(beta) + 1e-9)
    x = rng.standard_normal((B, T, C))
    got, _ = ref_snake(x, ea[0], ieb[0])
    want = oc.snake_beta(t64(x).transpose(1, 2), t64(alpha[0]), t64(beta[0])).transpose(1, 2).numpy()
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    for dil in (1, 3, 9):
        wo = rng.standard_normal((C, C, 7)) / np.sqrt(7 * C)  # disk layout [C_out, C_in, K]
        bo = rng.standard_normal(C)
        w7 = wo.transpose(2, 0, 1)  # [tap][out][in]
        got, _ = causal_taps(x, w7, dil)
        want = oc.causal_conv1d(t64(x).transpose(1, 2), t64(wo), t64(bo), dilation=dil).transpose(1, 2).numpy()
        np.testing.assert_allclose(got + bo, want, rtol=1e-12, atol=1e-12)
        # decode()'s residual unit: h + conv2(snake2(conv1(snake1(h))))
        w1o = rng.standard_normal((C, C, 1)) / np.sqrt(C)
        b1 = rng.standard_normal(C)
        r = t64(x).transpose(1, 2)
        u = oc.snake_beta(r, t64(alpha[1]), t64(beta[1]))
        u = oc.causal_conv1d(u, t64(wo), t64(bo), dilation=dil)
        u = oc.snake_beta(u, t64(alpha[2]), t64(beta[2]))
        u = oc.causal_conv1d(u, t64(w1o), t64(b1))
        want = (u + r).transpose(1, 2).numpy()
        a = ref_snake(x, ea[1], ieb[1])[0]
        xp, out, _, _ = ref_unit(a, w7, bo, ea[2], ieb[2], w1o[:, :, 0], b1, x, ea[0], ieb[0], dil, round16=False)
        np.testing.assert_allclose(xp, want, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(out, ref_snake(want, ea[0], ieb[0])[0], rtol=1e-12, atol=1e-12)
    # output conv: C -> 1, k = 7, then the clamp of decode()
    wo = rng.standard_normal((1, C, 7)) * 0.3
    bo = rng.standard_normal(1)
    xs = x * 2
    want = oc.causal_conv1d(t64(xs).transpose(1, 2), t64(wo), t64(bo)).clamp(-1.0, 1.0)[:, 0].numpy()
    got, _ = ref_out_conv(xs, wo[0].T, float(bo[0]))
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    assert (np.abs(want) == 1.0).any() and (np.abs(want) < 1.0).any()


def test_attention_and_rope_references_match_the_oracle():
    """One pre_transformer layer of oracle/codec.py, weighted so that its output exposes the attention: RMSNorm weights 1 and eps 0
    on rows of RMS exactly 1 (the norm is the identity), q / k / v projections that select columns of the row, an o_proj that writes
    the attention into channels the input leaves zero, no MLP, identity output projection.  The final RMSNorm's factor is undone
    from the pass-through channels.  GQA (nh = 2 nkv) and a causal window of 37 rows."""
    import torch

    from oracle import codec as oc

    rng = np.random.default_rng(1)
    nh, nkv, hd, T = 4, 2, 64, 37
    W = (nh + 2 * nkv) * hd
    D = W + nh * hd
    cfg = types.SimpleNamespace(head_dim=hd, rope_theta=10000.0, num_attention_heads=nh, num_key_value_heads=nkv, num_hidden_layers=1,
                                rms_norm_eps=0.0)
    o = oc.CodecDecoder.__new__(oc.CodecDecoder)
    o.c = cfg
    eye = np.eye(D)
    p = "decoder.pre_transformer"
    lp = p + ".layers.0"
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64))
    o.w = {p + ".input_proj.weight": t(eye), p + ".input_proj.bias": t(np.zeros(D)),
           lp + ".input_layernorm.weight": t(np.ones(D)), lp + ".post_attention_layernorm.weight": t(np.ones(D)),
           lp + ".self_attn.q_proj.weight": t(eye[:nh * hd]), lp + ".self_attn.k_proj.weight": t(eye[nh * hd:(nh + nkv) * hd]),
           lp + ".self_attn.v_proj.weight": t(eye[(nh + nkv) * hd:W]), lp + ".self_attn.o_proj.weight": t(eye[:, W:]),
           lp + ".self_attn_layer_scale.scale": t(np.ones(D)), lp + ".mlp_layer_scale.scale": t(np.zeros(D)),
           lp + ".mlp.gate_proj.weight": t(np.zeros((8, D))), lp + ".mlp.up_proj.weight": t(np.zeros((8, D))),
           lp + ".mlp.down_proj.weight": t(np.zeros((D, 8))), p + ".norm.weight": t(np.ones(D)), p + ".output_proj.weight": t(eye),
           p + ".output_proj.bias": t(np.zeros(D))}
    qkv = rng.standard_normal((1, T, W))
    x = np.concatenate([qkv, np.zeros((1, T, nh * hd))], -1)
    x /= np.sqrt(np.mean(x * x, -1, keepdims=True))
    y = o.pre_transformer(t(x)).numpy()
    rho = x[..., :1] / y[..., :1]  # the final RMSNorm's 1 / factor, from a pass-through channel
    want = y[..., W:] * rho
    inv = (1.0 / torch.pow(torch.tensor(10000.0, dtype=torch.float32), torch.arange(0, hd, 2, dtype=torch.float32) / hd)).numpy()
    roped, _ = ref_rope(x[..., :W], nh, nkv, inv)
    got, _, _, _ = ref_attention(roped, nh, nkv)
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-6)  # the oracle takes cos / sin in fp32
    np.testing.assert_allclose(y[..., :W] * rho, x[..., :W], rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------------ CPU: refusals without a device
def _status(fn):
    import qwen3tts_b200 as q

    with pytest.raises(q.Q3Error) as e:
        fn()
    return e.value.status


def test_probes_reject_out_of_range_arguments_before_any_launch():
    """Shapes the fused unit refuses (C % 32, C > 192, a halo beyond 192 rows, fewer than 32 row tiles), bad forms, flags, kernels,
    strips and row-op layouts return Q3TTS_ERR_INVALID_ARG from the host-side validation (no device needed)."""
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi as A

    rng = np.random.default_rng(2)

    def unit(form=1, B=1, T=4096, C=32, dil=1, **kw):
        z = lambda *s: rng.standard_normal(s).astype(np.float32)
        return q.codec_unit_probe(form, z(B, T, C), z(7, C, C), None, z(C), z(C), z(C, C), None, z(B, T, C), z(C), z(C), dil, **kw)

    def att(kernel=0, B=1, T=16, nh=2, nkv=2):
        return q.codec_attention_probe(kernel, np.zeros((B, T, (nh + 2 * nkv) * 64), np.float32), nh, nkv)

    def oc(kernel=0, B=1, T=64, C=32, strip=0):
        return q.codec_out_conv_probe(kernel, np.zeros((B, T, C), np.float32), np.zeros((7, C), np.float32), 0.0, strip=strip)

    def row(op, rows=4, ldx=16, C=16, T=0, w=True, b=True):
        return q.codec_rowop_probe(op, np.zeros((rows, ldx), np.float32), C, w=np.ones(7 * C, np.float32) if w else None,
                                   b=np.ones(C, np.float32) if b else None, T=T)

    bad = {
        "unit: C not a multiple of 32": lambda: unit(C=48),
        "unit: C above 192 (fused)": lambda: unit(C=224),
        "unit: C above 1536 (two GEMMs)": lambda: unit(form=0, C=1568, T=8),
        "unit: halo of 128 + 6 * 11 rows": lambda: unit(dil=11),
        "unit: 31 row tiles": lambda: unit(T=31 * 128),
        "unit: 2 items x 15 tiles": lambda: unit(B=2, T=15 * 128),
        "unit: dilation 0": lambda: unit(form=0, dil=0),
        "unit: form 2": lambda: unit(form=2),
        "unit: in place without the residual": lambda: unit(in_place=True, emit_residual=False),
        "unit: 0 weight copies": lambda: unit(weight_reps=0),
        "unit: 33 weight copies": lambda: unit(weight_reps=33),
        "attention: kernel 4": lambda: att(kernel=4),
        "attention: T 2401": lambda: att(T=2401),
        "attention: nh % nkv": lambda: att(nh=3, nkv=2),
        "attention: 65 items": lambda: att(B=65, T=1),
        "out conv: kernel 4": lambda: oc(kernel=4),
        "out conv: streaming C 160": lambda: oc(C=160),
        "out conv: strip 48": lambda: oc(strip=48),
        "out conv: strip 16": lambda: oc(strip=16),
        "out conv: strip on the SIMT kernel": lambda: oc(kernel=1, strip=64),
        "out conv: SIMT C 288": lambda: oc(kernel=2, C=288),
        "out conv: GEMM C 100": lambda: oc(kernel=3, C=100),
        "row op: unknown": lambda: q.lib().q3tts_codec_rowop_probe(0, 6, np.zeros(4, np.float32).ctypes.data_as(A.p_f32), 1, 4, 4, 0, None, None,
                                                                    0.0, np.zeros(4, np.float32).ctypes.data_as(A.p_f32)),
        "row op: dwconv7 rows % T": lambda: row("dwconv7", rows=5, T=2),
        "row op: layernorm ldx != C": lambda: row("layernorm", ldx=24),
        "row op: rmsnorm ldx < C": lambda: row("rmsnorm_f16", ldx=8, w=False),
        "row op: silu_mul ldx != 2C": lambda: row("silu_mul", ldx=16),
        "row op: snake without ieb": lambda: row("snake", b=False),
    }
    for what, fn in bad.items():
        if what == "row op: unknown":
            st = fn()
            assert st == A.ERR_INVALID_ARG, f"{what}: status {st}"
            continue
        st = _status(fn)
        assert st == A.ERR_INVALID_ARG, f"{what}: status {st}"


# ------------------------------------------------------------------------------------------------ GPU: fused residual unit
def _unit_inputs(rng, B, T, C, arg_scale=1.0, item_scale=None):
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    a = f(B, T, C) * 0.7
    res = f(B, T, C)
    if item_scale is not None:  # items of very different magnitude: a halo read across the batch boundary stands out
        a *= np.asarray(item_scale, np.float32)[:, None, None]
        res *= np.asarray(item_scale, np.float32)[:, None, None]
    w7 = f(7, C, C) / np.float32(np.sqrt(7 * C))
    w1 = f(C, C) / np.float32(np.sqrt(C))
    b7, b1 = f(C) * 0.1, f(C) * 0.1
    lo, hi = (-1.0, 1.5) if arg_scale == 1.0 else (np.log(arg_scale), np.log(3 * arg_scale))
    ea2, ea3 = [np.exp(rng.uniform(lo, hi, C)).astype(np.float32) for _ in range(2)]
    ieb2, ieb3 = [(1.0 / (np.exp(rng.uniform(-1, 1, C)) + 1e-9)).astype(np.float32) for _ in range(2)]
    return a, w7, b7, ea2, ieb2, w1, b1, res, ea3, ieb3


def _run_unit(form, inp, dil, label, in_place=False, emit=True, reps=1, biases=True, ref=None):
    import qwen3tts_b200 as q

    a, w7, b7, ea2, ieb2, w1, b1, res, ea3, ieb3 = inp
    if not biases:
        b7 = b1 = None
    x_out, out = q.codec_unit_probe(form, a, w7, b7, ea2, ieb2, w1, b1, res, ea3, ieb3, dil, in_place=in_place, emit_residual=emit,
                                    weight_reps=reps)
    if ref is None:
        d = lambda v: None if v is None else np.asarray(v, np.float64)
        ref = ref_unit(_r16(a), _r16(w7), d(b7), d(ea2), d(ieb2), _r16(w1), d(b1), _r16(res), d(ea3), d(ieb3), dil)
    x, o, e_x, e_o = ref
    key = "unit fused" if form == 1 else "unit two GEMMs"
    if emit:
        _check_interval(x_out, x, e_x, f"{label}: x'", key + " x'")
    else:
        assert x_out is None
    _check_interval(out, o, e_o, f"{label}: snake3(x')", key + " snake3(x')")
    return ref


UNIT_C = [32, 64, 96, 128, 160, 192]


@pytest.mark.gpu
@pytest.mark.parametrize("dil", [1, 3, 9])
@pytest.mark.parametrize("C", UNIT_C)
def test_unit_single_item_tile_edges(C, dil):
    """B = 1, T = 128 k + {0, 1, 127} (32, 34 and 37 tiles): both forms against one reference; production's 8 weight copies, in-place
    x', a separate x' buffer, no x' (the third unit of a block) and NULL biases."""
    rng = np.random.default_rng(zlib.crc32(repr(("single", C, dil)).encode()))
    for T, kw in ((128 * 32, dict(in_place=True, reps=8)), (128 * 33 + 1, dict(reps=1, biases=False)), (128 * 36 + 127, dict(emit=False, reps=8))):
        inp = _unit_inputs(rng, 1, T, C)
        ref = _run_unit(1, inp, dil, f"fused C {C} dil {dil} T {T}", **kw)
        _run_unit(0, inp, dil, f"two GEMMs C {C} dil {dil} T {T}", ref=ref, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("C", UNIT_C)
def test_unit_batch_boundary(C):
    """Three items of 1500 rows (12 tiles each, the last one 92 rows) whose magnitudes differ 160-fold, dilation 9 (a 54-row halo):
    the first rows of items 1 and 2 must read zeros, not the previous item's tail."""
    rng = np.random.default_rng(zlib.crc32(repr(("batch", C)).encode()))
    inp = _unit_inputs(rng, 3, 1500, C, item_scale=[8.0, 0.05, 1.0])
    ref = _run_unit(1, inp, 9, f"fused C {C} batch", reps=8)
    _run_unit(0, inp, 9, f"two GEMMs C {C} batch", reps=8, ref=ref)
    inp = _unit_inputs(rng, 2, 128 * 16 + 3, C, item_scale=[0.05, 8.0])
    ref = _run_unit(1, inp, 3, f"fused C {C} batch dil 3", in_place=True)
    _run_unit(0, inp, 3, f"two GEMMs C {C} batch dil 3", in_place=True, ref=ref)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,C,dil", [(1, 49920, 96, 9), (4, 5000, 192, 3), (2, 20000, 96, 1), (1, 160 * 128, 128, 3)])
def test_unit_persistent_tile_walk(B, T, C, dil):
    """More than 148 tiles (160, 157) and more than 2 x 148 (390: the real block-4 pass of 49 920 rows; 2 x 157): every CTA walks
    several tiles, crossing item boundaries mid-walk, with 8 weight copies (CTA i reads copy i % 8)."""
    rng = np.random.default_rng(zlib.crc32(repr(("walk", B, T, C, dil)).encode()))
    inp = _unit_inputs(rng, B, T, C, item_scale=[1.0 + 2.0 * (i % 2) for i in range(B)])
    ref = _run_unit(1, inp, dil, f"fused {B}x{T} C {C}", in_place=True, reps=8)
    _run_unit(0, inp, dil, f"two GEMMs {B}x{T} C {C}", in_place=True, reps=8, ref=ref)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [64, 192])
def test_unit_large_snake_arguments(C):
    """SnakeBeta with e^alpha of 20-60 on both activations: |v e^alpha| reaches several hundred, where __sinf's error is largest, and
    snake3's slope (1 + ieb e^alpha ~ 100) magnifies any rounding of x' before it (snake3 must see the fp32 x')."""
    rng = np.random.default_rng(zlib.crc32(repr(("args", C)).encode()))
    inp = _unit_inputs(rng, 1, 128 * 32 + 5, C, arg_scale=20.0)
    x = np.asarray(inp[7], np.float64)
    assert np.abs(x * inp[8]).max() > 200
    ref = _run_unit(1, inp, 3, f"fused C {C} large args", reps=8)
    _run_unit(0, inp, 3, f"two GEMMs C {C} large args", reps=8, ref=ref)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(1, 1), (1, 127), (2, 130), (3, 700)])
def test_unit_two_gemm_form_on_short_passes(B, T):
    """The shapes the decoder runs as two GEMM launches because the fused kernel refuses them (fewer than 32 row tiles)."""
    rng = np.random.default_rng(zlib.crc32(repr(("short", B, T)).encode()))
    for C, dil in ((32, 9), (96, 3), (256, 1)):
        inp = _unit_inputs(rng, B, T, C)
        _run_unit(0, inp, dil, f"two GEMMs {B}x{T} C {C}", in_place=True, reps=8)


# ------------------------------------------------------------------------------------------------ GPU: attention and RoPE
ATT_T = [1, 15, 16, 17, 63, 64, 65, 128, 750, 2400]


def _check_attention(kernel, qkv_roped, out, nh, nkv, label):
    mma, f16_out = kernel == 0, kernel in (0, 3)
    ref, vmax, wv, ds = ref_attention(qkv_roped, nh, nkv, causal=kernel != 2, f16=mma)
    B, T, _ = qkv_roped.shape
    rows_vis = np.broadcast_to((np.arange(T) + 1 if kernel != 2 else np.full(T, T))[None, :, None], vmax.shape)
    if mma:
        e = 2.0 ** -11 * wv + rows_vis * 2.0 ** -25 * vmax + 2 * ds * vmax + ATT_SIMT_REL * vmax
    else:
        e = ATT_SIMT_REL * vmax + 2 * ds * vmax
    e = np.repeat(e, 64, axis=-1)
    key = f"attention kernel {kernel}"
    if f16_out:
        _check_interval(out, ref, e, label, key)
    else:
        _check_abs(out, ref, e, label, key)


@pytest.mark.gpu
@pytest.mark.parametrize("nh,nkv", [(4, 4), (4, 2)], ids=["mha", "gqa"])
@pytest.mark.parametrize("kernel", [0, 1, 2, 3])
def test_attention_with_rope(kernel, nh, nkv):
    """Every T of ATT_T with B = 1 and 3, RoPE first (positions restart per item): the roped q / k against ref_rope, v and the
    untouched columns bit-identical; then the attention against ref_attention over the roped rows the kernel read."""
    import qwen3tts_b200 as q

    f = _inv_freq()
    for B in (1, 3):
        for T in ATT_T:
            rng = np.random.default_rng(zlib.crc32(repr((kernel, nh, nkv, B, T)).encode()))
            qkv = rng.standard_normal((B, T, (nh + 2 * nkv) * 64)).astype(np.float32)
            out, roped = q.codec_attention_probe(kernel, qkv, nh, nkv, f)
            want, mag = ref_rope(qkv, nh, nkv, f)
            rot = (nh + nkv) * 64
            assert np.array_equal(roped[..., rot:].view(np.uint32), qkv[..., rot:].view(np.uint32)), f"B {B} T {T}: v changed"
            _check_abs(roped[..., :rot], want[..., :rot], ROPE_ULPS * U * mag[..., :rot] + 1e-30, f"rope B {B} T {T}", "rope")
            _check_attention(kernel, roped, out, nh, nkv, f"kernel {kernel} nh {nh} nkv {nkv} B {B} T {T}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dominant_first", "dominant_last", "dominant_mid", "equal_keys", "large_scores"])
@pytest.mark.parametrize("kernel", [0, 1, 2, 3])
def test_attention_softmax_extremes(kernel, kind):
    """One key ahead of the others by a score gap of ~60 (key 0, the row's own key, a key of the second 64-key tile), all keys equal,
    and scores of +-40 everywhere; B = 2, GQA, no RoPE."""
    import qwen3tts_b200 as q

    nh, nkv = 4, 2
    for T in (17, 65, 200):
        rng = np.random.default_rng(zlib.crc32(repr((kernel, kind, T)).encode()))
        x = rng.standard_normal((2, T, (nh + 2 * nkv) * 64)).astype(np.float32)
        qh = x[..., :nh * 64].reshape(2, T, nh, 64)
        kh = x[..., nh * 64:(nh + nkv) * 64].reshape(2, T, nkv, 64)
        for kvh in range(nkv):  # both q heads of a group equal, so one key can dominate for both
            qh[:, :, 2 * kvh + 1] = qh[:, :, 2 * kvh]
        if kind.startswith("dominant"):
            j = {"dominant_first": 0, "dominant_mid": min(T - 1, 70)}.get(kind)
            kh *= 0.2
            for b in range(2):
                for kvh in range(nkv):
                    qv = qh[b, :, 2 * kvh].astype(np.float64)  # [T, 64]
                    if j is None:  # every row's own key dominates its (causal) window
                        kh[b, :, kvh] = qv * (60.0 / 0.125) / (qv * qv).sum(-1, keepdims=True)
                    else:
                        kh[b, j, kvh] = qv.mean(0) * (60.0 / 0.125) / (qv.mean(0) @ qv.mean(0))
        elif kind == "equal_keys":
            kh[:] = kh[:, :1]
        else:
            qh *= 6.0
            kh *= 6.0
        x[..., :nh * 64] = qh.reshape(2, T, -1)
        x[..., nh * 64:(nh + nkv) * 64] = kh.reshape(2, T, -1)
        out, _ = q.codec_attention_probe(kernel, x, nh, nkv)
        _check_attention(kernel, x, out, nh, nkv, f"kernel {kernel} {kind} T {T}")


# ------------------------------------------------------------------------------------------------ GPU: output conv
OUT_T = [1, 6, 7, 31, 32, 33, 255, 256, 257, 49920]


def _out_inputs(rng, B, T, C, specials):
    x = rng.standard_normal((B, T, C)).astype(np.float32)
    x *= np.asarray([0.1, 3.0, 1.0, 0.5][:B], np.float32)[:, None, None]  # item 0 inside the clip range, item 1 mostly clipped
    w = (rng.standard_normal((7, C)) / np.sqrt(7 * C)).astype(np.float32) * 2
    bias = np.float32(rng.uniform(-0.2, 0.2))
    if specials and T >= 40:
        b = B - 1
        x[b, 10, 3], x[b, 20, C - 1], x[b, 33, 0] = np.inf, np.nan, -np.inf  # rows > 6 apart: each output sees at most one
    return x, w, bias


def _check_out_conv(kernel, x, w, bias, y, label):
    xin = np.asarray(x, np.float64) if kernel == 1 else _r16(x)
    win = _r16(w) if kernel == 3 else np.asarray(w, np.float64)
    want, s = ref_out_conv(xin, win, float(bias))
    e = OUT_ACC_U * U * s + 2 * U
    e = np.where(np.isfinite(e), e, 0.0)  # outputs that saw +-Inf / NaN: exactly +-1 / 0
    _check_abs(y, want, e, label, f"out conv kernel {kernel}")


@pytest.mark.gpu
@pytest.mark.parametrize("C", [32, 64, 96, 128])
def test_out_conv_streaming_kernel(C):
    """Every T of OUT_T with B = 1 and 4, strips of 32, 64 and 256 outputs (the 6-row causal lead-in of every strip, the partial last
    group of 32 stores, rows clamped at T - 1), inputs that clip, +-Inf and NaN."""
    import qwen3tts_b200 as q

    for B in (1, 4):
        for T in OUT_T:
            rng = np.random.default_rng(zlib.crc32(repr(("stream", C, B, T)).encode()))
            x, w, bias = _out_inputs(rng, B, T, C, specials=True)
            for strip in (32, 64, 256):
                y = q.codec_out_conv_probe(0, x, w, bias, strip=strip)
                _check_out_conv(0, x, w, bias, y, f"stream C {C} B {B} T {T} strip {strip}")


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,C", [(1, 32), (1, 96), (1, 160), (2, 64), (2, 128), (2, 160), (3, 32), (3, 96), (3, 128), (3, 160)])
def test_out_conv_other_kernels(kernel, C):
    """The SIMT kernel on fp32 / fp16 input and the tcgen05 GEMM's pcm epilogue (the tensor-core pipeline's output conv when C is not
    one of the streaming kernel's), same cases."""
    import qwen3tts_b200 as q

    for B in (1, 4):
        for T in OUT_T:
            rng = np.random.default_rng(zlib.crc32(repr(("other", kernel, C, B, T)).encode()))
            x, w, bias = _out_inputs(rng, B, T, C, specials=True)
            y = q.codec_out_conv_probe(kernel, x, w, bias)
            _check_out_conv(kernel, x, w, bias, y, f"kernel {kernel} C {C} B {B} T {T}")


# ------------------------------------------------------------------------------------------------ GPU: row ops
ROW_C = [12, 96, 1024, 1536]


@pytest.mark.gpu
@pytest.mark.parametrize("C", ROW_C)
def test_row_ops(C):
    """dwconv7 (T = 1, 5, 7, 33 per item: causal taps must stop at every item boundary), LayerNorm (fp32 / fp16 out), RMSNorm with fp16
    out (ldx > dim, with and without weight), SnakeBeta and SiLU * up, on C not a multiple of 256 included."""
    import qwen3tts_b200 as q

    rng = np.random.default_rng(C)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    for B, T in ((5, 1), (3, 5), (2, 7), (3, 33)):
        x = f(B * T, C) * np.repeat(np.asarray([1.0, 40.0, 0.02, 3.0, 7.0][:B], np.float32), T)[:, None]
        w, b = f(7, C) * 0.3, f(C) * 0.1
        y = q.codec_rowop_probe("dwconv7", x, C, w=w, b=b, T=T)
        xs = x.reshape(B, T, C).astype(np.float64)
        want = np.zeros_like(xs) + b
        sabs = np.zeros_like(xs) + np.abs(b)
        for k in range(7):
            sh = 6 - k
            if sh >= T:
                continue
            want[:, sh:] += xs[:, :T - sh] * w[k]
            sabs[:, sh:] += np.abs(xs[:, :T - sh] * w[k])
        _check_abs(y.reshape(B, T, C), want, ROW_U * U * sabs, f"dwconv7 C {C} B {B} T {T}", "dwconv7")
    rows = 37
    x = f(rows, C) * 3 + f(rows, 1) * 2  # rows with a mean offset
    w, b = f(C), f(C) * 0.5
    mu = x.astype(np.float64).mean(-1, keepdims=True)
    xc = x - mu
    inv = 1.0 / np.sqrt((xc * xc).mean(-1, keepdims=True) + 1e-6)
    want = xc * inv * w + b
    e = ROW_U * U * (np.abs(xc * inv * w) + np.abs(x).mean(-1, keepdims=True) * inv * np.abs(w) + np.abs(b))
    _check_abs(q.codec_rowop_probe("layernorm", x, C, w=w, b=b, eps=1e-6), want, e, f"layernorm C {C}", "layernorm")
    _check_interval(q.codec_rowop_probe("layernorm_f16", x, C, w=w, b=b, eps=1e-6), want, e, f"layernorm_f16 C {C}", "layernorm_f16")
    ldx = C + 40
    xl = f(rows, ldx) * 2
    xr = xl[:, :C].astype(np.float64)
    inv = 1.0 / np.sqrt((xr * xr).mean(-1, keepdims=True) + 1e-6)
    for wn in (w, None):
        want = xr * inv * (1.0 if wn is None else wn)
        _check_interval(q.codec_rowop_probe("rmsnorm_f16", xl, C, w=wn, eps=1e-6), want, ROW_U * U * np.abs(want), f"rmsnorm_f16 C {C}", "rmsnorm_f16")
    ea = np.exp(rng.uniform(-1, 3, C)).astype(np.float32)
    ieb = (1.0 / (np.exp(rng.uniform(-1, 1, C)) + 1e-9)).astype(np.float32)
    xs = x.astype(np.float64)
    want, s = ref_snake(xs, ea, ieb)
    e = ROW_U * U * (np.abs(xs) + ieb) + 2 * ieb * np.abs(s) * U * (2 * np.abs(xs * ea) + 4)
    _check_abs(q.codec_rowop_probe("snake", x, C, w=ea, b=ieb), want, e, f"snake C {C}", "snake")
    gu = f(rows, 2 * C) * 4
    g, u = gu[:, :C].astype(np.float64), gu[:, C:].astype(np.float64)
    want = g / (1 + np.exp(-g)) * u
    _check_abs(q.codec_rowop_probe("silu_mul", gu, C), want, ROW_U * U * np.abs(want) + 1e-38, f"silu_mul C {C}", "silu_mul")
