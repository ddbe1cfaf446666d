"""Talker attention kernels (csrc/talker_kernels.cu) against a float64 reference, one launch at a time (q3tts_attention_probe).

kernel 0 = rope_attention_kernel (decode: norm + RoPE + append + window attention, one row per slot), kernel 1 =
qk_norm_rope_append + attention_kernel (prefill: several rows per slot, causal inside the launch), kernel 2 =
cp_pass0_attention_kernel (code-predictor pass 0: rows 2s, 2s+1 at positions 0, 1).

The reference (`reference` / `ref_attend`) is the operation of Model/Qwen3Layers.swift:167-218 on a ring: per-head RMSNorm,
rotate-half RoPE with the angle taken as the fp32 product fp32(pos) * inv_freq (what the kernels and MLX compute; only that rounding
is kept), append of k / v at pos % capacity, softmax over the window [win_start, pos] read through the ring, all in float64.
test_reference_matches_the_oracle anchors it on oracle/talker.py, so a wrong reference cannot agree with a wrong kernel.

What is asserted after every launch:
  * ring contents: every entry the launch must not write is bit-identical to its input (no stray writes); the appended V is a
    bit-exact copy of the row's v (fp16-rounded on fp16 rings); the appended K is the float64 roped k within K_ULPS fp32 ulp of
    |x| + |y| (the two normalised operands of its rotation; CUDA's rsqrtf alone is specified at 2 ulp, the norm weight, sincosf
    and the rotation's two products add one rounding each), plus 1 fp16 ulp of the value on fp16 rings;
  * outputs: against the reference evaluated over the ring the kernel returned (isolates the attention arithmetic from the rounding
    of the append): |err| <= OUT_REL * max|V_window| per (row, head), plus 1 fp16 ulp of the reference value for fp16 outputs.
"""
import zlib

import numpy as np
import pytest

# Measured on a B200 (1000 W), all cases of this file: appended K <= 2.2 fp32 ulp of |x| + |y|; fp32 outputs <= 2.7e-7 x max|V_window|.
K_ULPS = 4
OUT_REL = 2e-6
SCALE = np.float64(np.float32(1.0) / np.sqrt(np.float32(128.0)))  # the kernels' 1.0f / sqrtf(128.0f)
EPS = 1e-6
KV_HEADS = 2
U32 = np.uint32


def _inv_freq(theta=1e6):
    e = np.arange(0, 128, 2, dtype=np.float32) / np.float32(128.0)
    return (np.float32(1.0) / np.power(np.float32(theta), e)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ float64 reference
def _norm_rope(x, w, eps, pos, inv_freq):
    """x [..., 128] (float64 of fp32 values) at absolute position `pos` -> (roped, |x_n| + |y_n| per element)."""
    n = x / np.sqrt(np.mean(x * x, axis=-1, keepdims=True) + eps) * w
    ang = (np.float32(pos) * np.asarray(inv_freq, dtype=np.float32)).astype(np.float64)  # fp32 angle, as the kernels and MLX
    c, s = np.cos(ang), np.sin(ang)
    a, b = n[..., :64], n[..., 64:]
    mag = np.abs(a) + np.abs(b)
    return np.concatenate([a * c - b * s, b * c + a * s], -1), np.concatenate([mag, mag], -1)


def reference(qkv, heads, kv_heads, q_norm, k_norm, eps, inv_freq, row_pos):
    """-> q [m, heads, 128], k [m, kv_heads, 128] (roped), v [m, kv_heads, 128], |x| + |y| of k; float64."""
    x = np.asarray(qkv, dtype=np.float64).reshape(len(row_pos), heads + 2 * kv_heads, 128)
    qn, kn = np.asarray(q_norm, np.float64), np.asarray(k_norm, np.float64)
    q, k, kmag = [], [], []
    for r, p in enumerate(row_pos):
        q.append(_norm_rope(x[r, :heads], qn, eps, int(p), inv_freq)[0])
        kr, km = _norm_rope(x[r, heads:heads + kv_heads], kn, eps, int(p), inv_freq)
        k.append(kr)
        kmag.append(km)
    return np.stack(q), np.stack(k), x[:, heads + kv_heads:].copy(), np.stack(kmag)


def ref_attend(q, k_ring, v_ring, row_slot, row_pos, win_start, scale=SCALE):
    """softmax(q k^T * scale) v over keys [win_start[slot], pos] read at ring index position % capacity.
    -> out [m, heads * 128], max|V_window| [m, heads]."""
    m, heads, _ = q.shape
    kv_heads, cap = k_ring.shape[1], k_ring.shape[2]
    G = heads // kv_heads
    out = np.zeros((m, heads, 128))
    vmax = np.zeros((m, heads))
    for r in range(m):
        s, p = int(row_slot[r]), int(row_pos[r])
        w0 = 0 if win_start is None else int(win_start[s])
        idx = np.arange(w0, p + 1) % cap
        for kvh in range(kv_heads):
            K = np.asarray(k_ring[s, kvh, idx], np.float64)
            V = np.asarray(v_ring[s, kvh, idx], np.float64)
            sc = q[r, kvh * G:(kvh + 1) * G] @ K.T * scale  # [G, S]
            e = np.exp(sc - sc.max(-1, keepdims=True))
            out[r, kvh * G:(kvh + 1) * G] = (e / e.sum(-1, keepdims=True)) @ V
            vmax[r, kvh * G:(kvh + 1) * G] = np.abs(V).max()
    return out.reshape(m, heads * 128), vmax


def _ulp16(x):
    return np.spacing(np.abs(x).astype(np.float16)).astype(np.float64)


def _round_f16(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


# ------------------------------------------------------------------------------------------------ one launch, checked
STATS = {}


def _run_and_check(kernel, qkv, heads, q_norm, k_norm, inv_freq, row_slot, row_pos, win_start, k_in, v_in, kv_f16, out_f16, label):
    import qwen3tts_b200 as q

    kv_heads = k_in.shape[1]
    cap = k_in.shape[2]
    if kv_f16:  # the probe rounds the rings to fp16 on upload: start from representable values so "unchanged" is exact
        k_in, v_in = _round_f16(k_in), _round_f16(v_in)
    out, k_out, v_out = q.attention_probe(kernel, qkv, heads, kv_heads, q_norm, k_norm, EPS, inv_freq, row_slot, row_pos, win_start, k_in, v_in,
                                          kv_f16=kv_f16, out_f16=out_f16)
    qr, kr, vr, kmag = reference(qkv, heads, kv_heads, q_norm, k_norm, EPS, inv_freq, row_pos)
    # ring contents
    written = np.zeros(k_in.shape[:3], dtype=bool)
    for r in range(len(row_pos)):
        written[row_slot[r], :, row_pos[r] % cap] = True
    keep = ~written
    assert np.array_equal(k_out.view(U32)[keep], k_in.view(U32)[keep]), f"{label}: K ring entries outside the appended slots changed"
    assert np.array_equal(v_out.view(U32)[keep], v_in.view(U32)[keep]), f"{label}: V ring entries outside the appended slots changed"
    k_err = 0.0  # largest error / bar of the appended K
    for r in range(len(row_pos)):
        s, ring = row_slot[r], row_pos[r] % cap
        got_k = k_out[s, :, ring].astype(np.float64)
        bar = K_ULPS * 2.0 ** -23 * kmag[r]
        if kv_f16:
            bar = bar + _ulp16(kr[r])
        err = np.abs(got_k - kr[r])
        k_err = max(k_err, float((err / bar).max()))
        assert np.all(err <= bar), f"{label}: row {r} (slot {s}, pos {row_pos[r]}): appended K off by {err.max():.3e}"
        want_v = vr[r].astype(np.float32)
        if kv_f16:
            want_v = _round_f16(want_v)
        assert np.array_equal(v_out[s, :, ring].view(U32), want_v.view(U32)), f"{label}: row {r}: appended V is not a copy of v"
    # outputs, over the ring the kernel returned
    ref, vmax = ref_attend(qr, k_out, v_out, row_slot, row_pos, win_start)
    err = np.abs(out.astype(np.float64) - ref).reshape(len(row_pos), heads, 128)
    rel = err / vmax[:, :, None]
    bar = OUT_REL * vmax[:, :, None] + (_ulp16(ref).reshape(err.shape) if out_f16 else 0.0)
    bad = np.argwhere(err > bar)
    if len(bad):
        r, h, d = bad[0]
        raise AssertionError(f"{label}: {len(bad)} outputs off; first row {r} (slot {row_slot[r]}, pos {row_pos[r]}, window start "
                             f"{0 if win_start is None else win_start[row_slot[r]]}) head {h} dim {d}: got {out[r, h * 128 + d]:.7g}, "
                             f"want {ref[r, h * 128 + d]:.7g}, err / max|V| = {rel[r, h, d]:.3e}")
    key = (kernel, "kv16" if kv_f16 else "kv32", "out16" if out_f16 else "out32")
    k0, o0, b0 = STATS.get(key, (0.0, 0.0, 0.0))
    STATS[key] = (max(k0, k_err), max(o0, float(rel.max())), max(b0, float((err / bar).max())))
    return out, k_out, v_out


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for (kernel, kv, o), (ke, oe, ob) in sorted(STATS.items()):
        print(f"[attention probe] kernel {kernel} {kv} {o}: appended K uses {ke:.2f} of its bar; "
              f"max output error {oe:.3e} x max|V_window| ({ob:.2f} of its bar)")


def _inputs(rng, m, heads, kv_heads, n_slots, cap, q_scale=(0.5, 1.5)):
    qkv = rng.standard_normal((m, (heads + 2 * kv_heads) * 128)).astype(np.float32)
    q_norm = rng.uniform(*q_scale, 128).astype(np.float32)
    k_norm = rng.uniform(0.5, 1.5, 128).astype(np.float32)
    k_ring = rng.standard_normal((n_slots, kv_heads, cap, 128)).astype(np.float32)
    v_ring = rng.standard_normal((n_slots, kv_heads, cap, 128)).astype(np.float32)
    return qkv, q_norm, k_norm, k_ring, v_ring


# ------------------------------------------------------------------------------------------------ CPU: the reference itself
def test_reference_matches_the_oracle():
    """Same inputs through oracle/talker.py's attention (float64 weights that select q / k / v from the row, identity o_proj) and
    through `reference` + `ref_attend`: a causal prefill of 20 rows, and one decode row over a cache of 37 keys."""
    import torch

    from oracle import talker as otalker

    rng = np.random.default_rng(0)
    nh, nkv = 4, 2
    D = (nh + 2 * nkv) * 128
    o = otalker.TalkerOracle.__new__(otalker.TalkerOracle)
    sel = lambda a, b: torch.from_numpy(np.eye(D)[a * 128:b * 128])
    qn = rng.uniform(0.5, 1.5, 128)
    kn = rng.uniform(0.5, 1.5, 128)
    o.w = {"a.q_proj.weight": sel(0, nh), "a.k_proj.weight": sel(nh, nh + nkv), "a.v_proj.weight": sel(nh + nkv, nh + 2 * nkv),
           "a.q_norm.weight": torch.from_numpy(qn), "a.k_norm.weight": torch.from_numpy(kn), "a.o_proj.weight": torch.eye(nh * 128, dtype=torch.float64)}
    # dyadic frequencies: fp32(pos) * inv_freq is exact, so the oracle's float64 angle equals the kernels' fp32 product
    inv_freq = rng.integers(1, 1024, 64) / 1024.0
    oscale = np.float64(1.0 / np.sqrt(np.float32(128)))
    cap = 64
    # prefill: 20 rows at positions 7..26, window starting at 7
    L, p0 = 20, 7
    x = rng.standard_normal((L, D)).astype(np.float32).astype(np.float64)
    want, (kc, vc) = o._attention("a", torch.from_numpy(x), None, torch.arange(p0, p0 + L), torch.from_numpy(inv_freq), nh, nkv, 128, EPS)
    qr, kr, vr, _ = reference(x, nh, nkv, qn, kn, EPS, inv_freq, np.arange(p0, p0 + L))
    k_ring = np.zeros((1, nkv, cap, 128))
    v_ring = np.zeros((1, nkv, cap, 128))
    for r in range(L):
        k_ring[0, :, (p0 + r) % cap] = kr[r]
        v_ring[0, :, (p0 + r) % cap] = vr[r]
    got, _ = ref_attend(qr, k_ring, v_ring, np.zeros(L, int), np.arange(p0, p0 + L), np.array([p0]), scale=oscale)
    np.testing.assert_allclose(got, want.numpy(), rtol=1e-12, atol=1e-12 * np.abs(vr).max())
    np.testing.assert_allclose(kr.transpose(1, 0, 2), kc.numpy(), rtol=1e-12, atol=1e-12)
    # decode: one row at position 100 after 37 cached keys (positions 63..99), through a ring of 64 that wraps
    T, p = 37, 100
    kprev, vprev = rng.standard_normal((nkv, T, 128)), rng.standard_normal((nkv, T, 128))
    x1 = rng.standard_normal((1, D)).astype(np.float32).astype(np.float64)
    want, _ = o._attention("a", torch.from_numpy(x1), (torch.from_numpy(kprev), torch.from_numpy(vprev)), torch.arange(p, p + 1),
                           torch.from_numpy(inv_freq), nh, nkv, 128, EPS)
    qr, kr, vr, _ = reference(x1, nh, nkv, qn, kn, EPS, inv_freq, [p])
    k_ring = rng.standard_normal((1, nkv, cap, 128))
    v_ring = rng.standard_normal((1, nkv, cap, 128))
    for j in range(T):
        k_ring[0, :, (p - T + j) % cap] = kprev[:, j]
        v_ring[0, :, (p - T + j) % cap] = vprev[:, j]
    k_ring[0, :, p % cap], v_ring[0, :, p % cap] = kr[0], vr[0]
    got, _ = ref_attend(qr, k_ring, v_ring, [0], [p], np.array([p - T]), scale=oscale)
    np.testing.assert_allclose(got, want.numpy(), rtol=1e-12, atol=1e-12 * max(np.abs(vprev).max(), np.abs(vr).max()))


def test_probe_rejects_out_of_range_input_before_any_launch():
    """Invalid windows, slots, groups and row layouts return Q3TTS_ERR_INVALID_ARG from the host-side validation (no device needed)."""
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi as A

    rng = np.random.default_rng(1)
    heads, cap = 4, 16
    qkv, qn, kn, kr, vr = _inputs(rng, 2, heads, KV_HEADS, 2, cap)
    f = _inv_freq()
    call = lambda kernel, slots, pos, win, h=heads, kvh=KV_HEADS, x=qkv, **kw: q.attention_probe(kernel, x, h, kvh, qn, kn, EPS, f, slots, pos, win,
                                                                                               kr[:, :kvh], vr[:, :kvh], **kw)
    bad = {
        "window longer than the ring": lambda: call(0, [0, 1], [16, 3], [0, 0]),
        "window start after the position": lambda: call(0, [0, 1], [5, 3], [6, 0]),
        "negative window start": lambda: call(1, [0, 1], [5, 3], [-1, 0]),
        "slot out of range": lambda: call(0, [0, 2], [5, 3], None),
        "two decode rows in one slot": lambda: call(0, [1, 1], [5, 6], None),
        "two prefill rows at one position": lambda: call(1, [1, 1], [5, 5], None),
        "GQA group 3": lambda: call(0, [0, 1], [5, 3], None, h=6, x=np.zeros((2, (6 + 4) * 128), np.float32)),
        "kernel 2 at positions (1, 2)": lambda: call(2, [0, 0], [1, 2], None, out_f16=True),
        "kernel 2 on an fp16 cache": lambda: call(2, [0, 0], [0, 1], None, kv_f16=True, out_f16=True),
        "unknown kernel": lambda: call(3, [0, 1], [5, 3], None),
    }
    for what, fn in bad.items():
        with pytest.raises(q.Q3Error) as e:
            fn()
        assert e.value.status == A.ERR_INVALID_ARG, f"{what}: status {e.value.status}"


# ------------------------------------------------------------------------------------------------ GPU: decode kernel
S_VALUES = [1, 2, 15, 16, 17, 31, 32, 33, 64, 127, 128, 129, 192, 193, 207]
CAPS = [32, 208, 211, 512, 1000]
PLACEMENTS = {  # (S, cap) -> (win_start, pos)
    "first_lap": lambda S, cap: (0, S - 1),
    "start_at_ring_0": lambda S, cap: (2 * cap, 2 * cap + S - 1),
    "start_at_ring_end": lambda S, cap: (3 * cap - 1, 3 * cap + S - 2),
    "pos_at_ring_0": lambda S, cap: (3 * cap - S + 1, 3 * cap),
    "pos_at_ring_end": lambda S, cap: (4 * cap - S, 4 * cap - 1),
    "far": lambda S, cap: (3000 - (S % 7) - S + 1, 3000 - (S % 7)),
}
DTYPES = [(False, False), (False, True), (True, False), (True, True)]


def _s_values(cap):
    if cap == 32:  # the code predictor's cache: at most 17 positions
        return [s for s in S_VALUES if s <= 17]
    return sorted(set([s for s in S_VALUES if s <= cap] + [cap - 1]))


@pytest.mark.gpu
@pytest.mark.parametrize("kv_f16,out_f16", DTYPES, ids=["kv32-out32", "kv32-out16", "kv16-out32", "kv16-out16"])
@pytest.mark.parametrize("G", [1, 2, 4])
@pytest.mark.parametrize("placement", list(PLACEMENTS))
@pytest.mark.parametrize("cap", CAPS)
def test_decode_kernel_window_through_the_ring(cap, placement, G, kv_f16, out_f16):
    """One launch per case holds one slot per window length S (row_slot in reverse order, so row r is not slot r)."""
    rng = np.random.default_rng(zlib.crc32(repr((cap, placement, G, kv_f16, out_f16)).encode()))
    heads = G * KV_HEADS
    Ss = _s_values(cap)
    n = len(Ss)
    qkv, qn, kn, kr, vr = _inputs(rng, n, heads, KV_HEADS, n, cap)
    win = np.zeros(n, np.int32)
    row_slot = np.arange(n)[::-1].astype(np.int32)
    row_pos = np.zeros(n, np.int32)
    for r, S in enumerate(Ss):
        w0, pos = PLACEMENTS[placement](S, cap)
        assert pos - w0 + 1 == S and w0 >= 0
        win[row_slot[r]] = w0
        row_pos[r] = pos
    _run_and_check(0, qkv, heads, qn, kn, _inv_freq(), row_slot, row_pos, win, kr, vr, kv_f16, out_f16, f"decode cap {cap} {placement} G {G}")


STRESS = ["dominant_first", "dominant_current", "dominant_last_warp_group", "identical_keys", "large_q_norm"]


@pytest.mark.gpu
@pytest.mark.parametrize("kv_f16,out_f16", DTYPES, ids=["kv32-out32", "kv32-out16", "kv16-out32", "kv16-out16"])
@pytest.mark.parametrize("G", [1, 2, 4])
@pytest.mark.parametrize("kind", STRESS)
def test_decode_kernel_softmax_extremes(kind, G, kv_f16, out_f16):
    """One key ahead of all others by a score gap of ~80 (every other weight ~e^-80) at window index 0, at the current position, and at
    a key of the last warp's lane groups (j % 32 in 12..15, 28..31); all keys identical; q_norm weights ~6 (scores of tens)."""
    rng = np.random.default_rng(zlib.crc32(repr((kind, G, kv_f16, out_f16)).encode()))
    cap, heads = 208, G * KV_HEADS
    Ss = [17, 33, 129, 207]
    n = len(Ss)
    qkv, qn, kn, kr, vr = _inputs(rng, n, heads, KV_HEADS, n, cap, q_scale=(5.0, 7.0) if kind == "large_q_norm" else (0.5, 1.5))
    kr *= 0.3
    f = _inv_freq()
    row_slot = np.arange(n)[::-1].astype(np.int32)
    row_pos = np.array([700 + 13 * r for r in range(n)], np.int32)
    win = np.zeros(n, np.int32)
    x = qkv.reshape(n, heads + 2 * KV_HEADS, 128)
    gap = 80.0
    if kind == "dominant_current":  # k = every q head of its group, same norm weight: the new key is q itself
        w = np.float32(np.sqrt(gap / (128 * SCALE)))
        qn[:] = w
        kn[:] = w
        for kvh in range(KV_HEADS):
            x[:, kvh * G + 1:(kvh + 1) * G] = x[:, kvh * G:kvh * G + 1]
            x[:, heads + kvh] = x[:, kvh * G]
    elif kind.startswith("dominant"):
        for kvh in range(KV_HEADS):
            x[:, kvh * G + 1:(kvh + 1) * G] = x[:, kvh * G:kvh * G + 1]
    qr, krr, _, _ = reference(qkv, heads, KV_HEADS, qn, kn, EPS, f, row_pos)
    for r, S in enumerate(Ss):
        s, pos = row_slot[r], row_pos[r]
        win[s] = pos - S + 1
        if kind in ("dominant_first", "dominant_last_warp_group"):
            j = 0 if kind == "dominant_first" else (31 if S > 31 else 15)
            for kvh in range(KV_HEADS):
                qv = qr[r, kvh * G]
                kr[s, kvh, (win[s] + j) % cap] = qv * (gap / SCALE) / float(qv @ qv)
        elif kind == "identical_keys":
            for kvh in range(KV_HEADS):
                kr[s, kvh, (win[s] + np.arange(S - 1)) % cap] = krr[r, kvh]
    out, _, v_out = _run_and_check(0, qkv, heads, qn, kn, f, row_slot, row_pos, win, kr, vr, kv_f16, out_f16, f"softmax {kind} G {G}")
    if kind.startswith("dominant"):  # the result is the dominant key's value row
        for r, S in enumerate(Ss):
            s, pos = row_slot[r], row_pos[r]
            j = {"dominant_first": 0, "dominant_current": S - 1}.get(kind, 31 if S > 31 else 15)
            for kvh in range(KV_HEADS):
                v = v_out[s, kvh, (win[s] + j) % cap]
                for g in range(G):
                    h = kvh * G + g
                    np.testing.assert_allclose(out[r, h * 128:(h + 1) * 128], v, rtol=2e-3 if out_f16 else 1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------ GPU: prefill kernel
@pytest.mark.gpu
@pytest.mark.parametrize("kv_f16,out_f16", DTYPES, ids=["kv32-out32", "kv32-out16", "kv16-out32", "kv16-out16"])
@pytest.mark.parametrize("G", [1, 2, 4])
@pytest.mark.parametrize("cap", [208, 211, 512, 1000])
def test_prefill_kernel_causal_through_the_ring(cap, G, kv_f16, out_f16):
    """Three slots in one launch, rows shuffled: a fresh prompt of capacity - 16 positions; 37 rows whose positions cross ring index 0
    after 50 older keys of the window; 5 rows near position 2900 whose window starts at the first of them."""
    rng = np.random.default_rng(zlib.crc32(repr((cap, G, kv_f16, out_f16)).encode()))
    heads = G * KV_HEADS
    P = cap - 16
    p1 = 3 * cap - 10
    slots = [(0, 0, P), (1, p1 - 50, 37), (2, 2900, 5)]  # (slot, win_start, rows starting at win_start / p1 / 2900)
    rows = [(0, p) for p in range(P)] + [(1, p1 + i) for i in range(37)] + [(2, 2900 + i) for i in range(5)]
    order = rng.permutation(len(rows))
    row_slot = np.array([rows[i][0] for i in order], np.int32)
    row_pos = np.array([rows[i][1] for i in order], np.int32)
    win = np.array([w for _, w, _ in slots], np.int32)
    qkv, qn, kn, kr, vr = _inputs(rng, len(rows), heads, KV_HEADS, 3, cap)
    _run_and_check(1, qkv, heads, qn, kn, _inv_freq(), row_slot, row_pos, win, kr, vr, kv_f16, out_f16, f"prefill cap {cap} G {G}")


# ------------------------------------------------------------------------------------------------ GPU: code-predictor geometry
@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 2, 4])
def test_code_predictor_cache_geometry(G):
    """The code predictor's cache (32 positions, no window): pass 0 as kernel 2 and as kernel 1 (rows 2s, 2s+1 at positions 0, 1),
    passes 1..15 as kernel 0 (one row per slot at position g + 1, win_start NULL)."""
    rng = np.random.default_rng(G)
    heads, cap, n = G * KV_HEADS, 32, 5
    f = _inv_freq(1e4)
    qkv, qn, kn, kr, vr = _inputs(rng, 2 * n, heads, KV_HEADS, n, cap)
    row_slot = np.repeat(np.arange(n), 2).astype(np.int32)
    row_pos = np.tile([0, 1], n).astype(np.int32)
    _run_and_check(2, qkv, heads, qn, kn, f, row_slot, row_pos, None, kr, vr, False, True, f"cp pass 0 kernel 2 G {G}")
    for kv_f16, out_f16 in DTYPES:
        _run_and_check(1, qkv, heads, qn, kn, f, row_slot, row_pos, None, kr, vr, kv_f16, out_f16, f"cp pass 0 kernel 1 G {G}")
    qkv, qn, kn, kr, vr = _inputs(rng, n, heads, KV_HEADS, n, cap)
    row_slot = np.arange(n)[::-1].astype(np.int32)
    row_pos = np.array([1, 4, 9, 15, 16], np.int32)
    for kv_f16, out_f16 in DTYPES:
        _run_and_check(0, qkv, heads, qn, kn, f, row_slot, row_pos, None, kr, vr, kv_f16, out_f16, f"cp pass g kernel 0 G {G}")
