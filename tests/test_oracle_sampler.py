"""CPU checks of the sampler's reference and of the sampler stream itself.

* tests/sampler_ref.py (the float64 reference tests/test_gpu_sampler.py holds the device sampler to) equals `TalkerOracle.sample`
  bit for bit on finite tie-free rows, and keeps signed zeros tied at a threshold as the oracle does.
* `counter_uniform` + Gumbel-max samples softmax: chi-square tests over 10^5 counters at fixed seeds, before and after top-k / top-p
  (against the renormalised kept set), and consecutive counters / adjacent seeds are independent.
* Both sampler probes refuse out-of-range arguments on the host, before any device is looked for.
All draws use fixed seeds, so every statistic below is deterministic; each threshold is the chi-square quantile at 1 - 1e-6."""
import numpy as np
import pytest
from scipy import stats

import sampler_ref as R
from oracle import talker as otalker
from oracle.talker import counter_uniform

ALPHA = 1e-6  # a correct sampler fails one of these fixed-seed tests with probability ~1e-6 per test


def _oracle(vocab_size):
    """TalkerOracle.sample reads only cfg.vocab_size: an oracle without weights is enough for it."""
    o = otalker.TalkerOracle.__new__(otalker.TalkerOracle)
    o.cfg = type("Cfg", (), {"vocab_size": vocab_size})()
    return o


@pytest.mark.parametrize("V,codec_vocab", [(2048, 3072), (3072, 3072), (513, 3072)])
def test_reference_equals_oracle_on_tie_free_rows(V, codec_vocab):
    orc = _oracle(codec_vocab)
    rng = np.random.default_rng(V)
    modes = [dict(temperature=0.0), dict(temperature=0.9), dict(temperature=0.8, top_k=50), dict(temperature=1.0, top_p=0.8),
             dict(temperature=0.7, top_k=20, top_p=0.9), dict(temperature=1.3, top_k=V - 1, top_p=0.3)]
    n_checked = 0
    for mi, kw in enumerate(modes):
        for trial in range(8):
            lg = ((rng.permutation(V) - V / 2) * (12.0 / V)).astype(np.float32)  # distinct values: no ties
            assert np.unique(lg).size == V
            ts = set(rng.integers(0, V, size=trial * 3).tolist())
            req = otalker.Request(text_ids=[], seed=100 + trial, repetition_penalty=1.1, **kw)
            want_id, want = orc.sample(lg, req, ts if ts else None, counter=trial * 16 + mi)
            sets = np.zeros((1, V), bool)
            sets[0, list(ts)] = True
            ref = R.reference(lg[None], [kw.get("temperature", 0.9)], [kw.get("top_k", 0)], [kw.get("top_p", 1.0)], [1.1], sets, codec_vocab)
            assert np.array_equal(ref.processed[0].view(np.uint32), np.asarray(want, np.float32).view(np.uint32)), (kw, trial)
            ids, near, _ = R.expected_ids(ref.processed, ref.greedy, [100 + trial], [trial * 16 + mi])
            assert near[0] or ids[0] == want_id, (kw, trial)
            n_checked += 1
    assert n_checked == 48


def test_reference_keeps_signed_zero_ties():
    """-0.0 == +0.0: at a top-k or top-p threshold of zero every zero survives, whatever its sign (the oracle's float comparison)."""
    orc = _oracle(3072)
    lg = np.array([0.0, -0.0, -1.0, -0.0, 0.0], np.float32)
    for kw in (dict(top_k=1), dict(top_p=0.3), dict(top_k=2, top_p=0.05)):
        _, want = orc.sample(lg, otalker.Request(text_ids=[], temperature=1.0, **kw), None, 0)
        ref = R.reference(lg[None], [1.0], [kw.get("top_k", 0)], [kw.get("top_p", 1.0)], [1.0], None, 3072)
        assert np.array_equal(ref.processed[0].view(np.uint32), np.asarray(want, np.float32).view(np.uint32))
        assert np.isfinite(ref.processed[0]).tolist() == [True, True, False, True, True]
        assert np.signbit(ref.processed[0][[1, 3]]).all()


# ------------------------------------------------------------------------------------------------ distribution of the stream
def _draws(lg, seed, counters):
    """Gumbel-max ids of row lg (-inf = removed) for every counter, through oracle.talker.counter_uniform."""
    u = counter_uniform(seed, np.asarray(counters, np.uint64)[:, None], lg.size).astype(np.float64)
    z = np.where(np.isfinite(lg), lg.astype(np.float64) - np.log(-np.log(u)), -np.inf)
    return np.argmax(z, axis=1)


def test_vectorised_stream_equals_scalar_calls():
    for c in (0, 1, 17, 2 ** 40 + 3):
        assert np.array_equal(counter_uniform(9, np.array([[c]], np.uint64), 64)[0], counter_uniform(9, c, 64))


def _chi2(counts, probs):
    keep = probs > 0
    assert counts[~keep].sum() == 0, "an id outside the kept set was drawn"
    exp = probs[keep] * counts.sum()
    assert exp.min() >= 5, "expected counts too small for a chi-square test"
    stat = float(((counts[keep] - exp) ** 2 / exp).sum())
    return stat, stats.chi2.ppf(1 - ALPHA, keep.sum() - 1)


def _row64():
    return (np.random.default_rng(64).standard_normal(64) * 1.2).astype(np.float32)


@pytest.mark.parametrize("mode", ["plain", "top_k", "top_p", "top_k_top_p"])
def test_gumbel_max_over_counter_stream_samples_softmax(mode):
    """10^5 counters over 4 seeds: the drawn ids follow softmax of the processed row (the kept set renormalised after top-k / top-p)."""
    lg = _row64()
    k, p = {"plain": (0, 1.0), "top_k": (10, 1.0), "top_p": (0, 0.7), "top_k_top_p": (20, 0.8)}[mode]
    ref = R.reference(lg[None], [1.0], [k], [p], [1.0], None, 0)
    proc = ref.processed[0]
    probs = np.where(np.isfinite(proc), np.exp(proc.astype(np.float64) - proc.max()), 0.0)
    probs /= probs.sum()
    counts = np.zeros(64)
    for seed in (1, 2, 3, 0xDEADBEEF12345):
        counts += np.bincount(_draws(proc, seed, np.arange(25000) + seed * 7), minlength=64)
    stat, thr = _chi2(counts, probs)
    print(f"[{mode}] chi2 {stat:.1f} over {int((probs > 0).sum()) - 1} dof, threshold {thr:.1f}")
    assert stat < thr


@pytest.mark.parametrize("adjacent", ["counter", "seed"])
def test_adjacent_counters_and_seeds_are_independent(adjacent):
    """Joint frequencies of the ids drawn at (counter c, c + 1) -- or at seeds (s, s + 1) with the same counter -- equal the product of
    the marginals: a chi-square test of independence over a V = 8 row."""
    lg = np.array([0.9, 0.4, 0.0, -0.2, -0.5, -0.7, -1.0, 0.2], np.float32)
    n = 100000
    if adjacent == "counter":
        ids = _draws(lg, 5, np.arange(n + 1))
        a, b = ids[:-1], ids[1:]
    else:
        a = np.concatenate([_draws(lg, s, np.arange(n // 50)) for s in range(0, 100, 2)])
        b = np.concatenate([_draws(lg, s + 1, np.arange(n // 50)) for s in range(0, 100, 2)])
    table = np.zeros((8, 8))
    np.add.at(table, (a, b), 1)
    chi2, pval, dof, exp = stats.chi2_contingency(table, correction=False)
    assert exp.min() >= 5
    print(f"[{adjacent}] independence chi2 {chi2:.1f} over {dof} dof, p {pval:.3g}")
    assert pval > ALPHA


# ------------------------------------------------------------------------------------------------ refusals without a device
def _status(fn):
    import qwen3tts_b200 as q

    with pytest.raises(q.Q3Error) as e:
        fn()
    return e.value.status


def test_sampler_probe_refuses_bad_arguments_without_a_device():
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi as A

    lg = np.zeros((2, 64), np.float32)
    call = lambda form=0, x=lg, t=1.0, p=1.0, r=1.0: q.sampler_probe(form, x, t, 0, p, r, 1, 0)
    cases = {"form 2": dict(form=2), "form -1": dict(form=-1), "V 0": dict(x=np.zeros((2, 0), np.float32)),
             "V 4097": dict(x=np.zeros((1, 4097), np.float32)), "no rows": dict(x=np.zeros((0, 64), np.float32)),
             "temperature NaN": dict(t=np.nan), "temperature inf": dict(t=np.inf), "top_p NaN": dict(p=np.nan), "top_p 0": dict(p=0.0),
             "top_p < 0": dict(p=-0.5), "top_p inf": dict(p=np.inf), "penalty inf": dict(r=np.inf), "penalty NaN": dict(r=np.nan)}
    for what, kw in cases.items():
        assert _status(lambda: call(**kw)) == A.ERR_INVALID_ARG, what
    f, i = np.ones(2, np.float32), np.zeros(2, np.int32)
    u = np.zeros(2, np.uint64)
    ids = np.zeros(2, np.int32)
    L = A.lib()
    pf, pi = (lambda a: a.ctypes.data_as(A.p_f32)), (lambda a: a.ctypes.data_as(A.p_i32))
    for ld in (1, 63, -1):  # ld must be 0 (one shared row) or >= V
        assert L.q3tts_sampler_probe(0, 0, pf(lg), 2, 64, ld, 0, pf(f), pi(i), pf(f), pf(f), None, u.ctypes.data, u.ctypes.data, pi(ids), None) == A.ERR_INVALID_ARG
    assert L.q3tts_sampler_probe(0, 0, None, 2, 64, 64, 0, pf(f), pi(i), pf(f), pf(f), None, u.ctypes.data, u.ctypes.data, pi(ids), None) == A.ERR_INVALID_ARG


def test_sampler_slot_probe_refuses_bad_arguments_without_a_device():
    import qwen3tts_b200 as q
    from qwen3tts_b200 import _abi as A

    n, V = 2, 64

    def call(form=0, group=0, V=V, words=2, step=0, forced=None, n_forced=0, dump_slot=0, dump_frames=None, logits_cap=0, p=1.0, t=1.0):
        st = dict(active=1, finished=0, step=step, max_tokens=10, trailing_idx=0, total_text=0, consecutive_pad=0, n_forced=n_forced,
                  stream_variant=0, frame_alive=1, logits_cap=logits_cap)
        smp = dict(temperature=t, top_k=0, top_p=p, repetition_penalty=1.0, seed=1)
        return q.sampler_slot_probe(form, group, np.zeros((n, V), np.float32), st, smp, np.zeros((n, 16, words), np.uint32),
                                    np.zeros((n, 16), np.int32), 62, 63, V, forced=forced, dump_slot=dump_slot, dump_frames=dump_frames)

    forced = np.zeros((n, 4, 16), np.int32)
    cases = {"form 2": dict(form=2), "group 16": dict(group=16), "group -1": dict(group=-1), "V 4097": dict(V=4097, words=129),
             "set words too few": dict(words=1), "step < 0": dict(step=-1), "forced past max_frames": dict(forced=forced, n_forced=1, step=4),
             "dump slot out of range": dict(dump_frames=4, dump_slot=2), "logits_cap above dump_frames": dict(dump_frames=4, logits_cap=5),
             "top_p 0": dict(p=0.0), "temperature NaN": dict(t=np.nan)}
    for what, kw in cases.items():
        assert _status(lambda: call(**kw)) == A.ERR_INVALID_ARG, what
