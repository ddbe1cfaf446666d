"""The device sampler (csrc/sampler.cuh) one launch at a time against the float64 reference of tests/sampler_ref.py, in both of its
forms: form 0 = sample_block<0, 512> as sample_kernel / q3tts_sample_token run it, form 1 = sample_block<1, 480> on warps 0-14 of a
512-thread CTA as the persistent frame kernel runs it (q3tts_sampler_probe, q3tts_sampler_slot_probe).

* Kept sets: the finite entries of the processed row (after penalty, temperature, top-k and the valid-id mask) equal the reference's,
  bit for bit.  Top-p: the kept set matches for every id whose reference mass of strictly more probable ids is more than 1e-5 from p
  (the device sums expf in fp32 in block order); ids inside that band may go either way, but the kept set is a prefix in probability
  order.
* Ids: the argmax of processed + Gumbel(counter_uniform) on every row whose top two perturbed scores are more than 8 fp32 ulp apart;
  on the other rows one of those two.  The excused rows are counted and printed.
* Per-slot rules against the restatement of the generation loop in tests/sampler_ref.py."""
import numpy as np
import pytest

import sampler_ref as R

pytestmark = pytest.mark.gpu

FORMS = [0, 1]
BAND = 1e-5
UNWRITTEN = 0x7F7F7F7F  # the probes fill their output buffers with this pattern before the launch
# (V, codec_vocab): V straddles 480 / 512 threads, the warp width and the bitmap words; the valid-id mask runs when V == codec_vocab
SHAPES = [(1, 3072), (31, 3072), (33, 3072), (480, 3072), (481, 3072), (512, 3072), (513, 3072), (2048, 2048), (3072, 3072), (3072, 2048),
          (4095, 3072), (4096, 4096)]


def _cases(V, codec_vocab, rng):
    """Rows of (logits, temperature, top_k, top_p, penalty, set ids) at the edges where a sampler goes wrong."""
    rows = []
    add = lambda lg, t=1.0, k=0, p=1.0, r=1.0, s=(): rows.append((np.asarray(lg, np.float32), t, k, p, r, list(s)))
    ks = sorted({1, max(V - 1, 1), V, V + 7, int(rng.integers(1, V + 1))})
    ps = [1e-7, 0.5, 0.99, 1.0]
    # coarse grid: many ties at the top-k and top-p thresholds
    for k in ks + [0]:
        for p in ps:
            for t in (0.5, 1.0, 2.0):
                add(rng.integers(-6, 6, V) * 0.5, t, k, p)
    # signed zeros tied at the threshold
    for k in (1, 2, 3, 0):
        for p in (1e-7, 0.3, 1.0):
            lg = -rng.integers(0, 3, V).astype(np.float32)
            lg[rng.random(V) < 0.5] = 0.0
            lg[lg == 0] = np.where(rng.random(int((lg == 0).sum())) < 0.5, 0.0, -0.0)
            add(lg, 1.0, k, p)
            add(lg, 0.0)  # greedy: the first zero wins whatever its sign
    # -inf entries: fewer finite entries than k, a fully -inf row
    for k in (1, 5, V):
        lg = rng.standard_normal(V) * 2
        lg[rng.random(V) < 0.8] = -np.inf
        add(lg, 0.9, k, 0.9)
        add(lg, 0.9, k, 1.0)
    add(np.full(V, -np.inf), 1.0, 3, 0.5)
    add(np.full(V, -np.inf), 0.0)
    # top-k = 1 at an invalid id: every entry is -inf after the mask -> id 0
    if V == codec_vocab and V > 2049:
        for bad in (2048, 2149, V - 1):
            lg = rng.standard_normal(V)
            lg[bad] = 40.0
            add(lg, 1.0, 1, 1.0)
            add(lg, 1.0, 1, 0.5)
    # one dominant logit, also in the last warp of either form
    for pos in {0, V - 1, min(470, V - 1), min(500, V - 1), min(511, V - 1), int(rng.integers(0, V))}:
        lg = rng.standard_normal(V)
        lg[pos] = 30.0
        add(lg, 1.0)
        add(lg, 0.0)
        add(lg, 0.7, 0, 0.5)
    # logit scales and temperatures
    for scale in (1e-3, 1e4):
        for t in (0.05, 0.3, 1.0, 2.0):
            for k, p in ((0, 1.0), (7, 1.0), (0, 0.9)):
                add(rng.standard_normal(V) * scale, t, k, p)
    # penalty on positive, negative, zero and -inf logits at set ids 0, 31, 32, 2047, 2148 and V - 1
    ids = sorted({i for i in (0, 31, 32, 2047, 2148, V - 1) if i < V})
    for r in (1.3, 0.7, 1.0):
        for sign in (1.0, -1.0, 0.0, -np.inf):
            lg = rng.standard_normal(V) * 0.5
            lg[ids] = sign * (1.0 + 0.1 * np.arange(len(ids)))
            add(lg, 0.0, 0, 1.0, r, ids)
            add(lg, 0.8, 3, 0.9, r, ids)
            add(lg, 1.0, 0, 1.0, r, ids)
    # plain sampled rows: enough counters that the id check means something
    n_plain = 1200 - len(rows)
    for i in range(n_plain):
        k = [0, 0, 20, V // 2][i % 4]
        p = [1.0, 0.9, 1.0, 0.8][(i // 4) % 4]
        s = rng.integers(0, V, size=int(rng.integers(0, 12))).tolist()
        add(rng.standard_normal(V) * 2.5, float(rng.uniform(0.3, 1.5)), k, p, 1.1, s)
    return rows


def _run(form, V, codec_vocab, rows, seeds, counters, want_processed=True):
    import qwen3tts_b200 as q

    lg = np.stack([r[0] for r in rows])
    sets = np.stack([R.bitmap(r[5]) for r in rows])
    return q.sampler_probe(form, lg, [r[1] for r in rows], [r[2] for r in rows], [r[3] for r in rows], [r[4] for r in rows], seeds, counters,
                           token_sets=sets, codec_vocab=codec_vocab, want_processed=want_processed)


@pytest.fixture(scope="module")
def cases():
    out = {}
    for V, cv in SHAPES:
        rng = np.random.default_rng(V * 7 + cv)
        rows = _cases(V, cv, rng)
        n = len(rows)
        seeds = rng.integers(0, 2 ** 63, size=n, dtype=np.uint64)
        counters = rng.integers(0, 2 ** 40, size=n, dtype=np.uint64)
        lg = np.stack([r[0] for r in rows])
        sets = np.zeros((n, V), bool)
        for i, r in enumerate(rows):
            sets[i, r[5]] = True
        ref = R.reference(lg, [r[1] for r in rows], [r[2] for r in rows], [r[3] for r in rows], [r[4] for r in rows], sets, cv)
        out[(V, cv)] = (rows, seeds, counters, ref)
    return out


@pytest.mark.parametrize("form", FORMS)
def test_sampler_kept_sets_and_ids_against_float64_reference(form, cases):
    total_rows = total_sampled = total_excused = total_band = 0
    for (V, cv), (rows, seeds, counters, ref) in cases.items():
        ids, proc = _run(form, V, cv, rows, seeds, counters)
        ids_plain, _ = _run(form, V, cv, rows, seeds, counters, want_processed=False)
        assert np.array_equal(ids, ids_plain), f"V {V}: the dump instantiation draws other ids than the plain one"
        tp = ~ref.greedy & (np.array([r[3] for r in rows]) < 1.0)
        got_fin, want_fin = np.isfinite(proc), np.isfinite(ref.processed)
        for i in range(len(rows)):
            t, k, p, r, s = rows[i][1:]
            what = f"form {form} V {V} codec_vocab {cv} row {i} (T {t}, k {k}, p {p}, penalty {r}, set {s[:6]})"
            assert (proc[i].view(np.uint32) != UNWRITTEN).all(), f"{what}: processed row not written in full"
            if not tp[i]:
                assert np.array_equal(got_fin[i], want_fin[i]), f"{what}: kept set differs at {np.flatnonzero(got_fin[i] != want_fin[i])[:8]}"
            else:
                cand = np.isfinite(ref.before_top_p[i])
                sure = cand & ((ref.mass[i] == 0) | ~(np.abs(ref.mass[i] - p) <= BAND))  # a mass of exactly 0 is exact on the device too
                bad = sure & (got_fin[i] != want_fin[i])
                assert not bad.any(), f"{what}: top-p kept set differs outside the band at {np.flatnonzero(bad)[:8]}"
                assert not (got_fin[i] & ~cand).any(), f"{what}: top-p kept an id removed before it"
                kept_v, drop_v = ref.before_top_p[i][got_fin[i]], ref.before_top_p[i][cand & ~got_fin[i]]
                assert kept_v.size == 0 or drop_v.size == 0 or kept_v.min() > drop_v.max(), f"{what}: top-p kept set is not a prefix"
                assert np.array_equal(proc[i][got_fin[i]].view(np.uint32), ref.before_top_p[i][got_fin[i]].view(np.uint32)), what
                total_band += int((cand & ~sure).sum())
            # finite values bit for bit (penalty and temperature are IEEE divisions on both sides)
            m = got_fin[i] & want_fin[i]
            assert np.array_equal(proc[i][m].view(np.uint32), ref.processed[i][m].view(np.uint32)), f"{what}: processed values differ"
            assert (proc[i][~got_fin[i]] == -np.inf).all(), f"{what}: removed entries must be -inf"
        # ids from the device's processed rows (equal to the reference's outside the top-p band)
        want, near, second = R.expected_ids(proc, ref.greedy, seeds, counters)
        ok = (ids == want) | (near & (ids == second))
        bad = np.flatnonzero(~ok)
        assert bad.size == 0, f"form {form} V {V}: ids differ on rows {bad[:8]}: got {ids[bad[:8]]}, want {want[bad[:8]]}"
        total_rows += len(rows)
        total_sampled += int((~ref.greedy).sum())
        total_excused += int(near.sum())
    print(f"[form {form}] {total_rows} rows ({total_sampled} sampled): {total_excused} ids excused as near-ties (8 ulp), "
          f"{total_band} top-p candidates inside the 1e-5 band")
    assert total_excused <= total_sampled // 1000 + 2


@pytest.mark.parametrize("form", FORMS)
def test_signed_zero_ties_survive_the_thresholds(form):
    """[0, -0, -1, -0, 0]: top-k = 1 and top-p = 0.3 keep all four zeros; the processed row keeps each zero's sign."""
    lg = np.array([0.0, -0.0, -1.0, -0.0, 0.0], np.float32)
    for k, p in ((1, 1.0), (0, 0.3), (2, 0.05), (4, 1e-7)):
        ids, proc = _run(form, 5, 3072, [(lg, 1.0, k, p, 1.0, [])], [3], [4])
        assert np.isfinite(proc[0]).tolist() == [True, True, False, True, True], (k, p, proc[0])
        assert np.array_equal(proc[0].view(np.uint32)[[0, 1, 3, 4]], lg.view(np.uint32)[[0, 1, 3, 4]])
        assert ids[0] in (0, 1, 3, 4)


@pytest.mark.parametrize("form", FORMS)
def test_one_shared_row(form):
    """ld = 0: every row reads row 0; rows differ only by their counters."""
    import qwen3tts_b200 as q

    rng = np.random.default_rng(5)
    lg = (rng.standard_normal(513) * 2).astype(np.float32)
    n = 1000
    counters = np.arange(n, dtype=np.uint64) * 16 + 3
    ids, proc = q.sampler_probe(form, lg, 0.8, 0, 1.0, 1.0, 77, counters, n_rows=n, want_processed=True)
    full, _ = q.sampler_probe(form, np.tile(lg, (n, 1)), 0.8, 0, 1.0, 1.0, 77, counters)
    assert np.array_equal(ids, full)
    ref = R.reference(lg[None], [0.8], [0], [1.0], [1.0], None, 3072)
    assert np.array_equal(proc.view(np.uint32), np.tile(ref.processed, (n, 1)).view(np.uint32))
    assert np.unique(ids).size > 50


# ------------------------------------------------------------------------------------------------ per-slot rules
V0, VC = 3072, 2048  # code0 head / code-predictor heads (the valid-id mask runs on the code0 head only)
WORDS = V0 // 32


def _state(n, **kw):
    st = dict(active=1, finished=0, step=0, max_tokens=100, trailing_idx=0, total_text=0, consecutive_pad=0, n_forced=0, stream_variant=0,
              frame_alive=0, logits_cap=0)
    st.update(kw)
    return {f: np.broadcast_to(np.asarray(v, np.int32), (n,)).copy() for f, v in st.items()}


def _greedy_id(V, cv):
    def pick(row, set_ids):
        sets = None
        if set_ids:
            sets = np.zeros((1, V), bool)
            sets[0, [i for i in set_ids if i < V]] = True
        return int(R.reference(row[None], [0.0], [0], [1.0], [1.05], sets, cv).processed[0].argmax())
    return pick


def _probe(form, group, logits, st, sets, codes, temperature=0.0, forced=None, dump_frames=None, dump_slot=0, penalty=1.05):
    import qwen3tts_b200 as q

    V = logits.shape[1]
    smp = dict(temperature=temperature, top_k=0, top_p=1.0, repetition_penalty=penalty, seed=11)
    return q.sampler_slot_probe(form, group, logits, st, smp, sets, codes, R.EOS_ID, R.PAD_ID, V0, forced=forced, dump_slot=dump_slot,
                                dump_frames=dump_frames)


def _check_against_restatement(form, group, logits, st, sets, codes, forced=None, dump_frames=None, dump_slot=0):
    """One launch over every slot == the restatement applied to each slot alone."""
    V = logits.shape[1]
    got_st, got_sets, got_codes, dump = _probe(form, group, logits, st, sets, codes, forced=forced, dump_frames=dump_frames, dump_slot=dump_slot)
    for s in range(logits.shape[0]):
        one = {f: int(st[f][s]) for f in R.SLOT_INT_FIELDS}
        w_st, w_sets, w_codes, dumped = R.slot_step(group, one, logits[s], sets[s], codes[s], _greedy_id(V, V0),
                                                    forced=None if forced is None else forced[s], V=V)
        assert {f: int(got_st[f][s]) for f in R.SLOT_INT_FIELDS} == w_st, f"form {form} group {group} slot {s}"
        assert np.array_equal(got_sets[s], w_sets), f"form {form} group {group} slot {s}: token sets"
        assert np.array_equal(got_codes[s], w_codes), f"form {form} group {group} slot {s}: cur_codes"
        if dump is not None and s == dump_slot:
            step = one["step"]
            if dumped:
                assert np.array_equal(dump[step], logits[s]), "dump must hold the raw logits"
            assert (dump[np.arange(len(dump)) != (step if dumped else -1)].view(np.uint32) == UNWRITTEN).all(), "dump written outside its row"
    return got_st, got_sets, got_codes, dump


@pytest.mark.parametrize("form", FORMS)
def test_slot_rules_code0(form):
    """Group 0 over 8 slots of different states in one launch, each slot == the restatement: EOS / pad suppressed while text remains even
    when they dominate, EOS finishes, a pad run below 7 continues, a non-pad id resets the run, forced EOS / pad finish nothing,
    step >= max_tokens finishes without sampling, inactive and finished slots do nothing."""
    rng = np.random.default_rng(1)
    n = 10
    lg = rng.standard_normal((n, V0)).astype(np.float32)
    dom = [R.EOS_ID, R.PAD_ID, R.EOS_ID, R.PAD_ID, 17, R.EOS_ID, R.PAD_ID, 5, R.PAD_ID, R.EOS_ID]
    lg[np.arange(n), dom] = 50.0
    st = _state(n, trailing_idx=[0, 0, 3, 3, 3, 3, 3, 3, 3, 3], total_text=[2, 2, 3, 3, 3, 3, 3, 0, 3, 3],
                consecutive_pad=[0, 0, 0, 5, 4, 0, 0, 0, 6, 0], n_forced=[0, 0, 0, 0, 0, 1, 1, 0, 0, 0],
                step=[0, 1, 2, 3, 4, 2, 2, 9, 5, 3], max_tokens=[100, 100, 100, 100, 100, 100, 100, 9, 100, 100],
                active=[1, 1, 1, 1, 1, 1, 1, 1, 1, 0], finished=[0, 0, 0, 0, 0, 0, 0, 0, 0, 0])
    forced = np.full((n, 16, 16), 7, np.int32)
    forced[5, 2, 0], forced[6, 2, 0] = R.EOS_ID, R.PAD_ID
    sets = np.zeros((n, 16, WORDS), np.uint32)
    sets[:, 0] = R.bitmap([1, 2, 3], WORDS)
    codes = np.full((n, 16), -5, np.int32)
    got_st, got_sets, got_codes, _ = _check_against_restatement(form, 0, lg, st, sets, codes, forced=forced)
    assert got_codes[0, 0] not in (R.EOS_ID, R.PAD_ID) and got_codes[1, 0] not in (R.EOS_ID, R.PAD_ID)
    assert got_st["finished"].tolist() == [0, 0, 1, 0, 0, 0, 0, 1, 1, 0]
    assert got_st["consecutive_pad"].tolist()[:5] == [0, 0, 0, 6, 0]
    assert got_st["frame_alive"].tolist() == [1, 1, 0, 1, 1, 1, 1, 0, 0, 0]
    assert got_codes[5, 0] == R.EOS_ID and got_codes[6, 0] == R.PAD_ID
    assert np.array_equal(got_sets, sets), "group 0 records nothing: frame_finalize adds code0 to its set"


@pytest.mark.parametrize("form", FORMS)
def test_seventh_consecutive_pad_stops(form):
    """Frame by frame, state fed back (step + 1, frame_alive cleared, as step_advance does): pads 1-6 continue, the 7th finishes;
    a non-pad id in between resets the run."""
    n = 2
    lg = np.full((n, V0), -3.0, np.float32)
    lg[:, R.PAD_ID] = 20.0
    st = _state(n, trailing_idx=4, total_text=4)
    sets = np.zeros((n, 16, WORDS), np.uint32)
    codes = np.zeros((n, 16), np.int32)
    for frame in range(8):
        x = lg.copy()
        if frame == 3:
            x[1, 42] = 30.0  # slot 1 draws a non-pad id at frame 3
        st, sets, codes, _ = _check_against_restatement(form, 0, x, st, sets, codes)
        want_pad = [min(frame + 1, 7), (frame - 3) if frame > 3 else (0 if frame == 3 else frame + 1)]
        assert st["consecutive_pad"].tolist() == want_pad, frame
        assert st["finished"].tolist() == [int(frame >= 6), int(frame >= 10)], frame
        st["step"] += 1
        st["frame_alive"][:] = 0


@pytest.mark.parametrize("form", FORMS)
def test_slot_rules_code_predictor_groups(form):
    """Groups >= 1: nothing when frame_alive is 0; the id is recorded in the group's own set only; the stream variant drops the penalty
    of these groups; group 0 keeps its penalty in the stream variant."""
    n = 4
    lg = np.full((n, VC), -5.0, np.float32)
    lg[:, 10], lg[:, 20] = -1.0, -1.02  # dividing -1.02 by 1.05 makes id 20 the argmax (Qwen3Talker.swift:288-299)
    st = _state(n, frame_alive=[1, 0, 1, 1], stream_variant=[0, 0, 1, 0])
    sets = np.zeros((n, 16, WORDS), np.uint32)
    for g in (3, 15):
        sets[:, g] = R.bitmap([20], WORDS)
    codes = np.full((n, 16), -5, np.int32)
    got_st, got_sets, got_codes, _ = _check_against_restatement(form, 3, lg, st, sets, codes)
    assert got_codes[:, 3].tolist() == [20, -5, 10, 20]
    assert R.bitmap_ids(got_sets[2, 3]) == {10, 20} and R.bitmap_ids(got_sets[0, 3]) == {20}
    assert np.array_equal(np.delete(got_sets, 3, axis=1), np.delete(sets, 3, axis=1)), "only the group's own set changes"
    _check_against_restatement(form, 15, lg, st, sets, codes)
    # group 0 (code0 head) keeps its penalty in the stream variant
    l0 = np.full((2, V0), -5.0, np.float32)
    l0[:, 10], l0[:, 20] = -1.0, -1.02
    s0 = np.zeros((2, 16, WORDS), np.uint32)
    s0[:, 0] = R.bitmap([20], WORDS)
    st0 = _state(2, stream_variant=[0, 1], trailing_idx=1, total_text=1)
    _, _, c0, _ = _check_against_restatement(form, 0, l0, st0, s0, np.zeros((2, 16), np.int32))
    assert c0[:, 0].tolist() == [20, 20]


@pytest.mark.parametrize("form", FORMS)
def test_logits_dump_only_for_dump_slot_below_cap(form):
    rng = np.random.default_rng(3)
    n = 3
    lg = rng.standard_normal((n, V0)).astype(np.float32)
    for step, cap in ((0, 2), (1, 2), (2, 2), (5, 0)):
        st = _state(n, step=step, logits_cap=cap, trailing_idx=1, total_text=1)
        _, _, _, dump = _check_against_restatement(form, 0, lg, st, np.zeros((n, 16, WORDS), np.uint32), np.zeros((n, 16), np.int32),
                                                   dump_frames=3, dump_slot=1)
        assert (step < cap) == bool((dump.view(np.uint32) != UNWRITTEN).any()), (step, cap)


@pytest.mark.parametrize("form", FORMS)
def test_slot_sampling_matches_row_probe(form):
    """A sampled (temperature > 0) slot draws the id of sample_block at counter step * 16 + group, with the slot's penalty set."""
    import qwen3tts_b200 as q

    rng = np.random.default_rng(9)
    n = 64
    lg = (rng.standard_normal((n, VC)) * 2).astype(np.float32)
    st = _state(n, frame_alive=1, step=np.arange(n) * 3)
    sets = np.zeros((n, 16, WORDS), np.uint32)
    set_ids = [rng.integers(0, VC, size=8).tolist() for _ in range(n)]
    for s in range(n):
        sets[s, 6] = R.bitmap(set_ids[s], WORDS)
    got_st, got_sets, got_codes, _ = _probe(form, 6, lg, st, sets, np.zeros((n, 16), np.int32), temperature=0.9)
    row_sets = np.stack([R.bitmap(i) for i in set_ids])
    want, _ = q.sampler_probe(form, lg, 0.9, 0, 1.0, 1.05, 11, np.arange(n) * 3 * 16 + 6, token_sets=row_sets, codec_vocab=V0)
    assert np.array_equal(got_codes[:, 6], want)
    for s in range(n):
        assert R.bitmap_ids(got_sets[s, 6]) == set(set_ids[s]) | {int(want[s])}
