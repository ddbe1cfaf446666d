"""Float64 reference of the device sampler (csrc/sampler.cuh) with the oracle's semantics (oracle/talker.py `TalkerOracle.sample`),
vectorised over rows, and a restatement of the generation loop's per-slot rules (`TalkerOracle.generate_codes`, the sampling
points of its frame loop) for one sampling point of one group.

Order of `sampleToken` (Model/Qwen3Talker.swift:274-322): penalty by division whatever the sign -> greedy returns (before the mask)
-> division by the temperature -> top-k keeps the k-th largest value and every tie (float comparison, so -0.0 == +0.0) -> the
valid-id mask (< 2048, 2148, 2150) when V == codec_vocab -> top-p keeps id i iff the mass of strictly more probable ids is < p
-> Gumbel-max over `counter_uniform`."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from oracle.talker import counter_uniform

CODEBOOK = 2048
PAD_ID, EOS_ID = 2148, 2150


def bitmap(ids, words=128) -> np.ndarray:
    """uint32 bitmap of `words` words with the bits of `ids` set (the device's token-set layout)."""
    b = np.zeros(words, np.uint32)
    for t in ids:
        b[t >> 5] |= np.uint32(1 << (t & 31))
    return b


def bitmap_ids(b) -> set:
    b = np.asarray(b, np.uint32)
    return {w * 32 + i for w in range(b.size) for i in range(32) if (int(b[w]) >> i) & 1}


@dataclass
class Reference:
    processed: np.ndarray   # [n, V] fp32: the row just before the Gumbel step (greedy rows: after the penalty)
    mass: np.ndarray        # [n, V] float64: mass of strictly more probable ids (top-p rows; NaN elsewhere)
    before_top_p: np.ndarray  # [n, V] fp32: the row after top-k and the mask, before top-p
    greedy: np.ndarray      # [n] bool


def reference(logits, temperature, top_k, top_p, rep_penalty, sets, codec_vocab) -> Reference:
    """logits fp32 [n, V]; per-row temperature, top_k, top_p, rep_penalty [n]; sets bool [n, V] (ids in the row's token set) or None."""
    x = np.array(logits, np.float32)
    n, V = x.shape
    t = np.asarray(temperature, np.float32)
    k = np.asarray(top_k, np.int64)
    p = np.asarray(top_p, np.float32)
    r = np.asarray(rep_penalty, np.float32)
    if sets is not None:
        pen = np.asarray(sets, bool) & (r != 1.0)[:, None]
        x = np.where(pen, x / r[:, None], x).astype(np.float32)  # IEEE fp32 division, as on the device
    greedy = ~(t > 0)
    x = np.where(greedy[:, None], x, x / np.where(greedy, np.float32(1), t)[:, None]).astype(np.float32)
    tk = ~greedy & (k > 0) & (k < V)
    if tk.any():
        srt = np.sort(x, axis=1)
        thr = srt[np.arange(n), np.clip(V - k, 0, V - 1)]
        x = np.where(tk[:, None] & (x < thr[:, None]), np.float32(-np.inf), x)
    if V == codec_vocab:
        idx = np.arange(V)
        valid = (idx < CODEBOOK) | (idx == PAD_ID) | (idx == EOS_ID)
        x = np.where(~greedy[:, None] & ~valid[None, :], np.float32(-np.inf), x)
    before = x.copy()
    mass = np.full((n, V), np.nan)
    tp = ~greedy & (p < 1.0)
    if tp.any():
        with np.errstate(invalid="ignore", over="ignore"):
            x64 = x.astype(np.float64)
            m = x64.max(axis=1, keepdims=True)
            pr = np.exp(x64 - m)
            z = pr.sum(axis=1, keepdims=True)
            order = np.argsort(-x64, axis=1, kind="stable")
            xs = np.take_along_axis(x64, order, 1)
            ps = np.take_along_axis(pr, order, 1)
            excl = np.cumsum(ps, axis=1) - ps
            first = np.concatenate([np.ones((n, 1), bool), xs[:, 1:] != xs[:, :-1]], axis=1)  # ties share their prefix mass
            greater = np.maximum.accumulate(np.where(first, excl, 0.0), axis=1)
            mg = np.empty_like(greater)
            np.put_along_axis(mg, order, greater, 1)
            mg = mg / z
        mass = np.where(tp[:, None], mg, np.nan)
        keep = mg < p[:, None].astype(np.float64)
        x = np.where(tp[:, None] & ~keep, np.float32(-np.inf), x)
    return Reference(processed=x.astype(np.float32), mass=mass, before_top_p=before, greedy=greedy)


def gumbel_scores(processed, seeds, counters):
    """processed + Gumbel(u) in float64 (u = counter_uniform), -inf where processed is -inf; also the logit and noise terms."""
    n, V = processed.shape
    g = np.stack([-np.log(-np.log(counter_uniform(int(s), int(c), V).astype(np.float64))) for s, c in zip(seeds, counters)])
    x = processed.astype(np.float64)
    fin = np.isfinite(x)
    return np.where(fin, x + g, -np.inf), g


def expected_ids(processed, greedy, seeds, counters):
    """(id, near_tie, runner_up) per row.  Greedy rows: first index of the maximum, never excused.  Sampled rows: argmax of
    processed + Gumbel(u); `near_tie` when the top two perturbed scores are within 8 fp32 ulp of the largest magnitude among the
    winner's score, logit and noise (the device adds the noise in fp32 after two logf calls)."""
    n, V = processed.shape
    ids = np.argmax(processed, axis=1)  # first index; an all -inf row gives 0, as on the device
    near = np.zeros(n, bool)
    second = ids.copy()
    s = ~greedy
    if s.any():
        sc, g = gumbel_scores(processed[s], np.asarray(seeds)[s], np.asarray(counters)[s])
        win = np.argmax(sc, axis=1)
        rows = np.arange(win.size)
        top = sc[rows, win]
        sc2 = sc.copy()
        sc2[rows, win] = -np.inf
        run = np.argmax(sc2, axis=1)
        mag = np.maximum.reduce([np.abs(top), np.abs(processed[s][rows, win].astype(np.float64)), np.abs(g[rows, win])])
        with np.errstate(invalid="ignore"):
            tol = 8 * np.spacing(np.where(np.isfinite(mag), mag, 0).astype(np.float32)).astype(np.float64)
            nt = np.isfinite(top) & np.isfinite(sc2[rows, run]) & (top - sc2[rows, run] <= tol)
        ids[s] = np.where(np.isfinite(top), win, 0)
        second[s] = np.where(nt, run, ids[s])
        near[s] = nt
    return ids, near, second


# ------------------------------------------------------------------------------------------------ per-slot rules
SLOT_INT_FIELDS = ("active", "finished", "step", "max_tokens", "trailing_idx", "total_text", "consecutive_pad", "n_forced", "stream_variant",
                   "frame_alive", "logits_cap")


def slot_step(group, state, logits_row, sets, cur_codes, sampled_id, forced=None, eos=EOS_ID, pad=PAD_ID, V=None):
    """One sampling point of `group` for one slot, restating generate_codes' frame loop (EOS / pad suppression while text remains,
    the EOS and 7-pad stops unless forced, forced ids, the per-group sets) and the engine's max_tokens / frame_alive bookkeeping.
    state: dict of SLOT_INT_FIELDS; sets uint32 [16, words]; cur_codes [16]; sampled_id(row, set_ids or None) -> the sampler's id.
    Returns (state, sets, cur_codes, dumped) -- new copies; dumped is True when this point writes the slot's logits dump."""
    st = dict(state)
    sets = np.array(sets, np.uint32)
    codes = np.array(cur_codes, np.int32)
    V = len(logits_row) if V is None else V
    if group == 0:
        if not (st["active"] and not st["finished"] and st["step"] < st["max_tokens"]):
            st["frame_alive"] = 0
            if st["active"] and st["step"] >= st["max_tokens"]:
                st["finished"] = 1
            return st, sets, codes, False
    elif not st["frame_alive"]:
        return st, sets, codes, False
    dumped = st["step"] < st["logits_cap"]
    row = np.array(logits_row, np.float32)
    if group == 0 and st["trailing_idx"] < st["total_text"]:
        row[eos] = -np.inf
        row[pad] = -np.inf
    use_set = group == 0 or not st["stream_variant"]
    tok = sampled_id(row, bitmap_ids(sets[group]) if use_set else None)
    is_forced = st["n_forced"] > 0 and forced is not None
    if is_forced:
        tok = int(forced[st["step"]][group])
    if group == 0:
        if not is_forced:
            if tok == eos:
                st["finished"], st["frame_alive"] = 1, 0
                return st, sets, codes, dumped
            if tok == pad:
                st["consecutive_pad"] += 1
                if st["consecutive_pad"] > 6:
                    st["finished"], st["frame_alive"] = 1, 0
                    return st, sets, codes, dumped
            else:
                st["consecutive_pad"] = 0
        st["frame_alive"] = 1
    elif 0 <= tok < V:
        sets[group][tok >> 5] |= np.uint32(1 << (tok & 31))
    codes[group] = tok
    return st, sets, codes, dumped
