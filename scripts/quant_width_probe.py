"""Cost of the 4/8-bit container for 0.6B MLX checkpoints of 3, 4, 5, 6 and 8 bits (group 64) and for an mxfp4 checkpoint (held as 8-bit
affine groups of 32 with bf16 scales and biases).

For each width: handle load time, batch-1 ms per frame on the persistent frame kernel (device time of >= 100 teacher-forced frames, prefill
excluded), ms per frame step of a 64-row handle, and q3tts_timing.weight_bytes_per_frame (container bytes).  2/3-bit checkpoints stream 4-bit
words and 5/6-bit ones 8-bit words, so the expectation is 3 == 4 and 5 == 6 == 8 at batch 1 within run-to-run spread, and all widths equal
at 64 rows (the batched step reads the same fp16 copies).  Each width is measured `--reps` times, alternating widths inside a repetition.

    python scripts/quant_width_probe.py [--out results.json] [--bits 3 4 5 6 8 mxfp4] [--reps 3]
Needs a B200; the checkpoints go to a temporary directory."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "mlx-swift-qwen3-tts_b200"), os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402

import qwen3tts_b200 as q  # noqa: E402
import mlx_mxfp4  # noqa: E402
import mlx_widths  # noqa: E402
from oracle import checkpoint  # noqa: E402

FRAMES_B1 = 128
ROWS, FRAMES_B64 = 64, 24


def gpu_card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still worth printing; say why the card is unknown
        return f"unknown ({e})"


def requests(n, frames, seed):
    rng = np.random.default_rng(seed)
    forced = rng.integers(0, 2048, size=(n, frames, 16)).astype(np.int32)
    return [q.GenRequest(text_ids=[11, 21, 22] + rng.integers(100, 600, size=12).tolist(), speaker_id=2861, temperature=0.0, max_tokens=frames,
                         forced_codes=forced[i], keep_invalid_frames=True) for i in range(n)]


def step_ms(eng, reqs, frames, batch):
    if batch:
        eng.generate_codes_batch(reqs)
    else:
        eng.generate_codes(reqs[0])
    t = eng.timing()
    return (t.talker_ms - t.prefill_ms) / frames, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bits", nargs="+", default=["3", "4", "5", "6", "8"], help="widths, or mxfp4")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    card = gpu_card()
    print(f"card: {card}", flush=True)
    res = {b: {"load_s": [], "b1_ms_per_frame": [], "b64_ms_per_step": []} for b in a.bits}
    with tempfile.TemporaryDirectory() as tmp:
        dirs = {}
        for b in a.bits:
            t0 = time.time()
            if b in ("4", "8"):
                dirs[b] = checkpoint.write_checkpoint(os.path.join(tmp, f"b{b}"), "0.6b", bits=int(b), with_codec=False)
            elif b == "mxfp4":  # E2M1 leaves with E8M0 group scales (tests/mlx_mxfp4.py)
                dirs[b] = mlx_mxfp4.write_mxfp4_checkpoint(os.path.join(tmp, b), "0.6b")[0]
            else:  # 2/3/5/6-bit leaves in MLX's bit-stream layout (tests/mlx_widths.py)
                dirs[b] = mlx_widths.write_width_checkpoint(os.path.join(tmp, f"b{b}"), "0.6b", bits=int(b), group=64)[0]
            print(f"{b}-bit checkpoint written in {time.time() - t0:.0f} s", flush=True)
        r1, r64 = requests(1, FRAMES_B1, 1), requests(ROWS, FRAMES_B64, 2)
        for rep in range(a.reps):
            for b in a.bits:
                t0 = time.time()
                e1 = q.Engine(dirs[b], max_frames=FRAMES_B1 + 8, load_codec=False)
                res[b]["load_s"].append(time.time() - t0)
                step_ms(e1, r1, FRAMES_B1, False)  # warm-up
                ms, t = step_ms(e1, r1, FRAMES_B1, False)
                assert t.persistent_launches >= 1 and t.frames == FRAMES_B1, (t.persistent_launches, t.frames)
                res[b]["b1_ms_per_frame"].append(ms)
                res[b]["weight_bytes_per_frame"] = int(t.weight_bytes_per_frame)
                res[b]["quant_bits"], res[b]["checkpoint_quant_bits"] = e1.info.quant_bits, e1.info.checkpoint_quant_bits
                res[b]["quant_group_size"], res[b]["checkpoint_quant_mode"] = e1.info.quant_group_size, e1.info.checkpoint_quant_mode
                e1.close()
                e64 = q.Engine(dirs[b], max_batch=ROWS, max_frames=FRAMES_B64 + 8, load_codec=False)
                step_ms(e64, r64, FRAMES_B64, True)
                ms64, t = step_ms(e64, r64, FRAMES_B64, True)
                assert t.persistent_launches == 0
                res[b]["b64_ms_per_step"].append(ms64)
                e64.close()
                print(json.dumps({"rep": rep, "bits": b, "load_s": round(res[b]["load_s"][-1], 2), "b1_ms_per_frame": round(ms, 4),
                                  "b64_ms_per_step": round(ms64, 4)}), flush=True)
    summary = {"card": card, "model": "0.6b bf16 scales, g64 (mxfp4: g32)", "frames_b1": FRAMES_B1, "rows_b64": ROWS, "results": {}}
    for b in a.bits:
        r = res[b]
        summary["results"][b] = {k: (round(float(np.median(v)), 4) if isinstance(v, list) else v) for k, v in r.items()}
        summary["results"][b]["b1_spread_ms"] = round(float(np.max(r["b1_ms_per_frame"]) - np.min(r["b1_ms_per_frame"])), 4)
        summary["results"][b]["b64_spread_ms"] = round(float(np.max(r["b64_ms_per_step"]) - np.min(r["b64_ms_per_step"])), 4)
    print(json.dumps(summary, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(summary, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
