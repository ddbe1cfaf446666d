"""On-box: per-phase timing of the split-K cluster GEMM (q3tts_skinny_trace) for the batched-decode shapes.  Not the bench."""
import ctypes as C, os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "mlx-swift-qwen3-tts_b200"))
import numpy as np
from qwen3tts_b200 import _abi as A

M = int(sys.argv[1]) if len(sys.argv) > 1 else 64
BITS = int(sys.argv[2]) if len(sys.argv) > 2 else 0  # 0: fp16-copy kernel, 4 / 8: dequant-fused kernel
SHAPES = [("qkv", 4096, 1024, 0, 0), ("o", 1024, 2048, 0, 1), ("gate_up", 6144, 1024, 1, 0), ("down", 1024, 3072, 0, 1), ("lm_head", 2048, 1024, 0, 0)]
for name, N, K, swiglu, res in SHAPES:
    cap = 512
    st = np.zeros((cap, 16), dtype=np.uint64)
    tiles, split, stages = C.c_int32(), C.c_int32(), C.c_int32()
    us = C.c_double()
    A.check(A.lib().q3tts_skinny_trace_q(0, M, N, K, BITS, swiglu, res, 40, st.ctypes.data_as(C.POINTER(C.c_uint64)), cap, C.byref(tiles), C.byref(split),
                                         C.byref(stages), C.byref(us)), None)
    n = tiles.value * split.value
    s = st[:n].astype(np.int64)
    g0 = s[:, 0].min()
    rel = lambda a: (a - s[:, 1])  # cycles since CTA entry
    cyc = {k: rel(s[:, i]) for k, i in (("setup", 2), ("first_stage", 3), ("acc_done", 4), ("shipped", 5), ("peers_in", 6), ("epi_done", 7), ("exit", 8), ("w3_peers_in", 10), ("w3_reduced", 11), ("w3_finished_chunk0", 12), ("w3_done", 13), ("w3_dequant_done", 14), ("w3_dependency_resolved", 15))}
    out = {"shape": name, "bits": BITS, "M": M, "N": N, "K": K, "grid": [tiles.value, split.value], "stages": stages.value, "avg_us_per_launch": round(us.value, 2),
           "cta_start_spread_us": round(float(s[:, 0].max() - g0) / 1e3, 2), "kernel_span_us": round(float(s[:, 9].max() - g0) / 1e3, 2)}
    for k, v in cyc.items():
        out[k + "_cyc(med,max)"] = [int(np.median(v)), int(v.max())]
    print(json.dumps(out), flush=True)
