"""K-A2 time of bf16 vs fp32 gradients: device-gated rounds (K-A0 + K-A2, what the Accumulator launches) with all ranks
in one process, timed with the context's own CUDA events (mb_ar_round_times).

    python tools/ar_lowp_micro.py [--worlds 1,2,4,8] [--iters 30] [--out profiles/lowp_ar_micro.json]

Sizes: the IMPALA gradient set (1,094,476 elements) and 67,108,864 elements (256 MB in fp32, 128 MB in bf16), each in
fp32 and bf16, one-shot and two-shot (in place, as the Accumulator consumes it).  Before timing, every configuration's
result is checked bit for bit against the CPU restatement (oracle.allreduce_rankorder for fp32, tests/lowp_oracle.py for
bf16): on every element for the IMPALA size, on 1 Mi evenly strided elements for the large one.  Bus bandwidth uses the
bytes actually moved, with the same formula for both dtypes: bytes * 2(N-1)/N / K-A2 time.  The GPU's name and power
limit are read in the same run and written into the output."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import lowp_oracle as lo  # noqa: E402
import oracle  # noqa: E402
from moolib_b200 import _lib  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--worlds", default="1,2,4,8", help="world sizes above the GPU count are skipped")
ap.add_argument("--sizes", default="1094476,67108864")
ap.add_argument("--dtypes", default="f32,bf16")
ap.add_argument("--iters", type=int, default=30)
ap.add_argument("--out", default="")
a = ap.parse_args()
assert torch.cuda.is_available(), "ar_lowp_micro needs a GPU"
TORCH_DT = {"f32": torch.float32, "bf16": torch.bfloat16}
ALG = {"oneshot": _lib.MB_AR_ALGO_ONESHOT, "twoshot": _lib.MB_AR_ALGO_TWOSHOT}
WARMUP = 5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpus": q, "torch_device": torch.cuda.get_device_name(0), "device_count": torch.cuda.device_count()}


def as_np(t, dt):
    t = t.detach().cpu()
    return t.numpy() if dt == "f32" else t.view(torch.int16).numpy().view(np.uint16)


def expected(ins, dt, n):
    if dt == "f32":
        return oracle.allreduce_rankorder(ins, [(1, 0, 1)] * n, scale=False)[0]
    return lo.allreduce_rankorder(ins, [(1, 0, 1)] * n, dt, scale=False)[0]


def run(n, numel, dt, results):
    spec = [(numel, TORCH_DT[dt])]
    _, total, _ = _lib.layout([numel], [dt])
    ctx = [_lib.ArContext(r, n, r, total) for r in range(n)]
    hs = [c.export() for c in ctx]
    for r, c in enumerate(ctx):
        for q in range(n):
            if q != r:
                c.import_peer(q, hs[q])
    src = []
    for r in range(n):
        g = torch.Generator(device=f"cuda:{r}").manual_seed(100 + r)
        src.append(torch.randn(numel, device=f"cuda:{r}", generator=g).to(TORCH_DT[dt]))
    dst = [torch.empty(total, dtype=torch.uint8, device=f"cuda:{r}") for r in range(n)]
    sample = slice(None) if numel <= 4 << 20 else slice(0, numel, numel // (1 << 20))
    ins = [np.ascontiguousarray(as_np(s, dt)[sample]) for s in src]  # the ctypes oracle reads raw memory
    exp = expected(ins, dt, n)
    for algo in ("oneshot", "twoshot") if n > 1 else ("oneshot",):
        red, gate = [], []
        for it in range(WARMUP + a.iters):
            outs = []
            for r in range(n):
                with torch.cuda.device(r):
                    if it == 0:
                        ctx[r].stage_ex([src[r]])
                    else:
                        ctx[r].buffer_bytes(total).fill_(r + 1)  # outside the timed events
                    out = ctx[r].buffer_bytes(total) if algo == "twoshot" else dst[r]
                    outs.append(out)
            for r in range(n):
                with torch.cuda.device(r):
                    ctx[r].reduce_gated_ex(1, spec, flat_dst=outs[r], hdr=(1, 0, 1, 1), scale=False, algo=ALG[algo])
            for r in range(n):
                torch.cuda.synchronize(r)
            assert all(ctx[r].result()[1] == 0 for r in range(n)), (n, numel, dt, algo)
            if it == 0:
                for r in range(n):
                    got = as_np(outs[r][:numel * src[r].element_size()].view(TORCH_DT[dt]), dt)[sample]
                    assert got.tobytes() == exp.tobytes(), f"N={n} {numel} x {dt} {algo}: rank {r} differs from the oracle"
            ts = [ctx[r].round_times() for r in range(n)]
            if it >= WARMUP:
                red.append(max(t[1] for t in ts))
                gate.append(max(t[0] for t in ts))
            for r in range(n):
                ctx[r].advance()
        red.sort()
        gate.sort()
        med = red[len(red) // 2]
        nbytes = numel * src[0].element_size()
        row = {"n": n, "numel": numel, "dtype": dt, "bytes": nbytes,
               "algo": algo + (" (in place)" if algo == "twoshot" else ""), "reduce_us_p50": round(med, 2),
               "p10": round(red[len(red) // 10], 2), "p90": round(red[len(red) * 9 // 10], 2),
               "gate_us_p50": round(gate[len(gate) // 2], 2),
               "busbw_gbs": round(nbytes * 2 * (n - 1) / n / med / 1e3, 1), "checked_vs_oracle": True}
        print(json.dumps(row), flush=True)
        results.append(row)
    for c in ctx:
        c.close()


def main():
    info = gpu_info()
    print(json.dumps(info), flush=True)
    results = []
    for n in [int(x) for x in a.worlds.split(",") if int(x) <= torch.cuda.device_count()]:
        for numel in [int(x) for x in a.sizes.split(",")]:
            for dt in a.dtypes.split(","):
                run(n, numel, dt, results)
    # bf16 vs fp32 K-A2 time at the same element count (median over the timed rounds)
    ratio = []
    for r in results:
        if r["dtype"] == "bf16":
            f = next(x for x in results if x["dtype"] == "f32" and x["n"] == r["n"] and x["numel"] == r["numel"]
                     and x["algo"] == r["algo"])
            ratio.append({"n": r["n"], "numel": r["numel"], "algo": r["algo"], "fp32_us": f["reduce_us_p50"],
                          "bf16_us": r["reduce_us_p50"], "bf16_over_fp32": round(r["reduce_us_p50"] / f["reduce_us_p50"], 3)})
    doc = {"tool": "tools/ar_lowp_micro.py", "iters": a.iters, "warmup": WARMUP, "gpu": info, "rows": results,
           "bf16_vs_fp32": ratio}
    if a.out:
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)
    for x in ratio:
        print(json.dumps(x), flush=True)


if __name__ == "__main__":
    main()
