#!/usr/bin/env python
"""bench.py -- IMPALA / V-trace learner frames/sec on synthetic 84x84x4 uint8 observations (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (config.workload): BASELINE.json configs[1] at N=1, configs[2] at N>1 -- the actor-learner loop of the
reference's examples/vtrace (examples/impala.py here) with a 256-env synthetic EnvPool x 2 buffers, unroll_length 20
(T=21), batch_size 32 per learner, virtual_batch_size 32*N, the atari ResNet (1,094,476 fp32 parameters), Adam,
grad-norm clipping.  One process = one learner = one GPU; a "step" is one optimizer step (640 frames per learner);
frames/s = unroll_length * batch_size * optimizer_steps / s, the reference's own env_train_steps definition
(examples/vtrace/experiment.py:155,207-211), summed over all N learners.

Before anything is timed, two CHECKED reductions run through the public Accumulator on the real 36-tensor gradient
layout (rank r contributes r+1, then randn(seed=r)): every rank's result must equal the CPU oracle bit for bit and all
ranks must hold identical bits -- the `"parity"` object of the JSON line; a mismatch ends the run with exit code 3.

Two timed regions of exactly K steps each (after --settle untimed steady-state steps and W warm-up steps each), barrier +
cuda synchronize on both sides, CUDA events, max over ranks:
  value : observations already resident in HBM, no host reads inside the loop
  e2e   : observations arrive in pinned host slabs (the EnvPool result format) and are copied H2D every actor step,
          the grad-norm is read back to the host every optimizer step (as experiment.py:166 does) -- through the
          public moolib API (Batcher / Accumulator).
Both go through moolib_b200's Batcher (copy kernels) and Accumulator (stage + NVLink allreduce kernels).
`roofline` is the dominant moolib_b200 kernel family by device time inside the `value` region (the UnrollBatcher gather:
one launch per unroll), timed with CUDA events around every Batcher launch; `per_op` lists all of them and their
aggregate.  `roofline_nvlink` is K-A2 inside the same region, timed by the allreduce context's own CUDA events on the
reduce stream (K-A0 = the wait for the slowest peer is reported separately).  Successive launches touch different
buffers (T=21 x 256 envs x 28 KB = 152 MB per unroll, > L2), so inputs are larger than L2 (config.l2 says so).

`--impl reference` runs the UNMODIFIED reference (oracle/_ref, compiled from /root/reference by oracle/build_ref.sh)
through the same loop on the host cores (device "cpu": its Batcher / Accumulator / RPC allreduce are CPU code and so is
the model then), bounded in wall time; rank 0 only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "impala_learner_frames_per_sec"
UNIT = "frames/s"
ROW_BYTES = 4 * 84 * 84


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--settle", type=int, default=56,
                    help="untimed optimizer steps in front of the W warm-up steps of each arm: the learner-batch queue fills "
                         "to its cap over ~3 unroll cycles (~40 steps) and until then every cycle makes the caching allocator "
                         "cudaMalloc another set of 152 MB unroll buffers (a device-synchronising call); cuDNN's autotuner "
                         "settles too.  Lock-step learners stall on ANY rank's hiccup, so N ranks see N times as many")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--max-seconds", type=float, default=150.0, help="wall-time bound of the reference / cpu legs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-cuda", type=int, default=1, help="also time the reference built with -DUSE_CUDA (info only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed optimizer step of each arm computed to "
                         "DIR/<arm>_<name>.npy (rank 0; see dump_arrays).  The loop then runs reproducibly, which "
                         "costs time: the timings of such a run are not benchmark numbers")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class ClockSampler:
    """SM clocks / throttle reasons DURING the timed region (B200_PROFILING.md), read through NVML from a thread of this
    process every 100 ms.  (Round 1 ran `nvidia-smi -lms 200` as a child process: its queries, and the fork of this
    process that started it, showed up as 5-30 ms hiccup steps in the arm it was sampling.)  Falls back to nvidia-smi
    when NVML cannot be loaded."""

    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"))

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc, self.thread, self.stop_flag = gpu_index, [], None, None, threading.Event()
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else gpu_index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self._sample()  # the first query initialises driver state: keep it out of the timed region
            self.rows.clear()
        except Exception:
            self.nvml = None

    def _sample(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        self.rows.append((sm, mx, {name for name, const in self.REASONS if mask & getattr(n, const, 0)}))

    def _loop(self):
        while not self.stop_flag.is_set():
            try:
                self._sample()
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        names = [n for n, _ in self.REASONS]
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                self.rows.append((int(float(r[0])), int(float(r[1])),
                                  {n for n, v in zip(names, r[3:7]) if v.lower().startswith("active")}))
            except Exception:
                pass

    def stop(self):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(timeout=1.0)
        if self.proc:
            self.proc.terminate()
        sm = sorted(r[0] for r in self.rows)
        reasons = set()
        for r in self.rows:
            reasons |= r[2]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((r[1] for r in self.rows), default=None),
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


class BatchOpTimer:
    """hooks for examples.impala.LearnerLoop: CUDA events around every Batcher.stack / Batcher.cat in the timed region,
    on the stream the kernels are launched on (torch's current stream)."""

    def __init__(self, torch, kernel_launches):
        self.torch, self.kernel_launches = torch, kernel_launches
        self.enabled = False
        self.records = []  # (op, start_evt, end_evt, payload_bytes, launches)

    @staticmethod
    def payload(item):
        n = 0
        stack = [item]
        while stack:
            x = stack.pop()
            if isinstance(x, dict):
                stack.extend(x.values())
            elif isinstance(x, (list, tuple)):
                stack.extend(x)
            elif hasattr(x, "element_size"):
                n += x.numel() * x.element_size()
        return n

    def batch_op(self, op, fn, item, items_moved=1):
        if not self.enabled:
            fn(item)
            return
        s, e = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        l0 = self.kernel_launches()
        s.record()
        fn(item)
        e.record()
        self.records.append((op, s, e, self.payload(item) * items_moved, self.kernel_launches() - l0))

    def summary(self, hbm_gbs, peak_kind):
        by = {}
        for op, s, e, nbytes, launches in self.records:
            ms = s.elapsed_time(e)
            d = by.setdefault(op, {"ms": 0.0, "payload": 0, "launches": 0, "calls": 0})
            d["ms"] += ms
            d["payload"] += nbytes
            d["launches"] += launches
            d["calls"] += 1
        out = {}
        for op, d in by.items():
            if d["launches"] == 0 or d["ms"] <= 0:
                continue
            alg = 2 * d["payload"]  # read every source byte once + write every destination byte once
            out[op] = {"launches": d["launches"], "avg_launch_us": round(d["ms"] * 1e3 / d["launches"], 3),
                       "total_ms": round(d["ms"], 4), "alg_bytes_per_launch": alg // d["launches"],
                       "alg_bytes_total": alg, "achieved_gbs": round(alg / d["ms"] / 1e6, 1),
                       "frac": round(alg / d["ms"] / 1e6 / hbm_gbs, 4)}
        if out:
            tot_ms = sum(o["total_ms"] for o in out.values())
            tot_b = sum(o["alg_bytes_total"] for o in out.values())
            out["_all"] = {"launches": sum(o["launches"] for o in out.values()), "total_ms": round(tot_ms, 4),
                           "alg_bytes_total": tot_b, "achieved_gbs": round(tot_b / tot_ms / 1e6, 1),
                           "frac": round(tot_b / tot_ms / 1e6 / hbm_gbs, 4)}
        return out


def measured_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(q * len(xs)))] if xs else None


def parity_rounds(acc, model, pump, rank, world, torch, dist):
    """Two CHECKED reductions through the public Accumulator on the real 36-tensor gradient layout, before any timed
    region (reference semantics: src/group.h:570-654 tree sum, src/accumulator.cc:433-452 x 1.0f/numGradients; the
    reference's own check is test/test_reduce.py:66-81).  Round A: rank r contributes r+1 everywhere.  Round B:
    randn(seed=r).  Every rank compares its result bit for bit with the CPU oracle in the kernel's summation order
    (oracle = checker only) and the CRCs of all ranks must agree."""
    import zlib

    import numpy as np

    import oracle

    params = [p for p in model.parameters() if p.requires_grad]
    numels = [p.numel() for p in params]
    offs, total = oracle.flat_layout(numels)
    out = {"n": world, "rounds": [], "exact": True, "tensors": len(params), "floats": int(sum(numels))}

    def inputs_of(kind, q):
        f = np.zeros(total, dtype=np.float32)
        if kind == "rank+1":
            for o, n in zip(offs, numels):
                f[o:o + n] = float(q + 1)
        else:
            g = torch.Generator().manual_seed(7700 + q)
            for o, n in zip(offs, numels):
                f[o:o + n] = torch.randn(n, generator=g).numpy()
        return f

    for kind in ("rank+1", "randn"):
        t0 = time.time()
        while not acc.wants_gradients():
            pump()
            if time.time() - t0 > 120:
                raise RuntimeError(f"rank {rank}: parity round {kind}: accumulator never asked for gradients")
        mine = inputs_of(kind, rank)
        with torch.no_grad():
            for p, o, n in zip(params, offs, numels):
                p.grad.copy_(torch.from_numpy(mine[o:o + n]).view_as(p))  # in place: .grad lives in the NVLink staging
        acc.reduce_gradients(32)
        t0 = time.time()
        while not acc.has_gradients():
            pump()
            if time.time() - t0 > 120:
                raise RuntimeError(f"rank {rank}: parity round {kind}: no result")
        got = np.zeros(total, dtype=np.float32)
        for p, o, n in zip(params, offs, numels):
            got[o:o + n] = p.grad.detach().reshape(-1).cpu().numpy()
        exact, eh = oracle.allreduce_rankorder([inputs_of(kind, q) for q in range(world)], [(1, 0, 32)] * world)
        ok = got.tobytes() == exact.tobytes()
        stats = acc.get_gradient_stats()
        ok = ok and (stats["num_gradients"], stats["num_skipped"], stats["batch_size"]) == tuple(eh[:3])
        crc = zlib.crc32(got.tobytes())
        crcs = [crc]
        if world > 1:
            crcs = [None] * world
            dist.all_gather_object(crcs, crc)
            oks = [None] * world
            dist.all_gather_object(oks, bool(ok))
            ok = all(oks)
        same = len(set(crcs)) == 1
        out["rounds"].append({"input": kind, "bit_exact_vs_oracle_all_ranks": bool(ok), "identical_on_all_ranks": same,
                              "crc32": f"{crcs[0]:08x}", "max_abs": float(np.abs(got).max())})
        out["exact"] = out["exact"] and bool(ok) and same
        acc.zero_gradients()
    return out


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 22  # elements; the parameters (1,094,476) stay whole, the 19M-element observation batch is sampled


def dump_arrays(arm, res, model):
    """What the last timed optimizer step of one arm computed, as float32 / float64 arrays (integers and bools
    converted exactly): every leaf of the learner batch the Batcher delivered for it (`<arm>_batch_<keys>`; a leaf of
    more than DUMP_SAMPLE elements is reduced to the flattened elements at DUMP_SAMPLE sorted indices drawn by
    numpy.random.default_rng(0), the same for every run), its loss, and the model parameters after the step
    (flattened in model.parameters() order).  The synthetic observations, the initial model and the action sampler are
    seeded and the loop runs reproducibly, so a run with the same arguments computes the same; `<arm>_counters` =
    (optimizer steps, actor steps, env frames) shows that two runs took the same path."""
    import numpy as np
    import torch

    def host(t):
        t = t.detach()
        if t.dtype == torch.float64 or (not t.is_floating_point() and t.element_size() > 2):
            t = t.to(torch.float64)
        else:
            t = t.to(torch.float32)
        a = t.cpu().numpy()
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[idx]
        return a

    out = {}

    def walk(name, x):
        if isinstance(x, dict):
            for k, v in x.items():
                walk(f"{name}_{k}", v)
        elif isinstance(x, (list, tuple)):
            for i, v in enumerate(x):
                walk(f"{name}_{i}", v)
        elif isinstance(x, torch.Tensor):
            out[name] = host(x)

    walk(f"{arm}_batch", res.last_batch)
    out[f"{arm}_loss"] = host(res.last_loss)
    out[f"{arm}_params"] = host(torch.cat([p.detach().reshape(-1) for p in model.parameters()]))
    out[f"{arm}_counters"] = np.array([res.optimizer_steps, res.actor_steps, res.env_train_steps], dtype=np.float64)
    return out


def write_dump(directory, arrays):
    import numpy as np

    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def nvlink_roofline(tm, world):
    """K-A2 inside the timed region, from the Accumulator's own CUDA events on its reduce stream."""
    red = [t for t, ok in zip(tm["reduce_us"], tm["reduced"]) if ok]
    gate = [t for t, ok in zip(tm["gate_us"], tm["reduced"]) if ok]
    if not red:
        return None
    S = tm["bytes"]
    avg = sum(red) / len(red)
    two = world > 2 and S >= ((4 << 20) if world <= 4 else (1 << 20))
    busbw = S * 2 * (world - 1) / world / avg / 1e3 if world > 1 else 0.0  # GB/s
    ingress = (S * 2 * (world - 1) / world if two else S * (world - 1)) / avg / 1e3
    return {"kernel": ("ar_twoshot_kernel" if two else "ar_oneshot_kernel") + f"<{world}>", "algo": "twoshot" if two else "oneshot",
            "bytes": S, "rounds": len(red), "avg_us": round(avg, 2), "p50_us": round(_pct(red, 0.5), 2),
            "p90_us": round(_pct(red, 0.9), 2), "gate_wait_p50_us": round(_pct(gate, 0.5), 2),
            "gate_wait_p90_us": round(_pct(gate, 0.9), 2), "busbw_gbs": round(busbw, 1),
            "ingress_gbs": round(ingress, 1), "peak": 770.0, "peak_kind": "B200_PROFILING.md measured peer copy per direction",
            "frac_of_770": round(ingress / 770.0, 4), "short_rounds": tm["short_rounds"],
            "stage_launches": tm["stage_launches"], "zero_copy_rounds": tm["zero_copy_rounds"]}


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank, local, world = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("gloo")
    import moolib_b200 as api
    from moolib_b200 import _C
    from examples import impala

    device = f"cuda:{local}"
    master = os.environ.get("MASTER_ADDR", "127.0.0.1")
    port = int(os.environ.get("MASTER_PORT", 29400)) + 23
    addr = f"{master}:{port}"
    broker = None
    if rank == 0:
        broker = api.Broker()
        broker.listen(addr)

    service = {"fn": lambda: None}

    def barrier():
        # Peers may still need this rank's control plane while it waits (e.g. the elected leader serving the model to
        # a late joiner), so keep servicing it instead of blocking inside gloo.
        if world > 1:
            w = dist.barrier(async_op=True)
            while not w.is_completed():
                service["fn"]()
                time.sleep(0.0002)

    # --dump-outputs runs the loop reproducibly (see Flags.sync_ticks; fixed cuDNN algorithms instead of autotuned ones)
    # so that two runs, or two builds, can be compared output for output; its timings are not the benchmark's
    reproducible = args.dump_outputs is not None
    dump = reproducible and rank == 0
    flags = impala.Flags(actor_batch_size=args.envs, virtual_batch_size=32 * world, device=device, keep_last_batch=dump,
                         sync_ticks=reproducible)
    model, optimizer = impala.make_learner(flags)
    if reproducible:
        torch.backends.cudnn.benchmark = False
        torch.backends.cudnn.deterministic = True
    rpc = api.Rpc()
    rpc.set_name(f"learner{rank}")
    rpc.connect(addr)
    group = api.Group(rpc, "impala")
    group.set_sort_order(rank)
    acc = api.Accumulator("impala", model.parameters(), model.buffers(), group=group)
    acc.set_virtual_batch_size(flags.virtual_batch_size)

    def pump():
        if broker is not None:
            broker.update()
        group.update()
        acc.update()
        if acc.wants_state():
            acc.set_state({"optimizer": optimizer.state_dict()})
        if acc.has_new_state():
            acc.state()

    service["fn"] = pump
    hbm, peak_kind = measured_peaks()
    K, W, S = args.steps, args.warmup, max(0, args.settle)
    results = {}
    dumped = {}
    timer = BatchOpTimer(torch, _C.kernel_launches)

    def wait_for_full_group():
        # all N learners must be members before the clock starts, otherwise early steps run with a smaller group
        t0 = time.time()
        while len(group.members()) != world or not acc.connected():
            pump()
            time.sleep(0.001)
            if time.time() - t0 > 120:
                raise RuntimeError(f"rank {rank}: group did not form: {group.members()}")
        barrier()

    wait_for_full_group()
    parity = parity_rounds(acc, model, pump, rank, world, torch, dist)
    if not parity["exact"]:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "error": "allreduce parity check failed", "parity": parity}), flush=True)
        sys.exit(3)
    barrier()

    def dbg(msg):
        if os.environ.get("BENCH_DEBUG"):
            print(f"[rank {rank}] t={time.time() % 1000:.2f} {msg}", file=sys.stderr, flush=True)

    for mode in ("value", "e2e"):
        flags.host_obs = mode == "e2e"
        flags.read_metrics = mode == "e2e"
        dbg(f"{mode}: creating env pool")
        envs = impala.SyntheticEnvPool(flags, device)
        dbg(f"{mode}: env pool ready")
        state = {"t0": None}
        start_evt, end_evt = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(local) if (rank == 0 and mode == "value") else None

        def on_step(res, mode=mode, state=state, start_evt=start_evt, end_evt=end_evt, sampler=sampler):
            n = res.optimizer_steps
            if os.environ.get("BENCH_DEBUG"):
                print(f"[rank {rank}] {mode} step {n} t={time.time() % 1000:.2f} actor={res.actor_steps}",
                      file=sys.stderr, flush=True)
            if n == S + W:
                torch.cuda.synchronize()
                barrier()
                if sampler:
                    sampler.start()
                state["launch0"] = _C.kernel_launches()
                state["actor0"] = res.actor_steps
                state["frames0"] = res.env_train_steps
                state["stats0"] = (res.t_learn, res.t_act, res.t_opt, res.t_idle, res.n_learn, res.n_skip, res.n_idle)
                timer.enabled = mode == "value"
                acc.reduce_timings(clear=True)
                state["t0"] = time.perf_counter()
                state["step_t"] = [state["t0"]]
                start_evt.record()
                return True
            if state.get("t0") is not None and n < S + W + K:
                state["step_t"].append(time.perf_counter())
            if n == S + W + K:
                end_evt.record()
                dbg(f"{mode}: end recorded, synchronizing")
                torch.cuda.synchronize()
                dbg(f"{mode}: synchronized")
                state["t1"] = time.perf_counter()
                state["step_t"].append(state["t1"])
                state["ar"] = acc.reduce_timings()
                state["launches"] = _C.kernel_launches() - state["launch0"]
                state["actor_steps"] = res.actor_steps - state["actor0"]
                state["frames"] = res.env_train_steps - state["frames0"]
                s0 = state["stats0"]
                s1 = (res.t_learn, res.t_act, res.t_opt, res.t_idle, res.n_learn, res.n_skip, res.n_idle)
                state["loop"] = {k: round(b - a, 4) for k, a, b in zip(
                    ("t_learn_s", "t_act_s", "t_opt_s", "t_idle_s", "n_learn", "n_skip", "n_idle"), s0, s1)}
                timer.enabled = False
                barrier()
                return False
            return True

        res = impala.run_learner(api, flags, acc, model, optimizer, envs, on_step, max_seconds=3600, group=group,
                                 broker=broker, hooks=timer)
        dbg(f"{mode}: loop finished")
        if dump:
            # the loop stopped right after the last timed step: the model still holds its result
            dumped.update(dump_arrays(mode, res, model))
            res.last_batch = None
        ms = start_evt.elapsed_time(end_evt)
        wall = (state["t1"] - state["t0"]) * 1e3
        t = torch.tensor([ms, wall], dtype=torch.float64)
        fr = torch.tensor([float(state["frames"])], dtype=torch.float64)
        slowest = rank
        if world > 1:
            all_ms = [None] * world
            dist.all_gather_object(all_ms, float(ms))
            slowest = max(range(world), key=lambda i: all_ms[i])
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(fr, op=dist.ReduceOp.SUM)
        st = state["step_t"]
        step_ms = [(b - a) * 1e3 for a, b in zip(st, st[1:])]
        # frames = the reference's env_train_steps (examples/vtrace/experiment.py:155): unroll_length * batch_size per
        # gradient batch computed, summed over all learners.  With virtual_batch_size == batch_size * N it equals
        # unroll_length * batch_size * N * optimizer_steps whenever every learner contributes exactly once per round.
        frames = fr[0].item()
        results[mode] = {"ms": t[0].item(), "wall_ms": t[1].item(), "frames": frames,
                         "frames_per_opt_step": frames / max(K, 1), "loop": state["loop"],
                         "value": frames / (t[0].item() / 1e3), "launches": state["launches"],
                         "actor_steps": state["actor_steps"], "loss": float(res.last_loss),
                         "h2d": envs.h2d_bytes, "d2h": envs.d2h_bytes, "ar": state["ar"], "slowest_rank": slowest,
                         "step_ms": {"p50": round(_pct(step_ms, 0.5), 3), "p90": round(_pct(step_ms, 0.9), 3),
                                     "max": round(max(step_ms), 3), "clock": "host wall between optimizer steps, rank 0"}}
        if sampler:
            results["clocks"] = sampler.stop()
        # let the peers drain before the next mode
        for _ in range(50):
            pump()
            time.sleep(0.001)
        dbg(f"{mode}: drained")
        barrier()
        dbg(f"{mode}: barrier passed")

    if rank == 0:
        v, e = results["value"], results["e2e"]
        ops = timer.summary(hbm, peak_kind)
        # the dominant moolib_b200 kernel family = the Batcher op with the most device time inside the timed region
        named = {k: o for k, o in ops.items() if not k.startswith("_")}
        dom_name = max(named, key=lambda k: named[k]["total_ms"]) if named else None
        dom = named.get(dom_name, {})
        # H2D per optimizer step: actor steps per optimizer step x one [B] observation slab; D2H: the grad-norm read
        actor_per_step = e["actor_steps"] / max(K, 1)
        line = {
            "metric": METRIC, "value": round(v["value"], 1), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "settle_steps": S,
            "ms_per_step": round(v["ms"] / K, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "IMPALA vtrace learner loop (examples/impala.py), synthetic 84x84x4 u8 obs, "
                                   f"{args.envs}-env pool x2 buffers, T=21, batch 32/learner, atari ResNet 1,094,476 params"
                                   + (", 1 learner on 1 B200 (BASELINE configs[1])" if world == 1 else
                                      f", {world} learner peers, kernel allreduce over NVLink (BASELINE configs[2])"),
                       "global_batch": 32 * world, "unroll_length": 20, "parallelism": f"dp{world}",
                       "l2": "inputs larger than L2 (152 MB time batches, rotating observation pool)"},
            "e2e": {"value": round(e["value"], 1), "unit": UNIT, "ms_per_step": round(e["ms"] / K, 4),
                    "h2d_bytes_per_step": int(actor_per_step * e["h2d"]), "d2h_bytes_per_step": 4},
            "gpu_launches": int(v["launches"]),
            "roofline": {"bound": "hbm", "kernel": f"Batcher.{dom_name} (dominant moolib_b200 op by device time in the step)",
                         "achieved": dom.get("achieved_gbs"), "peak": hbm, "unit": "GB/s", "frac": dom.get("frac"),
                         # dram__bytes_read.sum + dram__bytes_write.sum of this launch shape from the committed ncu --set full
                         # capture (profiles/r02_ncu_gather_152MB.md: 152.30 MB read = the payload exactly, 101.79 MB written,
                         # the rest of the writes is still in L2 at kernel end); algorithmic = 304.5 MB.  Not re-measured
                         # in this run (a number taken under a profiler is never a bench value).
                         "traffic": 254086656 if (args.envs == 256 and dom_name == "unroll_gather") else None,
                         "traffic_source": "profiles/r02_ncu_gather_152MB.md",
                         "note": "in-loop figure: the gather's sources are the actor's last 21 step outputs (152 MB > L2 in "
                                 "total, the most recent ones may still be L2-resident, hence a fraction that can read "
                                 "slightly above 1); isolated and L2-flushed the same launch runs at 0.82 of the measured "
                                 "peak (profiles/r02_sweep_batch_stack_1gpu.jsonl)",
                         "peak_kind": peak_kind, "per_op": ops, "aggregate_frac": ops.get("_all", {}).get("frac")},
            "roofline_nvlink": nvlink_roofline(v["ar"], world),
            "parity": parity,
            "step_ms": {"value": v["step_ms"], "e2e": e["step_ms"]},
            "slowest_rank": {"value": v["slowest_rank"], "e2e": e["slowest_rank"]},
            "clocks": results.get("clocks"),
            "wall_ms_per_step": round(v["wall_ms"] / K, 4),
            "frames_per_opt_step": {"value": v["frames_per_opt_step"], "e2e": e["frames_per_opt_step"],
                                    "nominal": 640 * world},
            "optimizer_steps_per_s": {"value": round(K / (v["ms"] / 1e3), 2), "e2e": round(K / (e["ms"] / 1e3), 2)},
            "loop_stats_rank0": {"value": v["loop"], "e2e": e["loop"]},
        }
        if reproducible:
            line["reproducible_mode"] = "--dump-outputs: device synchronised every loop iteration, fixed cuDNN algorithms"
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_leg(args)
            if args.ref_cuda:
                line["reference_cuda_model"] = reference_cuda_leg(args)
        if dump:
            write_dump(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    barrier()
    if world > 1:
        dist.destroy_process_group()


def _run_child(extra_env, argv, timeout):
    env = dict(os.environ)
    env.update(extra_env)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, env=env, capture_output=True,
                           text=True, timeout=timeout)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": (r.stderr or r.stdout)[-400:]}
    except Exception as ex:  # noqa: BLE001
        return {"error": repr(ex)[:400]}


def cpu_baseline_leg(args):
    """The reference's own CPU path (oracle/_ref) on this box's host cores, bounded sample of the same workload."""
    out = _run_child({}, ["--impl", "reference", "--gpus", "1", "--steps", "8", "--warmup", "3", "--max-seconds", "100"],
                     timeout=400)
    if "cpu_baseline" in out:
        return out["cpu_baseline"]
    return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": "failed",
            "error": out.get("error") or out.get("unavailable") or str(out)[:300]}


def reference_cuda_leg(args):
    """Information only: the reference compiled with -DUSE_CUDA (oracle/_ref_cuda) driving the SAME loop with the model
    on the GPU -- what a moolib user has today (its Batcher issues per-leaf copy_, its Accumulator stages gradients
    through pinned host memory and reduces on the CPU)."""
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref_cuda", "moolib")):
        return {"unavailable": "oracle/_ref_cuda not built"}
    out = _run_child({"MB_REF_CUDA": "1"}, ["--impl", "reference", "--gpus", "1", "--steps", str(min(args.steps, 40)),
                                            "--warmup", str(min(args.warmup, 8)), "--max-seconds", "60"], timeout=300)
    return {k: out.get(k) for k in ("value", "unit", "ms_per_step", "frames_per_opt_step", "optimizer_steps_per_s",
                                    "steps", "error", "unavailable") if k in out}


def run_reference(args):
    rank, local, world = dist_env()
    use_cuda = os.environ.get("MB_REF_CUDA") == "1"
    if rank != 0 and not use_cuda:
        return
    ref_dir = os.path.join(ROOT, "oracle", "_ref_cuda" if use_cuda else "_ref")
    import torch
    sys.path.insert(0, ref_dir)
    try:
        import moolib as ref
    except Exception as ex:  # the oracle always exists in this repo; say so loudly if the build is missing
        print(json.dumps({"impl": "reference", "unavailable": f"oracle/_ref not built: {ex!r}"[:200]}))
        return
    from examples import impala

    # MB_REF_CUDA=1 (information only, not the driver's reference arm): the reference compiled with -DUSE_CUDA, one
    # process per GPU under torchrun exactly like our arm, models on the GPUs, ITS OWN RPC transport between the processes.
    multi = use_cuda and world > 1
    if multi:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("gloo")
    n_peers = 1 if use_cuda else max(world, args.gpus)
    device = f"cuda:{local}" if use_cuda else "cpu"
    cores = os.cpu_count()
    # ATen's CPU kernels stop scaling (and start thrashing) far below the core count of a 128-core host for these
    # small convolutions; the reference's own scheduler also takes min(cores-1, 64) threads (src/async.cc:67-83)
    threads = max(1, min(cores, 32) // max(n_peers, world if multi else 1))
    torch.set_num_threads(threads)
    K, W = args.steps, args.warmup
    if n_peers > 1:
        # N CPU peers share this one process: a step costs N forward/backward passes on the host cores.  Keep the sample
        # bounded: one warm-up step, then as many of the K steps as fit into --max-seconds.
        W = min(W, 1)
    if multi:
        port = int(os.environ.get("MASTER_PORT", 29400)) + 41
    else:
        port = 29400 + 57 + (os.getpid() % 500)
    addr = f"127.0.0.1:{port}"
    broker = None
    if rank == 0:
        broker = ref.Broker()
        broker.listen(addr)
    total_peers = world if multi else n_peers
    loops = []
    # N reference peers share ONE host process in the CPU arm (rank 0 only runs it): bound the sample by shrinking the
    # actor pool per peer -- the learner batch (T=21 x 32) and the reduction (N peers, 4.38 MB) are the full-size ones.
    envs_per_peer = args.envs if (n_peers == 1) else max(32, args.envs // n_peers)
    for i in range(n_peers):
        flags = impala.Flags(actor_batch_size=envs_per_peer, virtual_batch_size=32 * total_peers, device=device,
                             host_obs=True, read_metrics=True)
        flags.seed += i + rank
        model, opt = impala.make_learner(flags)
        acc = ref.Accumulator("impala", model.parameters(), model.buffers())
        acc.set_virtual_batch_size(flags.virtual_batch_size)
        acc.connect(addr)
        envs = impala.SyntheticEnvPool(flags, device)
        loops.append(impala.LearnerLoop(ref, flags, acc, model, opt, envs, broker=broker if i == 0 else None))

    def sync():
        if use_cuda:
            torch.cuda.synchronize()

    t_begin = time.time()
    t0 = None
    done_steps = 0
    while True:
        for lp in loops:
            lp.tick()
        n = min(lp.res.optimizer_steps for lp in loops)
        if t0 is None and n >= W:
            sync()
            t0 = time.perf_counter()
            base = [lp.res.optimizer_steps for lp in loops]
            base_frames = [lp.res.env_train_steps for lp in loops]
        if t0 is not None:
            done_steps = min(lp.res.optimizer_steps - b for lp, b in zip(loops, base))
            if done_steps >= K or time.time() - t_begin > args.max_seconds:
                break
        elif time.time() - t_begin > args.max_seconds:
            break
    sync()
    if t0 is None or sum(lp.res.env_train_steps - b for lp, b in zip(loops, base_frames)) == 0:
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "no gradient batch completed within --max-seconds"}))
        os._exit(0)
    dt = time.perf_counter() - t0
    total_steps = sum(lp.res.optimizer_steps - b for lp, b in zip(loops, base))
    frames = sum(lp.res.env_train_steps - b for lp, b in zip(loops, base_frames))  # experiment.py:155
    if multi:
        t = torch.tensor([float(frames), float(total_steps), dt], dtype=torch.float64)
        tmax = t.clone()
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        frames, total_steps, dt = t[0].item(), t[1].item(), tmax[2].item()
        # keep serving the peers until everybody has its numbers
        w = dist.barrier(async_op=True)
        while not w.is_completed():
            for lp in loops:
                lp.tick()
    value = frames / dt
    sample = (f"{done_steps} of {K} optimizer steps per peer x {total_peers} peer(s)"
              f"{' (one process per GPU)' if multi else ' in one process'}, device={device}, "
              f"{envs_per_peer} envs per peer, T=21, batch 32 per peer, {dt:.1f} s")
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": args.gpus,
            "steps": done_steps, "warmup": W, "ms_per_step": round(dt * 1e3 / max(done_steps, 1), 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "IMPALA vtrace learner loop (examples/impala.py) driven through the UNMODIFIED "
                                   f"reference moolib ({'oracle/_ref_cuda, models on the GPUs' if use_cuda else 'oracle/_ref, host cores'})",
                       "global_batch": 32 * total_peers, "parallelism": f"dp{total_peers}"},
            "frames_per_opt_step": round(frames / max(total_steps / total_peers, 1), 1),
            "optimizer_steps_per_s": round(total_steps / total_peers / dt, 3),
            "cpu_baseline": {"value": round(value, 1), "unit": UNIT, "cores": cores, "kind": "reference",
                             "sample": sample, "aten_threads_per_peer": threads},
            "e2e": {"value": round(value, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if rank == 0:
        print(json.dumps(line), flush=True)
    os._exit(0)  # the reference's RPC threads do not always join cleanly at interpreter exit


def main():
    args = parse_args()
    if os.environ.get("BENCH_DEBUG"):
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["BENCH_DEBUG"]), repeat=False, file=sys.stderr)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
