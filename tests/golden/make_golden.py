"""Generates the golden fixtures in tests/golden/ by running the UNMODIFIED reference (oracle/_ref, built by
oracle/build_ref.sh from /root/reference) in this container.  The fixtures travel to the GPU box; the reference
source tree does not.

    python tests/golden/make_golden.py            # writes batcher_golden.npz, allreduce_golden.npz, accumulator_golden.npz

Inputs are regenerated from the stored seeds with numpy's PCG64 (stable across versions); outputs are stored verbatim,
except the batches of the random Batcher trials (batcher_random_golden.npz), which are stored as digests.
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402

moolib = oracle.load_reference()

DTYPES = {"u8": np.uint8, "f32": np.float32, "i64": np.int64, "bool": np.bool_}


def gen_input(seed, shape, dt):
    rng = np.random.Generator(np.random.PCG64(seed))
    if dt == "u8":
        return rng.integers(0, 256, size=shape, dtype=np.uint8)
    if dt == "i64":
        return rng.integers(-2**40, 2**40, size=shape, dtype=np.int64)
    if dt == "bool":
        return rng.integers(0, 2, size=shape).astype(np.bool_)
    return rng.standard_normal(size=shape).astype(np.float32)


def batcher_trials():
    """(mode, size, dim, shape, dtype, n_items, seed)"""
    rng = np.random.Generator(np.random.PCG64(20260921))
    trials = []
    for i in range(40):
        mode = "stack" if i % 2 == 0 else "cat"
        size = int(rng.integers(1, 12))
        dim = int(rng.integers(0, 3))
        nd = int(rng.integers(dim + 1, dim + 3))
        shape = [int(rng.integers(1, 6)) for _ in range(nd)]
        dt = ["u8", "f32", "i64", "bool"][i % 4]
        n = int(rng.integers(size, 3 * size + 4))
        trials.append((mode, size, dim, shape, dt, n, 1000 + i))
    # the IMPALA shapes, scaled down in batch: state rows of 84*84*4 u8, time-stack then cat to a narrower batch
    trials.append(("stack", 3, 0, [2, 4, 84, 84], "u8", 7, 5000))
    trials.append(("cat", 3, 1, [2, 4, 4, 84, 84], "u8", 2, 5001))
    trials.append(("cat", 4, 1, [5, 6], "f32", 5, 5002))
    trials.append(("cat", 7, 0, [3, 17], "u8", 9, 5003))   # odd byte counts: unaligned rows
    return trials


def make_batcher():
    out = {}
    trials = batcher_trials()
    for ti, (mode, size, dim, shape, dt, n, seed) in enumerate(trials):
        b = moolib.Batcher(size=size, dim=dim)
        k = 0
        for j in range(n):
            x = torch.from_numpy(gen_input(seed * 100 + j, shape, dt))
            getattr(b, mode)(x)
            while not b.empty():
                out[f"t{ti}_b{k}"] = b.get().numpy().copy()
                k += 1
        out[f"t{ti}_nb"] = np.array(k)
    # one nested case: dict with tuple/list/non-tensor leaves, stack then cat (moolib.cc:619-691 prepareForBatchCopy)
    b = moolib.Batcher(size=3, dim=0)
    for j in range(3):
        item = {
            "a": torch.from_numpy(gen_input(7000 + j, [2, 3], "f32")),
            "n": (torch.from_numpy(gen_input(7100 + j, [4], "u8")), [torch.from_numpy(gen_input(7200 + j, [1], "i64"))]),
            "tag": "first" if j == 0 else "later",
        }
        b.stack(item)
    r = b.get()
    out["nested_a"] = r["a"].numpy().copy()
    out["nested_n0"] = r["n"][0].numpy().copy()
    out["nested_n1"] = r["n"][1][0].numpy().copy()
    out["nested_tag"] = np.array(r["tag"])
    meta = np.array([repr(t) for t in trials])
    np.savez_compressed(os.path.join(HERE, "batcher_golden.npz"), trials=meta, **out)
    print("batcher:", len(trials), "trials,", len(out), "arrays")


def batcher_random_trials():
    """(size, dim, shape, n_items) drawn the way the reference's test/unit/test_batcher.py:13-52 draws them."""
    import random
    rnd = random.Random(1234)
    trials = []
    for _ in range(64):
        size, dim = rnd.randint(1, 20), rnd.randint(0, 2)
        dims = rnd.randint(dim + 1, dim + 2)
        n = rnd.randint(20, 60)
        shape = [rnd.randint(1, 4) for _ in range(dims)]
        trials.append((size, dim, shape, n))
    return trials


def make_batcher_random():
    """Every random trial in both modes: how many batches the reference emits after each item, and a digest of every
    batch (tests/helpers.digest; the batches themselves would be ~400 KB of random floats)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import batcher_random_seed, digest
    out = {}
    trials = batcher_random_trials()
    for ti, (size, dim, shape, n) in enumerate(trials):
        for mode in ("stack", "cat"):
            b = moolib.Batcher(size=size, dim=dim)
            emitted, digests = [], []
            for j in range(n):
                getattr(b, mode)(torch.from_numpy(gen_input(batcher_random_seed(ti, mode, j), shape, "f32")))
                k = 0
                while not b.empty():
                    digests.append(digest(b.get().numpy()))
                    k += 1
                emitted.append(k)
            out[f"r{ti}_{mode}_emitted"] = np.array(emitted, dtype=np.int32)
            out[f"r{ti}_{mode}_digests"] = np.array(digests, dtype="<u8")
    np.savez_compressed(os.path.join(HERE, "batcher_random_golden.npz"),
                        trials=np.array([repr(t) for t in trials]), **out)
    print("batcher_random:", len(trials), "trials x 2 modes")


class Peers:
    """N reference Rpc peers + a Broker in this process on loopback (the layout of test/test_reduce.py:97-104)."""

    def __init__(self, n, port, group_name="g"):
        self.addr = f"127.0.0.1:{port}"
        self.broker_rpc = moolib.Rpc()
        self.broker_rpc.set_name("broker")
        self.broker = moolib.Broker(self.broker_rpc)
        self.broker_rpc.listen(self.addr)
        self.rpcs, self.groups = [], []
        for i in range(n):
            r = moolib.Rpc()
            r.set_name(f"peer{i}")
            r.set_timeout(30)
            r.connect(self.addr)
            g = moolib.Group(r, group_name)
            g.set_timeout(30)
            g.set_sort_order(i)
            self.rpcs.append(r)
            self.groups.append(g)
        t0 = time.time()
        while True:
            self.pump()
            if all(g.active() and len(g.members()) == n for g in self.groups):
                # stable membership for a little while
                ids = {g.sync_id() for g in self.groups}
                if len(ids) == 1:
                    break
            if time.time() - t0 > 60:
                raise RuntimeError("group did not form")
            time.sleep(0.02)
        assert self.groups[0].members() == [f"peer{i}" for i in range(n)], self.groups[0].members()

    def pump(self):
        self.broker.update()
        for g in self.groups:
            g.update()


def make_allreduce():
    out = {}
    port = 4500
    cases = []
    for n in (2, 3, 4, 5, 8):
        peers = Peers(n, port)
        port += 1
        for rep in range(3):
            seed = 9000 + n * 10 + rep
            numel = [4096, 1000, 7][rep]
            ins = [torch.from_numpy(gen_input(seed * 16 + r, [numel], "f32")) for r in range(n)]
            futs = [peers.groups[r].all_reduce(f"ar{rep}", ins[r].clone()) for r in range(n)]
            res = [f.result(30) for f in futs]
            for r in range(1, n):
                assert torch.equal(res[0], res[r]), "reference peers disagree"
            out[f"n{n}_r{rep}"] = res[0].numpy().copy()
            cases.append((n, rep, seed, numel))
            peers.pump()
        del peers
    np.savez_compressed(os.path.join(HERE, "allreduce_golden.npz"), cases=np.array(cases), **out)
    print("allreduce:", len(cases), "cases")


def make_allreduce_2049():
    """group.all_reduce of 4 peers on 3 rounds of 2049 floats drawn from default_rng(2026) (odd: vectorised loops end
    in a partial tail)."""
    n, numel = 4, 2049
    peers = Peers(n, 4700, group_name="live")
    rng = np.random.default_rng(2026)
    out = {}
    for rep in range(3):
        ins = [rng.standard_normal(numel).astype(np.float32) for _ in range(n)]
        futs = [peers.groups[r].all_reduce(f"live{rep}", torch.from_numpy(ins[r].copy())) for r in range(n)]
        res = [f.result(30).numpy() for f in futs]
        assert all(r.tobytes() == res[0].tobytes() for r in res), "reference peers disagree"
        out[f"rep{rep}"] = res[0].copy()
        peers.pump()
    np.savez_compressed(os.path.join(HERE, "allreduce_2049_golden.npz"), n=np.array(n), numel=np.array(numel), **out)
    print("allreduce_2049: 3 rounds")


def make_accumulator():
    """Controlled Accumulator rounds on nn.Linear(32, 31) (BASELINE.json configs[0]); every round records each peer's
    contributions, the reduced stats and the averaged gradients all peers end up with."""
    out = {}
    rounds_meta = []
    port = 4600
    for n in (2, 4):
        addr = f"127.0.0.1:{port}"
        port += 1
        broker = moolib.Broker()
        broker.listen(addr)
        models, accs, rpcs, groups = [], [], [], []
        torch.manual_seed(0)
        for i in range(n):
            m = torch.nn.Linear(32, 31)
            # explicit Rpc + Group so that the member index of peer i is i (sort order, src/broker.h:168-173)
            r = moolib.Rpc()
            r.set_name(f"peer{i}")
            r.connect(addr)
            grp = moolib.Group(r, "acc")
            grp.set_sort_order(i)
            a = moolib.Accumulator("acc", m.parameters(), m.buffers(), group=grp)
            a.set_virtual_batch_size(10 * n)
            models.append(m)
            accs.append(a)
            rpcs.append(r)
            groups.append(grp)

        def pump():
            broker.update()
            for grp in groups:
                grp.update()
            for a in accs:
                a.update()

        t0 = time.time()
        while not all(a.connected() for a in accs):
            pump()
            for a in accs:
                if a.wants_state():
                    a.set_state({"x": 1})
                if a.has_new_state():
                    a.state()
            time.sleep(0.01)
            assert time.time() - t0 < 120, "accumulators did not connect"

        def run_round(tag, plan, vbs):
            """plan[i] = list of seeds: peer i contributes len(plan[i]) gradients (0 = skip only)."""
            for a in accs:
                a.set_virtual_batch_size(vbs)
            t0 = time.time()
            while not all(a.wants_gradients() for a in accs):
                pump()
                assert time.time() - t0 < 60
            maxc = max(len(p) for p in plan)
            for c in range(maxc):
                for i, a in enumerate(accs):
                    # every peer takes part in every count round: contribute if it has one left, else skip
                    t1 = time.time()
                    while not a.wants_gradients():
                        pump()
                        assert time.time() - t1 < 60
                    if c < len(plan[i]):
                        gw = gen_input(plan[i][c], [31, 32], "f32")
                        gb = gen_input(plan[i][c] + 1, [31], "f32")
                        models[i].weight.grad = torch.from_numpy(gw.copy())
                        models[i].bias.grad = torch.from_numpy(gb.copy())
                        a.reduce_gradients(10)
                    else:
                        a.skip_gradients()
                # let the count round finish before the next contribution
                for _ in range(20):
                    pump()
                    time.sleep(0.002)
            t0 = time.time()
            while not all(a.has_gradients() for a in accs):
                pump()
                time.sleep(0.001)
                assert time.time() - t0 < 60, "no gradients"
            stats = accs[0].get_gradient_stats()
            w0, b0 = models[0].weight.grad.clone(), models[0].bias.grad.clone()
            for i in range(1, n):
                assert torch.equal(models[i].weight.grad, w0) and torch.equal(models[i].bias.grad, b0)
                assert accs[i].get_gradient_stats() == stats
            out[f"{tag}_w"] = w0.numpy().copy()
            out[f"{tag}_b"] = b0.numpy().copy()
            rounds_meta.append(repr((tag, n, plan, vbs, stats["num_gradients"], stats["num_skipped"],
                                     stats["batch_size"])))
            for a in accs:
                a.zero_gradients()
            pump()

        run_round(f"n{n}_plain", [[100 + 10 * i] for i in range(n)], 10 * n)
        run_round(f"n{n}_plain2", [[300 + 10 * i] for i in range(n)], 10 * n)
        # peer 0 contributes twice (local accumulation, accumulator.cc:959-975), the others once
        run_round(f"n{n}_accum", [[500, 502]] + [[510 + 10 * i] for i in range(1, n)], 10 * (n + 1))
        # the last peer never has a gradient: it only skips (group.h:206-208 empty-gradient adoption)
        run_round(f"n{n}_skip", [[700 + 10 * i] for i in range(n - 1)] + [[]], 10 * (n - 1))
        assert groups[0].members() == [f"peer{i}" for i in range(n)], groups[0].members()
        del accs, models, groups, rpcs, broker
    np.savez_compressed(os.path.join(HERE, "accumulator_golden.npz"), rounds=np.array(rounds_meta), **out)
    print("accumulator:", len(rounds_meta), "rounds")
    for r in rounds_meta:
        print("  ", r)


def make_envpool():
    """Reference EnvPool (forked workers + POSIX shm) stepping tests/envs_for_tests.FrameEnv with seeded actions."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from envs_for_tests import FrameEnv
    bs, steps = 6, 24
    envs = moolib.EnvPool(FrameEnv, num_processes=3, batch_size=bs, num_batches=2)
    rng = np.random.Generator(np.random.PCG64(77))
    out = {"bs": np.array(bs), "steps": np.array(steps)}
    for t in range(steps):
        action = torch.from_numpy(rng.integers(0, 18, size=bs, dtype=np.int64))
        obs = envs.step(t % 2, action).result()
        out[f"state{t}"] = obs["state"].numpy().copy()
        out[f"reward{t}"] = obs["reward"].numpy().copy()
        out[f"done{t}"] = obs["done"].numpy().copy()
    np.savez_compressed(os.path.join(HERE, "envpool_golden.npz"), **out)
    print("envpool:", steps, "steps of", bs, "envs")


def make_vtrace():
    """The reference's own V-trace (examples/common/vtrace.py, pure PyTorch, imported from the reference tree) and its
    observation normalisation `x.float() / 255.0` (examples/atari/models.py:94) on seeded inputs."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_vtrace", "/root/reference/examples/common/vtrace.py")
    ref_vtrace = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_vtrace)
    out, cases = {}, []
    for ci, (T, B, clip, clip_pg) in enumerate([(20, 32, 1.0, 1.0), (5, 7, 1.0, 1.0), (1, 3, 1.0, 1.0), (20, 64, 0.8, 2.0),
                                                (11, 130, None, None)]):
        lr = gen_input(8000 + 10 * ci, [T, B], "f32") * 0.5
        disc = (gen_input(8001 + 10 * ci, [T, B], "bool") | gen_input(8002 + 10 * ci, [T, B], "bool")).astype(np.float32) * 0.99
        rew = gen_input(8003 + 10 * ci, [T, B], "f32")
        val = gen_input(8004 + 10 * ci, [T, B], "f32")
        boot = gen_input(8005 + 10 * ci, [B], "f32")
        r = ref_vtrace.from_importance_weights(torch.from_numpy(lr), torch.from_numpy(disc), torch.from_numpy(rew),
                                               torch.from_numpy(val), torch.from_numpy(boot), clip, clip_pg)
        out[f"c{ci}_vs"] = r.vs.numpy().copy()
        out[f"c{ci}_pg"] = r.pg_advantages.numpy().copy()
        cases.append(repr((T, B, clip, clip_pg)))
    x = gen_input(8900, [3, 5, 4, 8, 8], "u8")
    out["norm_in_seed"] = np.array(8900)
    out["norm_out"] = (torch.from_numpy(x).float() / 255.0).numpy().copy()
    np.savez_compressed(os.path.join(HERE, "vtrace_golden.npz"), cases=np.array(cases), **out)
    print("vtrace:", len(cases), "cases")


if __name__ == "__main__":
    which = sys.argv[1:] or ["batcher", "batcher_random", "allreduce", "allreduce_2049", "accumulator", "envpool",
                             "vtrace"]
    if "vtrace" in which:
        make_vtrace()
    if "batcher" in which:
        make_batcher()
    if "batcher_random" in which:
        make_batcher_random()
    if "allreduce" in which:
        make_allreduce()
    if "allreduce_2049" in which:
        make_allreduce_2049()
    if "accumulator" in which:
        make_accumulator()
    if "envpool" in which:
        make_envpool()
