"""Generates tests/golden/lowp_golden.npz: the UNMODIFIED reference (oracle/_ref, built by oracle/build_ref.sh) reducing
bfloat16 and float16 tensors, in this container.

    python tests/golden/make_golden_lowp.py

* group.all_reduce of bf16 and fp16 tensors at N = 2, 3, 4, 8 peers, sizes that end in partial 16 B vectors;
* Accumulator rounds on nn.Linear(32, 31).to(bfloat16) at N = 2 and 4: plain, local accumulation (peer 0 contributes
  twice), a skipping peer, and a single-contributor round.

Inputs are the float32 draws of make_golden.gen_input (PCG64 seeds) rounded to the dtype by torch; outputs are stored
verbatim as uint16 bit patterns.
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import Peers, gen_input, moolib  # noqa: E402

DT = {"bf16": torch.bfloat16, "f16": torch.float16}


def lowp_input(seed, shape, dt):
    return torch.from_numpy(gen_input(seed, shape, "f32")).to(DT[dt])


def bits(t):
    return t.contiguous().view(torch.int16).numpy().view(np.uint16).copy()


def make_allreduce(out, meta):
    port = 4800
    for n in (2, 3, 4, 8):
        peers = Peers(n, port, group_name="lowp")
        port += 1
        for dt in ("bf16", "f16"):
            for numel in (7, 1001, 4097):
                seed = 20000 + 1000 * n + numel + (500000 if dt == "f16" else 0)
                name = f"ar_{dt}_{numel}"
                ins = [lowp_input(seed * 16 + r, [numel], dt) for r in range(n)]
                futs = [peers.groups[r].all_reduce(name, ins[r].clone()) for r in range(n)]
                res = [f.result(30) for f in futs]
                assert all(x.dtype == DT[dt] for x in res)
                assert all(torch.equal(bits_t, res[0]) for bits_t in res), "reference peers disagree"
                out[f"ar_n{n}_{dt}_{numel}"] = bits(res[0])
                meta.append(repr(("allreduce", n, dt, numel, seed)))
                peers.pump()
        del peers


def make_accumulator(out, meta):
    port = 4900
    for n in (2, 4):
        addr = f"127.0.0.1:{port}"
        port += 1
        broker = moolib.Broker()
        broker.listen(addr)
        models, accs, rpcs, groups = [], [], [], []
        torch.manual_seed(0)
        for i in range(n):
            m = torch.nn.Linear(32, 31).to(torch.bfloat16)
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
            for c in range(max(len(p) for p in plan)):
                for i, a in enumerate(accs):
                    t1 = time.time()
                    while not a.wants_gradients():
                        pump()
                        assert time.time() - t1 < 60
                    if c < len(plan[i]):
                        models[i].weight.grad = lowp_input(plan[i][c], [31, 32], "bf16")
                        models[i].bias.grad = lowp_input(plan[i][c] + 1, [31], "bf16")
                        a.reduce_gradients(10)
                    else:
                        a.skip_gradients()
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
            assert w0.dtype == torch.bfloat16
            for i in range(1, n):
                assert torch.equal(models[i].weight.grad, w0) and torch.equal(models[i].bias.grad, b0)
            out[f"acc_{tag}_w"] = bits(w0)
            out[f"acc_{tag}_b"] = bits(b0)
            meta.append(repr(("accumulator", tag, n, plan, vbs, stats["num_gradients"], stats["num_skipped"],
                              stats["batch_size"])))
            for a in accs:
                a.zero_gradients()
            pump()

        run_round(f"n{n}_plain", [[1100 + 10 * i] for i in range(n)], 10 * n)
        run_round(f"n{n}_accum", [[1500, 1502]] + [[1510 + 10 * i] for i in range(1, n)], 10 * (n + 1))
        run_round(f"n{n}_skip", [[1700 + 10 * i] for i in range(n - 1)] + [[]], 10 * (n - 1))
        run_round(f"n{n}_single", [[1900]] + [[] for _ in range(1, n)], 10)
        assert groups[0].members() == [f"peer{i}" for i in range(n)], groups[0].members()
        del accs, models, groups, rpcs, broker


if __name__ == "__main__":
    out, meta = {}, []
    make_allreduce(out, meta)
    make_accumulator(out, meta)
    np.savez_compressed(os.path.join(HERE, "lowp_golden.npz"), meta=np.array(meta), **out)
    print("lowp:", len(meta), "cases")
    for m in meta:
        print("  ", m)
