"""Pins the CPU oracle (oracle/) to the reference: against the golden fixtures generated from the unmodified
reference (tests/golden/make_golden.py)."""
import ast

import numpy as np
import torch

import oracle
from helpers import batcher_random_seed, batcher_trials, digest, gen_input, tree_masks


def _replay_batcher(make, trial):
    mode, size, dim, shape, dt, n, seed = trial
    b = make(size, dim)
    outs = []
    for j in range(n):
        x = torch.from_numpy(gen_input(seed * 100 + j, shape, dt))
        getattr(b, mode)(x)
        while not b.empty():
            outs.append(b.get())
    return outs


def test_oracle_batcher_matches_golden(golden_dir):
    g = np.load(f"{golden_dir}/batcher_golden.npz")
    for ti, trial in enumerate(batcher_trials(g)):
        outs = _replay_batcher(lambda size, dim: oracle.OracleBatcher(size, dim=dim), trial)
        assert len(outs) == int(g[f"t{ti}_nb"]), trial
        for k, o in enumerate(outs):
            ref = g[f"t{ti}_b{k}"]
            assert o.numpy().dtype == ref.dtype and o.numpy().shape == ref.shape
            assert o.numpy().tobytes() == ref.tobytes(), (trial, k)


def test_oracle_c_stack_and_cat_match_golden(golden_dir):
    """The C byte-movement functions (oracle_stack_slot / oracle_cat_narrow) replay the same trials."""
    g = np.load(f"{golden_dir}/batcher_golden.npz")
    for ti, (mode, size, dim, shape, dt, n, seed) in enumerate(batcher_trials(g)):
        nb = int(g[f"t{ti}_nb"])
        items = [gen_input(seed * 100 + j, shape, dt) for j in range(n)]
        if mode == "stack":
            for k in range(nb):
                bshape = shape[:dim] + [size] + shape[dim:]
                dst = np.zeros(bshape, dtype=items[0].dtype)
                for s in range(size):
                    oracle.stack_slot(dst, s, np.ascontiguousarray(items[k * size + s]), dim)
                assert dst.tobytes() == g[f"t{ti}_b{k}"].tobytes()
        else:
            # cat with carry (src/moolib.cc:767-811)
            bshape = list(shape)
            bshape[dim] = size
            dst = np.zeros(bshape, dtype=items[0].dtype)
            fill, k = 0, 0
            for it in items:
                off, m = 0, it.shape[dim]
                while off < m:
                    take = min(m - off, size - fill)
                    oracle.cat_narrow(dst, fill, np.ascontiguousarray(it), off, take, dim)
                    fill += take
                    off += take
                    if fill == size:
                        assert dst.tobytes() == g[f"t{ti}_b{k}"].tobytes(), (ti, k)
                        k += 1
                        fill = 0
                        dst = np.zeros(bshape, dtype=items[0].dtype)
            assert k == nb


def test_oracle_tree_allreduce_matches_golden(golden_dir):
    """group.all_reduce of the reference = oracle tree sum for one of the legal arrival orders, bit for bit."""
    g = np.load(f"{golden_dir}/allreduce_golden.npz")
    for n, rep, seed, numel in g["cases"]:
        ins = [gen_input(int(seed) * 16 + r, [int(numel)], "f32") for r in range(n)]
        ref = g[f"n{n}_r{rep}"]
        hdrs = [(1, 0, 1)] * n
        hit = False
        for mask in tree_masks(int(n)):
            out, _ = oracle.allreduce_tree(ins, hdrs, order=mask, scale=False)
            if out.tobytes() == ref.tobytes():
                hit = True
                break
        assert hit, f"no arrival order reproduces the reference for n={n} rep={rep}"
        # and the product's rank order stays inside the stated tolerance of the reference
        ours, _ = oracle.allreduce_rankorder(ins, hdrs, scale=False)
        assert (np.abs(ours.astype(np.float64) - ref) <= oracle.allreduce_tolerance(ins, ref)).all()


def _acc_round_inputs(n, plan):
    """Per-peer staged gradient (weight[31,32] ++ bias[31] in the flat layout) and header."""
    ins, hdrs = [], []
    numels = [31 * 32, 31]
    offs, total = oracle.flat_layout(numels)
    for i in range(n):
        if not plan[i]:
            ins.append(None)
            hdrs.append((0, 1, 0))
            continue
        staging = np.zeros(total, dtype=np.float32)
        for c, seed in enumerate(plan[i]):
            gw = gen_input(seed, [31, 32], "f32").reshape(-1).copy()
            gb = gen_input(seed + 1, [31], "f32").copy()
            oracle.stage(staging, [gw, gb], accumulate=c > 0, zero_src=True)
            assert not gw.any() and not gb.any()
        ins.append(staging)
        # every count round a peer takes part in without a gradient of its own is a skip
        hdrs.append((len(plan[i]), 0, 10 * len(plan[i])))
    return ins, hdrs, offs, numels


def test_oracle_accumulator_rounds_match_golden(golden_dir):
    g = np.load(f"{golden_dir}/accumulator_golden.npz")
    for r in g["rounds"]:
        tag, n, plan, vbs, ngrad, nskip, bsz = ast.literal_eval(str(r))
        ins, hdrs, offs, numels = _acc_round_inputs(n, plan)
        # skips: peers with fewer contributions than the longest plan skipped the extra count rounds
        maxc = max(len(p) for p in plan)
        hdrs = [(h[0], maxc - len(plan[i]), h[2]) for i, h in enumerate(hdrs)]
        ref = np.concatenate([g[f"{tag}_w"].reshape(-1), g[f"{tag}_b"].reshape(-1)])
        hit = False
        for mask in tree_masks(n):
            out, oh = oracle.allreduce_tree(ins, hdrs, order=mask, scale=True)
            flat = np.concatenate([out[offs[0]:offs[0] + numels[0]], out[offs[1]:offs[1] + numels[1]]])
            assert oh[:3] == (ngrad, nskip, bsz), (tag, oh)
            if flat.tobytes() == ref.tobytes():
                hit = True
                break
        assert hit, tag


def test_fill_batch_and_scatter_actions():
    slab = np.zeros((8, 4, 4), dtype=np.float32)
    rows = [gen_input(40 + i, [4, 4], "f32") for i in range(8)]
    for i in (3, 0, 7, 1, 2, 6, 5, 4):
        oracle.fill_batch(slab, i, rows[i])
    assert slab.tobytes() == np.stack(rows).tobytes()
    counters = np.array([0, 5, 0xFFFFFFFF, 7], dtype=np.uint32)
    acts = np.array([3, 0, 1, 17], dtype=np.int64)
    oracle.scatter_actions(counters, acts)
    assert counters.tolist() == [4, 6, 1, 25]  # prev + 1 + a, uint32 wrap (src/env.cc:340-345)


def test_oracle_batcher_matches_live_reference(golden_dir):
    """64 random trials drawn as test/unit/test_batcher.py:13-52 draws them, in both modes: after every item the
    restatement has emitted as many batches as the reference did (tests/golden/batcher_random_golden.npz), and every
    batch has the digest of the reference's batch (dtype, shape and bytes)."""
    g = np.load(f"{golden_dir}/batcher_random_golden.npz")
    for ti, t in enumerate(g["trials"]):
        size, dim, shape, n = ast.literal_eval(str(t))
        for mode in ("stack", "cat"):
            emitted, ref = g[f"r{ti}_{mode}_emitted"], g[f"r{ti}_{mode}_digests"]
            assert len(emitted) == n and len(ref) == int(emitted.sum())
            b = oracle.OracleBatcher(size, dim=dim)
            k = 0
            for j in range(n):
                getattr(b, mode)(torch.from_numpy(gen_input(batcher_random_seed(ti, mode, j), shape, "f32")))
                got = 0
                while not b.empty():
                    assert digest(b.get().numpy()) == ref[k], (ti, mode, j)
                    k += 1
                    got += 1
                assert got == emitted[j], (ti, mode, j)


def test_oracle_tree_allreduce_matches_live_reference(golden_dir):
    """group.all_reduce of the compiled reference with 4 in-process peers (test/test_reduce.py layout, recorded in
    tests/golden/allreduce_2049_golden.npz) equals the C restatement of the tree for one of the legal arrival orders --
    bit for bit, 2049 floats per peer -- and the product's rank order is within tolerance of it."""
    g = np.load(f"{golden_dir}/allreduce_2049_golden.npz")
    n, numel = int(g["n"]), int(g["numel"])
    rng = np.random.default_rng(2026)
    for rep in range(3):
        ins = [rng.standard_normal(numel).astype(np.float32) for _ in range(n)]
        ref = g[f"rep{rep}"]
        assert any(oracle.allreduce_tree(ins, [(1, 0, 1)] * n, order=m, scale=False)[0].tobytes() == ref.tobytes()
                   for m in tree_masks(n)), rep
        ours, _ = oracle.allreduce_rankorder(ins, [(1, 0, 1)] * n, scale=False)
        assert (np.abs(ours.astype(np.float64) - ref) <= oracle.allreduce_tolerance(ins, ref)).all()
