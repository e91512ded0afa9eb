"""bf16 / fp16 allreduce, CPU side: the flat layout of mixed dtype lists (mb_ar_layout), the CPU restatement's
round-to-nearest-even conversions against torch, and the restatement replaying the reference's own bf16 / fp16 outputs
(tests/golden/lowp_golden.npz, made by tests/golden/make_golden_lowp.py) within the stated tolerance."""
import ast
import os

import numpy as np
import pytest
import torch

import lowp_oracle as lo
from helpers import gen_input
from moolib_b200 import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
TORCH_DT = {"bf16": torch.bfloat16, "f16": torch.float16}


# ---- layout ----------------------------------------------------------------------------------------------------------

def test_layout_all_fp32_is_the_fp32_rule():
    for numels in ([5, 8, 3], [992, 31], [0, 1, 7, 8, 9, 4097], [1]):
        off, total, segs = _lib.layout(numels, ["f32"] * len(numels))
        assert total == _lib.flat_numel(numels) * 4
        import oracle
        foff, ftotal = oracle.flat_layout(numels)
        assert off == [4 * o for o in foff] and total == 4 * ftotal
        assert segs == [(0, total, _lib.MB_DT_F32)]


def test_layout_groups_dtypes_and_aligns_every_tensor():
    numels = [9, 7, 0, 1, 31, 8, 4097, 3]
    dts = ["bf16", "f32", "f16", "bf16", "f32", "f16", "bf16", "f16"]
    off, total, segs = _lib.layout(numels, dts)
    size = {"f32": 4, "bf16": 2, "f16": 2}
    # runs in the order fp32, bf16, fp16; list order inside a run; 16 B aligned, padded to 4 / 8 elements
    at = 0
    expect = {}
    for d in ("f32", "bf16", "f16"):
        begin = at
        for i, (n, dt) in enumerate(zip(numels, dts)):
            if dt == d:
                expect[i] = at
                at += -(-n * size[d] // 16) * 16
        assert (begin, at, _lib.dtype_code(d)) in segs
    assert off == [expect[i] for i in range(len(numels))]
    assert total == at and all(o % 16 == 0 for o in off)
    assert [s[2] for s in segs] == [_lib.MB_DT_F32, _lib.MB_DT_BF16, _lib.MB_DT_F16]
    assert segs[0][0] == 0 and segs[0][1] == segs[1][0] and segs[1][1] == segs[2][0] and segs[2][1] == total


def test_layout_skips_empty_runs_and_rejects_other_dtypes():
    off, total, segs = _lib.layout([0, 5], ["f32", "bf16"])
    assert off == [0, 0] and total == 16 and segs == [(0, 16, _lib.MB_DT_BF16)]
    with pytest.raises(ValueError, match="supported"):
        _lib.dtype_code(torch.float64)
    with pytest.raises(_lib.MoolibB200Error, match="MB_DT_BF16"):
        _lib.layout([4], [7])


# ---- the restatement's conversions --------------------------------------------------------------------------------------

def _patterns():
    """A dense sample of the 2^32 fp32 bit patterns: every 251st pattern, every sign/exponent/top-mantissa combination
    with the low bits at the rounding boundaries of both dtypes, and the special values."""
    strided = np.arange(0, 2 ** 32, 251, dtype=np.uint64).astype(np.uint32)
    hi = np.arange(0, 2 ** 16, dtype=np.uint32) << 16
    lows = np.array([0, 1, 0x0FFF, 0x1000, 0x1001, 0x1FFF, 0x2000, 0x3000, 0x7FFF, 0x8000, 0x8001, 0xFFFF, 0xE000,
                     0x6000], dtype=np.uint32)
    edge = (hi[:, None] | lows[None, :]).reshape(-1)
    special = np.array([0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00001, 0x7F800001, 0, 0x80000000, 1, 0x477FF000,
                        0x477FEFFF, 0x33000000, 0x33000001, 0x387FFFFF, 0x38800000], dtype=np.uint32)
    return np.concatenate([strided, edge, special]).view(np.float32)


@pytest.mark.parametrize("dt", ["bf16", "f16"])
def test_rne_conversion_matches_torch(dt):
    x = _patterns()
    for k in range(0, x.size, 1 << 23):
        chunk = x[k:k + (1 << 23)]
        ours = lo.to_bits(chunk, dt)
        ref = torch.from_numpy(chunk).to(TORCH_DT[dt]).view(torch.int16).numpy().view(np.uint16)
        nan = np.isnan(chunk)
        assert np.array_equal(ours[~nan], ref[~nan]), dt
        assert np.isnan(lo.to_f32(ours[nan], dt)).all()


@pytest.mark.parametrize("dt", ["bf16", "f16"])
def test_widening_is_exact(dt):
    h = np.arange(2 ** 16, dtype=np.uint32).astype(np.uint16)
    ours = lo.to_f32(h, dt)
    ref = torch.from_numpy(h.view(np.int16)).view(TORCH_DT[dt]).float().numpy()
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(ours), nan)
    assert np.array_equal(ours[~nan].view(np.uint32), ref[~nan].view(np.uint32))


def test_stage_add_rounds_in_the_dtype_like_aten():
    for dt in ("bf16", "f16"):
        a = torch.from_numpy(gen_input(1, [4097], "f32")).to(TORCH_DT[dt])
        b = torch.from_numpy(gen_input(2, [4097], "f32")).to(TORCH_DT[dt])
        ab = lambda t: t.view(torch.int16).numpy().view(np.uint16)  # noqa: E731
        assert np.array_equal(lo.stage_add(ab(a), ab(b), dt), ab(a.clone().add_(b)))


# ---- replaying the reference's outputs ----------------------------------------------------------------------------------

def _golden():
    return np.load(os.path.join(HERE, "golden", "lowp_golden.npz"))


def _bits(seed, shape, dt):
    return torch.from_numpy(gen_input(seed, shape, "f32")).to(TORCH_DT[dt]).view(torch.int16).numpy().view(np.uint16).reshape(-1)


def test_allreduce_replays_reference_within_tolerance():
    g = _golden()
    cases = [ast.literal_eval(str(m)) for m in g["meta"] if "'allreduce'" in str(m)]
    assert len(cases) == 24
    worst = 0.0
    for _, n, dt, numel, seed in cases:
        ins = [_bits(seed * 16 + r, [numel], dt) for r in range(n)]
        ours, tot = lo.allreduce_rankorder(ins, [(1, 0, 1)] * n, dt, scale=False)
        ref = g[f"ar_n{n}_{dt}_{numel}"]
        of, rf = lo.to_f32(ours, dt).astype(np.float64), lo.to_f32(ref, dt).astype(np.float64)
        tol = lo.allreduce_tolerance([lo.to_f32(a, dt) for a in ins], rf, dt)
        err = np.abs(of - rf)
        assert (err <= tol).all(), (n, dt, numel, float((err / np.maximum(tol, 1e-30)).max()))
        worst = max(worst, float((err / np.maximum(tol, 1e-30)).max()))
        assert tot == (n, 0, n, n)
    # the bound is not vacuous: the reference's per-add rounding shows up, and it stays well inside the bound
    assert 0.0 < worst <= 1.0


def _acc_rounds(g):
    return [ast.literal_eval(str(m)) for m in g["meta"] if "'accumulator'" in str(m)]


def _acc_inputs(plan, dt="bf16"):
    ins, hdrs = [], []
    for seeds in plan:
        if not seeds:
            ins.append(None)
            hdrs.append((0, 1, 0))
            continue
        st = None
        for s in seeds:
            x = np.concatenate([_bits(s, [31, 32], dt), _bits(s + 1, [31], dt)])
            st = x if st is None else lo.stage_add(st, x, dt)
        ins.append(st)
        hdrs.append((len(seeds), 0, 10 * len(seeds)))
    return ins, hdrs


def test_accumulator_rounds_replay_reference():
    g = _golden()
    rounds = _acc_rounds(g)
    assert len(rounds) == 8
    for _, tag, n, plan, vbs, ng, nskip, bs in rounds:
        ins, hdrs = _acc_inputs(plan)
        ours, tot = lo.allreduce_rankorder(ins, hdrs, "bf16")
        assert tot[0] == ng and tot[2] == bs
        ref = np.concatenate([g[f"acc_{tag}_w"].reshape(-1), g[f"acc_{tag}_b"]])
        contributors = sum(a is not None for a in ins)
        if contributors == 1:
            # a single contributor: widen, x fp32(1/numGradients), round once == the reference's copy_ + mul_
            assert ours.tobytes() == ref.tobytes(), tag
            continue
        of, rf = lo.to_f32(ours, "bf16").astype(np.float64), lo.to_f32(ref, "bf16").astype(np.float64)
        tol = lo.allreduce_tolerance([lo.to_f32(a, "bf16") for a in ins if a is not None], rf, "bf16",
                                     scale_factor=1.0 / ng)
        assert (np.abs(of - rf) <= tol).all(), tag
