"""bf16 / fp16 gradients over NVLink: the _ex C-ABI (K-A1, K-A0 + K-A2 one-shot / two-shot / two-shot in place) on
every GPU of the box from one process, the Accumulator with bf16 and mixed models, and Group.all_reduce on bf16 / fp16
CUDA tensors.  Every result is checked bit for bit against the CPU restatement (tests/lowp_oracle.py for bf16 / fp16,
oracle.allreduce_rankorder for fp32 tensors of a mixed list).  Multi-GPU cases skip below their world size."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

import lowp_oracle as lo
import moolib_b200 as moolib
import oracle
from helpers import gen_input
from moolib_b200 import _C, _lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NGPU = torch.cuda.device_count() if torch.cuda.is_available() else 0
TORCH_DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
SIZES = [0, 1, 7, 8, 9, 4097]
LISTS = {
    "bf16": [(n, "bf16") for n in SIZES],
    "f16": [(n, "f16") for n in SIZES],
    "mixed": [(n, d) for n in SIZES for d in ("bf16", "f32", "f16")],
}
WORLDS = [n for n in (1, 2, 4, 8) if n <= NGPU]


def u16(t):
    return t.detach().cpu().contiguous().view(torch.int16).numpy().view(np.uint16).reshape(-1)


def host_values(spec, rank, seed):
    """Rank `rank`'s CPU tensors for a list spec [(numel, dtype)]."""
    return [torch.from_numpy(gen_input(seed + 97 * rank + i, [n], "f32")).to(TORCH_DT[d]) for i, (n, d) in enumerate(spec)]


def expected(spec, per_rank, hdrs, scale):
    """Per tensor: the bytes of the rank-order result; per_rank[r] is None for a rank without gradients."""
    out = []
    for i, (n, d) in enumerate(spec):
        if d == "f32":
            ins = [None if v is None else v[i].numpy() for v in per_rank]
            e, _ = oracle.allreduce_rankorder(ins, hdrs, scale=scale, numel=n)
        else:
            ins = [None if v is None else u16(v[i]) for v in per_rank]
            e, _ = lo.allreduce_rankorder(ins, hdrs, d, scale=scale, numel=n)
        out.append(e.tobytes())
    return out


def device_bytes(t):
    if t.numel() == 0:
        return b""
    return t.detach().cpu().contiguous().view(torch.uint8).numpy().tobytes()


def make_ctxs(n, max_bytes):
    ctxs = [_lib.ArContext(r, n, r, max_bytes) for r in range(n)]
    hs = [c.export() for c in ctxs]
    for r, c in enumerate(ctxs):
        for q in range(n):
            if q != r:
                c.import_peer(q, hs[q])
    return ctxs


def sync_all(n):
    for r in range(n):
        torch.cuda.synchronize(r)


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("kind", sorted(LISTS))
def test_ex_rounds_all_algorithms_bit_exact(world, kind):
    spec = LISTS[kind]
    _, total, segs = _lib.layout([n for n, _ in spec], [d for _, d in spec])
    ctxs = make_ctxs(world, total)
    try:
        host = [host_values(spec, r, 1000) for r in range(world)]
        srcs = [[t.to(f"cuda:{r}") for t in host[r]] for r in range(world)]
        algos = [("oneshot", _lib.MB_AR_ALGO_ONESHOT, False)]
        if world > 1:
            algos += [("twoshot", _lib.MB_AR_ALGO_TWOSHOT, False), ("inplace", _lib.MB_AR_ALGO_TWOSHOT, True)]
        cases = [("all", [(1, 0, 10, 1)] * world)]
        if world > 1:
            cases.append(("skip", [(1, 0, 10, 1)] * (world - 1) + [(0, 1, 0, 0)]))
        cases.append(("none", [(0, 1, 0, 0)] * world))
        for case, hdrs in cases:
            per_rank = [host[r] if hdrs[r][3] else None for r in range(world)]
            for scale in (True, False):
                exp = expected(spec, per_rank, [h[:3] for h in hdrs], scale)
                for gated in (False, True):
                    for name, algo, inplace in algos:
                        dsts, flats = [], []
                        for r in range(world):
                            with torch.cuda.device(r):
                                ctxs[r].stage_ex(srcs[r])  # K-A1 (=): the padding becomes zero
                                if inplace:
                                    flats.append(ctxs[r].buffer_bytes(total))
                                    dsts.append(None)
                                else:
                                    dsts.append([torch.full((n,), float("nan"), dtype=TORCH_DT[d], device=f"cuda:{r}")
                                                 for n, d in spec])
                        for r in range(world):
                            with torch.cuda.device(r):
                                kw = dict(flat_dst=flats[r]) if inplace else {}
                                tensors = spec if inplace else dsts[r]
                                if gated:
                                    # min_batch 0: the gate opens even when no rank has gradients (batch 0)
                                    ctxs[r].reduce_gated_ex(0, tensors, hdr=hdrs[r], scale=scale, algo=algo, **kw)
                                else:
                                    ctxs[r].allreduce_ex(tensors, hdr=hdrs[r], scale=scale, algo=algo, **kw)
                        sync_all(world)
                        for r in range(world):
                            res, status = ctxs[r].result()
                            assert status == 0, (case, name, r)
                            assert res[0] == sum(h[0] for h in hdrs) and res[3] == sum(h[3] for h in hdrs)
                            if gated:
                                ctxs[r].advance()
                            if inplace:
                                offs, _, _ = _lib.layout([n for n, _ in spec], [d for _, d in spec])
                                flat = device_bytes(flats[r])
                                got = [flat[o:o + n * (4 if d == "f32" else 2)] for o, (n, d) in zip(offs, spec)]
                            else:
                                got = [device_bytes(t) for t in dsts[r]]
                            for i, (n, d) in enumerate(spec):
                                assert got[i] == exp[i], f"{kind} {case} scale={scale} gated={gated} {name} rank {r} " \
                                                         f"tensor {i} ({n} x {d})"
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("kind", sorted(LISTS))
def test_stage_ex_accumulates_like_aten_add(kind):
    spec = LISTS[kind]
    offs, total, _ = _lib.layout([n for n, _ in spec], [d for _, d in spec])
    ctx = _lib.ArContext(0, 1, 0, total)
    try:
        a = host_values(spec, 0, 5000)
        b = host_values(spec, 0, 6000)
        da = [t.cuda() for t in a]
        db = [t.cuda() for t in b]
        buf = ctx.buffer_bytes(total)
        buf.fill_(0xAB)
        ctx.stage_ex(da)
        ctx.stage_ex(db, accumulate=True, zero_src=True)
        torch.cuda.synchronize()
        flat = device_bytes(buf)
        for i, (n, d) in enumerate(spec):
            size = 4 if d == "f32" else 2
            exp = a[i].clone().add_(b[i])  # ATen on the CPU: fp32 add, one rounding to the dtype
            assert flat[offs[i]:offs[i] + n * size] == device_bytes(exp), (kind, i, n, d)
            pad_end = offs[i] + -(-n * size // 16) * 16
            assert flat[offs[i] + n * size:pad_end] == bytes(pad_end - offs[i] - n * size)  # padding stays zero
            assert device_bytes(db[i]) == bytes(n * size)  # sources zeroed
    finally:
        ctx.close()


def test_ex_rejects_other_dtypes_and_fp32_lists_run_the_fp32_entry_points():
    ctx = _lib.ArContext(0, 1, 0, 1 << 16)
    try:
        t = torch.zeros(8, dtype=torch.float64, device="cuda")
        with pytest.raises(ValueError, match="supported"):
            ctx.stage_ex([t])
        # all-fp32 list through the _ex entry points == mb_ar_stage + mb_ar_allreduce, bit for bit
        x = [torch.from_numpy(gen_input(7 + i, [n], "f32")).cuda() for i, n in enumerate([7, 4097, 1])]
        d1 = [torch.empty_like(v) for v in x]
        d2 = [torch.empty_like(v) for v in x]
        ctx.stage_ex(x)
        ctx.allreduce_ex(d1, hdr=(3, 0, 1, 1))
        ctx.stage(x)
        ctx.allreduce(d2, hdr=(3, 0, 1, 1))
        torch.cuda.synchronize()
        assert all(torch.equal(p.view(torch.int32), q.view(torch.int32)) for p, q in zip(d1, d2))
    finally:
        ctx.close()


# ---- Accumulator, one process ------------------------------------------------------------------------------------------

def connect(name, m, port):
    addr = f"127.0.0.1:{port}"
    broker = moolib.Broker()
    broker.listen(addr)
    acc = moolib.Accumulator(name, m.parameters(), m.buffers())
    acc.connect(addr)
    t0 = time.time()
    while not (acc.connected() and acc.wants_gradients()):
        broker.update()
        acc.update()
        assert time.time() - t0 < 60
    return broker, acc


def wait_grads(broker, acc):
    t0 = time.time()
    while not acc.has_gradients():
        broker.update()
        acc.update()
        assert time.time() - t0 < 30


def grad_bits(m):
    return [u16(p.grad) if p.dtype != torch.float32 else p.grad.detach().cpu().numpy().reshape(-1).view(np.uint16)
            for p in m.parameters()]


def make_model(mixed):
    torch.manual_seed(3)
    if mixed:
        return torch.nn.Sequential(torch.nn.LayerNorm(32), torch.nn.Linear(32, 31).to(torch.bfloat16)).cuda()
    return torch.nn.Linear(32, 31).to(torch.bfloat16).cuda()


def forward(m, x, mixed):
    if mixed:
        return m[1](m[0](x).to(torch.bfloat16)).float()
    return m(x.to(torch.bfloat16)).float()


@pytest.mark.parametrize("mixed", [False, True], ids=["bf16", "bf16+fp32"])
def test_accumulator_bf16_and_mixed_models_one_process(mixed):
    m = make_model(mixed)
    ref = make_model(mixed)
    ref.load_state_dict(m.state_dict())
    broker, acc = connect("lowp" + str(int(mixed)), m, 47500 + int(mixed))
    params = list(m.parameters())
    numel = [p.numel() for p in params]
    dts = [str(p.dtype).replace("torch.", "") for p in params]
    offs, total, _ = _lib.layout(numel, dts)
    x = torch.from_numpy(gen_input(11, [20, 32], "f32")).cuda()

    # round 1: .grad are ordinary tensors (made before the NVLink context existed): K-A1 + K-A2
    acc.set_virtual_batch_size(1)
    (forward(m, x, mixed) ** 2).sum().backward()
    (forward(ref, x, mixed) ** 2).sum().backward()
    before = _C.kernel_launches()
    acc.reduce_gradients(1)
    wait_grads(broker, acc)
    assert _C.kernel_launches() - before == 2
    assert all(p.grad.dtype == p.dtype for p in params)
    for p, q in zip(params, ref.parameters()):  # one contribution: x fp32(1.0), rounded once == the gradient itself
        assert torch.equal(p.grad, q.grad)
    acc.zero_gradients()
    ref.zero_grad()

    # rounds 2..3: .grad are views of the NVLink staging ring in the layout of mb_ar_layout; a real backward() writes
    # where the peers read; one launch per round (N=1: the gate is a host comparison, K-A2 only)
    for rnd in range(2):
        base = params[0].grad.data_ptr() - offs[0]
        assert [p.grad.data_ptr() - base for p in params] == offs
        y = torch.from_numpy(gen_input(20 + rnd, [20, 32], "f32")).cuda()
        (forward(m, y, mixed) ** 2).sum().backward()
        (forward(ref, y, mixed) ** 2).sum().backward()
        before = _C.kernel_launches()
        acc.reduce_gradients(1)
        wait_grads(broker, acc)
        assert _C.kernel_launches() - before == 1
        for p, q in zip(params, ref.parameters()):
            assert torch.equal(p.grad, q.grad), rnd
        acc.zero_gradients()
        ref.zero_grad()
    tm = acc.reduce_timings()
    assert tm["zero_copy_rounds"] == 2 and tm["bytes"] == total

    # two local contributions before the gate opens: the second is folded in by K-A1 (`+=` in the dtype), then scaled by
    # fp32(1/2) and rounded once
    acc.set_virtual_batch_size(2)
    gs = []
    for c in range(2):
        t0 = time.time()
        while not acc.wants_gradients():
            broker.update()
            acc.update()
            assert time.time() - t0 < 30
        y = torch.from_numpy(gen_input(40 + c, [20, 32], "f32")).cuda()
        (forward(m, y, mixed) ** 2).sum().backward()
        gs.append([p.grad.detach().cpu().clone() for p in params])
        acc.reduce_gradients(1)
        for _ in range(5):
            broker.update()
            acc.update()
    wait_grads(broker, acc)
    for i, p in enumerate(params):
        if p.dtype == torch.float32:
            st = np.zeros(numel[i], np.float32)
            oracle.stage(st, [gs[0][i].numpy().reshape(-1).copy()])
            oracle.stage(st, [gs[1][i].numpy().reshape(-1).copy()], accumulate=True)
            e, _ = oracle.allreduce_rankorder([st], [(2, 0, 2)])
            assert p.grad.cpu().numpy().reshape(-1).tobytes() == e.tobytes(), i
        else:
            st = lo.stage_add(u16(gs[0][i]), u16(gs[1][i]), "bf16")
            e, _ = lo.allreduce_rankorder([st], [(2, 0, 2)], "bf16")
            assert u16(p.grad).tobytes() == e.tobytes(), i
    assert acc.get_gradient_stats() == {"num_gradients": 2, "num_skipped": 0, "batch_size": 2}
    acc.zero_gradients()
    assert not any(device_bytes(p.grad).strip(b"\0") for p in params)


def test_accumulator_refuses_other_dtypes():
    m = torch.nn.Linear(4, 3).double().cuda()
    with pytest.raises(RuntimeError, match="float32, bfloat16 or float16"):
        moolib.Accumulator("f64", m.parameters(), m.buffers())


PARALLEL = r"""
import os, sys, time, numpy as np, torch
sys.path.insert(0, os.environ['MB_ROOT']); sys.path.insert(0, os.path.join(os.environ['MB_ROOT'], 'tests'))
import moolib_b200 as moolib
from helpers import gen_input
addr = '127.0.0.1:' + os.environ['MB_PORT']
broker = moolib.Broker(); broker.listen(addr)
m = torch.nn.Linear(32, 31).to(torch.bfloat16).cuda()
acc = moolib.Accumulator('accp', m.parameters(), m.buffers())
acc.set_parallel_gradients(2)
acc.set_virtual_batch_size(10)
acc.connect(addr)
t0 = time.time()
while not (acc.connected() and acc.wants_gradients()):
    broker.update(); acc.update(); assert time.time() - t0 < 60
bf = lambda s, sh: torch.from_numpy(gen_input(s, sh, 'f32')).to(torch.bfloat16)
gs = [(bf(50 + 2 * k, [31, 32]), bf(51 + 2 * k, [31])) for k in range(6)]
fed = applied = 0
t0 = time.time()
while applied < 6:
    assert time.time() - t0 < 60
    broker.update(); acc.update()
    if acc.has_gradients():
        assert m.weight.grad.dtype == torch.bfloat16
        assert torch.equal(m.weight.grad.cpu(), gs[applied][0]) and torch.equal(m.bias.grad.cpu(), gs[applied][1]), applied
        acc.zero_gradients(); applied += 1
    elif fed < 6 and acc.wants_gradients():
        if os.environ.get('MOOLIB_B200_STRICT_COUNTING') == '0':
            m.weight.grad = gs[fed][0].cuda(); m.bias.grad = gs[fed][1].cuda()
        else:
            with torch.no_grad():
                m.weight.grad.copy_(gs[fed][0]); m.bias.grad.copy_(gs[fed][1])
        acc.reduce_gradients(10); fed += 1
print('PARALLEL OK', acc.reduce_timings())
os._exit(0)
"""


@pytest.mark.parametrize("strict", ["1", "0"], ids=["device-gate", "host-counted"])
def test_accumulator_bf16_parallel_gradients_and_host_counting(strict, tmp_path):
    """set_parallel_gradients(2) with a bf16 model, with the device gate and with MOOLIB_B200_STRICT_COUNTING=0."""
    script = tmp_path / "parallel.py"
    script.write_text(PARALLEL)
    env = dict(os.environ, MB_ROOT=ROOT, MB_PORT=str(47510 + int(strict)), MOOLIB_B200_STRICT_COUNTING=strict)
    r = subprocess.run([sys.executable, str(script)], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "PARALLEL OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


# ---- Group.all_reduce ----------------------------------------------------------------------------------------------------

def test_group_all_reduce_bf16_fp16_in_place_and_fp64_refused():
    addr = "127.0.0.1:47520"
    broker = moolib.Broker()
    broker.listen(addr)
    rpc = moolib.Rpc()
    rpc.set_name("solo")
    rpc.connect(addr)
    group = moolib.Group(rpc, "lowp")
    t0 = time.time()
    while not (group.active() and len(group.members()) == 1):
        broker.update()
        group.update()
        assert time.time() - t0 < 60
    for dt in (torch.bfloat16, torch.float16):
        x = torch.from_numpy(gen_input(3, [4097], "f32")).to(dt).cuda()
        before = x.clone()
        f = group.all_reduce("t" + str(dt), x)
        t0 = time.time()
        while not f.done():
            broker.update()
            group.update()
            assert time.time() - t0 < 60
        r = f.result()
        assert r.data_ptr() == x.data_ptr() and r.dtype == dt and torch.equal(x, before)
    with pytest.raises(RuntimeError, match="float32, bfloat16 and float16"):
        group.all_reduce("f64", torch.zeros(8, dtype=torch.float64, device="cuda"))


WORKER = r"""
import os, sys, time, zlib, numpy as np, torch
sys.path.insert(0, os.environ['MB_ROOT']); sys.path.insert(0, os.path.join(os.environ['MB_ROOT'], 'tests'))
import lowp_oracle as lo, moolib_b200 as moolib
from helpers import gen_input
rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
torch.cuda.set_device(int(os.environ['LOCAL_RANK']))
addr = '127.0.0.1:' + os.environ['MB_PORT']
broker = None
if rank == 0:
    broker = moolib.Broker(); broker.listen(addr)
rpc = moolib.Rpc(); rpc.set_name(f'peer{rank}'); rpc.set_timeout(30); rpc.connect(addr)
group = moolib.Group(rpc, 'g'); group.set_sort_order(rank)
torch.manual_seed(2000 + rank)   # every peer starts from DIFFERENT bf16 weights: the elected leader's must win
m = torch.nn.Linear(32, 31).to(torch.bfloat16).cuda()
acc = moolib.Accumulator('acc', m.parameters(), m.buffers(), group=group)
acc.set_virtual_batch_size(10 * world)
def pump():
    if broker: broker.update()
    group.update(); acc.update()
    if acc.wants_state(): acc.set_state({'k': 1})
    if acc.has_new_state(): acc.state()
t0 = time.time()
while not (acc.connected() and len(group.members()) == world):
    pump(); time.sleep(0.001); assert time.time() - t0 < 90, group.members()
u16 = lambda t: t.detach().cpu().contiguous().view(torch.int16).numpy().view(np.uint16).reshape(-1)
crc = zlib.crc32(np.concatenate([u16(p) for p in m.parameters()]).tobytes())
print(f'PARAMCRC {rank} {crc:08x}', flush=True)
bf = lambda s, sh: torch.from_numpy(gen_input(s, sh, 'f32')).to(torch.bfloat16)
# group.all_reduce on bf16 / fp16 CUDA tensors, in place, identical bits on every rank
for dt, tag in ((torch.bfloat16, 'bf16'), (torch.float16, 'f16')):
    x = torch.from_numpy(gen_input(900 + rank, [4097], 'f32')).to(dt).cuda()
    f = group.all_reduce('t' + tag, x)
    t0 = time.time()
    while not f.done():
        pump(); assert time.time() - t0 < 60
    f.result()
    ins = [u16(torch.from_numpy(gen_input(900 + q, [4097], 'f32')).to(dt)) for q in range(world)]
    e, _ = lo.allreduce_rankorder(ins, [(1, 0, 1)] * world, tag, scale=False)
    assert u16(x).tobytes() == e.tobytes(), tag
for rnd in range(4):
    t0 = time.time()
    while not acc.wants_gradients():
        pump(); assert time.time() - t0 < 60
    skip = rnd == 2 and rank == world - 1
    acc.set_virtual_batch_size(10 * (world - 1) if rnd == 2 else 10 * world)
    if skip:
        acc.skip_gradients()
    else:
        m.weight.grad = bf(100 * rnd + 2 * rank, [31, 32]).cuda(); m.bias.grad = bf(100 * rnd + 2 * rank + 1, [31]).cuda()
        acc.reduce_gradients(10)
    t0 = time.time()
    while not acc.has_gradients():
        pump(); assert time.time() - t0 < 60, f'round {rnd}'
    ins, hdrs = [], []
    for q in range(world):
        if rnd == 2 and q == world - 1:
            ins.append(None); hdrs.append((0, 1, 0)); continue
        ins.append(np.concatenate([u16(bf(100 * rnd + 2 * q, [31, 32])), u16(bf(100 * rnd + 2 * q + 1, [31]))]))
        hdrs.append((1, 0, 10))
    e, eh = lo.allreduce_rankorder(ins, hdrs, 'bf16')
    assert m.weight.grad.dtype == torch.bfloat16
    assert np.concatenate([u16(m.weight.grad), u16(m.bias.grad)]).tobytes() == e.tobytes(), f'rank {rank} round {rnd}'
    s = acc.get_gradient_stats()
    assert (s['num_gradients'], s['num_skipped'], s['batch_size']) == eh[:3], (s, eh)
    acc.zero_gradients()
for _ in range(200):
    pump(); time.sleep(0.001)
print(f'rank {rank} OK', flush=True)
os._exit(0)
"""


@pytest.mark.parametrize("world", [n for n in (2, 4, 8) if n <= NGPU])
def test_accumulator_bf16_across_processes(world, tmp_path):
    """One process per GPU (CUDA IPC): bf16 rounds incl. a skipping peer, bf16 / fp16 group.all_reduce, and a
    differently initialised peer that ends with the leader's bf16 parameters (sent over the control plane)."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MB_ROOT=ROOT, MB_PORT=str(47600 + world))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", str(29800 + world), str(script)],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("OK") == world
    crcs = {ln.split()[2] for ln in r.stdout.splitlines() if ln.startswith("PARAMCRC")}
    assert len(crcs) == 1, f"peers hold different bf16 models after the model sync: {crcs}"
