"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the bfloat16 / float16 NVLink allreduce (mb_ar_*_ex).

Per element: widen every contributing rank's value to fp32, sum in fp32 in ascending rank order, multiply by the fp32
reciprocal 1.0f/sum(num_gradients) when scaling, round ONCE to nearest-even in the dtype.  Local accumulation (K-A1 `+=`)
rounds in the dtype after every add, like ATen's add_.

Values travel as uint16 bit patterns; the conversions are explicit integer round-to-nearest-even (fp16 subnormals
included), with no half-precision type from numpy or the compiler.  NaN becomes the canonical NaN 0x7fff that the
device's cvt.rn.{bf16,f16}x2.f32 produces.  Nothing here is used by the product path.
"""
import numpy as np

U_ROUNDOFF = {"bf16": 2.0 ** -8, "f16": 2.0 ** -11, "f32": 2.0 ** -24}


def _u32(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def f32_to_bf16_bits(x):
    """fp32 -> bf16 bit patterns, round to nearest even."""
    u = _u32(x).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    nan = (u & 0x7FFFFFFF) > 0x7F800000
    return np.where(nan, np.uint16(0x7FFF), r).astype(np.uint16)


def f32_to_f16_bits(x):
    """fp32 -> IEEE binary16 bit patterns, round to nearest even, subnormals and overflow to infinity included."""
    u = _u32(x).astype(np.int64)
    sign = (u >> 16) & 0x8000
    a = u & 0x7FFFFFFF
    # normal range: rebias the exponent (127 -> 15) and round the low 13 mantissa bits
    v = a - (112 << 23)
    normal = (v + 0xFFF + ((v >> 13) & 1)) >> 13
    # below 2^-14: the result is round(m * 2^(e - 126)) with the implicit bit restored (zero / fp32 subnormals -> 0)
    e = a >> 23
    m = (a & 0x7FFFFF) | 0x800000
    shift = np.clip(126 - e, 1, 62)
    q = m >> shift
    rem = m & ((np.int64(1) << shift) - 1)
    half = np.int64(1) << (shift - 1)
    sub = q + ((rem > half) | ((rem == half) & ((q & 1) == 1))).astype(np.int64)
    sub = np.where(shift > 25, 0, sub)
    h = np.where(a < 0x38800000, sub, normal)
    h = np.where(a >= 0x477FF000, 0x7C00, h)  # >= 65520 rounds to infinity
    h = np.where(a == 0x7F800000, 0x7C00, h)
    h = h | sign
    h = np.where(a > 0x7F800000, 0x7FFF, h)
    return h.astype(np.uint16)


def bf16_bits_to_f32(h):
    return (np.asarray(h, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)


def f16_bits_to_f32(h):
    """binary16 -> fp32 (exact), by integer arithmetic."""
    h = np.asarray(h, dtype=np.uint16).astype(np.uint32)
    sign = (h & 0x8000) << 16
    e = (h >> 10) & 0x1F
    m = h & 0x3FF
    normal = ((e + 112) << 23) | (m << 13)
    # subnormal: m * 2^-24, exact in fp32
    sub = (m.astype(np.float64) * 2.0 ** -24).astype(np.float32).view(np.uint32)
    special = (0xFF << 23) | (m << 13)
    r = np.where(e == 0, sub, np.where(e == 31, special, normal))
    return (r | sign).astype(np.uint32).view(np.float32)


def to_bits(x, dt):
    return f32_to_bf16_bits(x) if dt == "bf16" else f32_to_f16_bits(x)


def to_f32(h, dt):
    return bf16_bits_to_f32(h) if dt == "bf16" else f16_bits_to_f32(h)


def stage_add(acc_bits, g_bits, dt):
    """K-A1 `+=` in the dtype: round(widen(acc) + widen(g))."""
    return to_bits(to_f32(acc_bits, dt) + to_f32(g_bits, dt), dt)


def allreduce_rankorder(inputs, hdrs, dt, scale=True, numel=None):
    """inputs[r]: uint16 bit patterns of rank r (all the same length) or None (the rank skipped); hdrs[r] =
    (num_gradients, num_skipped, batch_size).  Returns (uint16 result, summed header incl. has_grads); no rank with
    gradients gives zeros (of `numel` elements)."""
    tot = [0, 0, 0, 0]
    for r, h in enumerate(hdrs):
        tot[0] += h[0]
        tot[1] += h[1]
        tot[2] += h[2]
        tot[3] += inputs[r] is not None
    n = numel if numel is not None else next((a.size for a in inputs if a is not None), 0)
    acc = None
    for a in inputs:
        if a is None:
            continue
        w = to_f32(a, dt)
        acc = w.copy() if acc is None else (acc + w).astype(np.float32)
    if acc is None:
        acc = np.zeros(n, dtype=np.float32)
    if scale and tot[0]:
        s = np.float32(1.0) / np.float32(tot[0])
        acc = (acc * s).astype(np.float32)
    return to_bits(acc, dt), tuple(tot)


def allreduce_tolerance(inputs, reference_out, dt, scale_factor=1.0):
    """Per-element bound between this restatement and the reference's tree (DESIGN.md §2):
    |ours - ref| <= (N+1) * u * max(|ref|, sum_i |g_i| * scale), u = 2^-8 (bf16), 2^-11 (fp16); N = contributing ranks.
    inputs / reference_out as fp32 values.  dt='f32' gives the fp32 bar's form with u = 2^-24."""
    s = np.zeros_like(reference_out, dtype=np.float64)
    n = 0
    for a in inputs:
        if a is not None:
            s += np.abs(a.astype(np.float64))
            n += 1
    return (n + 1) * U_ROUNDOFF[dt] * np.maximum(np.abs(reference_out.astype(np.float64)), s * scale_factor)
