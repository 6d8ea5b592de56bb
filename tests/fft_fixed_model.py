"""Bit-exact NumPy model of the two fixed-point complex FFTs of CMSIS-DSP V1.5.3 (TEST INFRASTRUCTURE ONLY):

- arm_cfft_q15 (arm_cfft_q15.c:77) in its ARM_MATH_DSP branch, the one a Cortex-M4 build compiles: dual 16-bit lanes with
  saturating (__QADD16, __QSUB16, __QASX, __QSAX) and halving (__SHADD16, __SHSUB16, __SHASX, __SHSAX) adds, and twiddle
  products that keep the high half-word of a wrapping 32-bit sum of two 16 x 16 products (__SMUAD, __SMUSDX, __SMUSD, __SMUADX);
- arm_cfft_q31 (arm_cfft_q31.c:77): wrapping 32-bit sums, the high word of 64-bit products in the radix-4 butterflies, and the
  rounded mult_32x32_keep32_R / multAcc_ / multSub_ macros (arm_math.h) in the radix-4-by-2 stage.

N = 4^m runs arm_radix4_butterfly_{,inverse_}q15 / q31 with twiddle step 1. N = 2 * 4^m runs arm_cfft_radix4by2_{,inverse_}q15 / q31:
a radix-2 stage, the two half-length radix-4 transforms with twiddle step 2 on the same table, and a final doubling. Then
arm_bitreversal_16 / _32 puts the result in natural order.

Written from the CMSIS loop structure: the butterflies of a stage are enumerated in the reference's loop order, and the twiddle
index starts at 0 for each group and steps by the twiddle modifier per butterfly. Every butterfly of one stage touches its own four
samples, so a stage is then evaluated at once over all its butterflies and over a batch of transforms. All arithmetic is int64
NumPy with explicit saturation and wrapping. This module does not load the library under test.
"""
import functools

import numpy as np

SIZES = (16, 32, 64, 128, 256, 512, 1024, 2048, 4096)


# ------------------------------------------------------------------ twiddle tables ------------------------------------------------------------------
def twiddle_q15(N):
    """twiddleCoef_N_q15 (arm_common_tables.c): 3 N / 4 pairs (cos, sin) of 2 pi k / N, floor (v * 2^15) clipped to q15."""
    a = 2.0 * np.pi * np.arange(3 * N // 4) / N
    v = np.stack([np.cos(a), np.sin(a)], 1).reshape(-1)
    return np.clip(np.floor(v * 32768.0), -32768, 32767).astype(np.int16)


def twiddle_q31(N):
    """twiddleCoef_N_q31 (arm_common_tables.c): 3 N / 4 pairs (cos, sin) of 2 pi k / N, floor (v * 2^31 + 0.05) clipped to q31."""
    a = 2.0 * np.pi * np.arange(3 * N // 4) / N
    v = np.stack([np.cos(a), np.sin(a)], 1).reshape(-1)
    return np.clip(np.floor(v * 2147483648.0 + 0.05), -2147483648, 2147483647).astype(np.int32)


# ------------------------------------------------------------------ integer helpers ------------------------------------------------------------------
def _wrap32(v):
    return ((v + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)


def _wrap16(v):
    return ((v + (1 << 15)) & 0xFFFF) - (1 << 15)


def _sat16(v):
    return np.clip(v, -32768, 32767)


# A q15 complex word is a pair (x, y) = (low half-word: real, high half-word: imaginary), each lane an int64 array.
def qadd16(a, b): return _sat16(a[0] + b[0]), _sat16(a[1] + b[1])
def qsub16(a, b): return _sat16(a[0] - b[0]), _sat16(a[1] - b[1])
def shadd16(a, b): return (a[0] + b[0]) >> 1, (a[1] + b[1]) >> 1
def shsub16(a, b): return (a[0] - b[0]) >> 1, (a[1] - b[1]) >> 1
def qasx(a, b): return _sat16(a[0] - b[1]), _sat16(a[1] + b[0])      # low: a.lo - b.hi, high: a.hi + b.lo
def qsax(a, b): return _sat16(a[0] + b[1]), _sat16(a[1] - b[0])      # low: a.lo + b.hi, high: a.hi - b.lo
def shasx(a, b): return (a[0] - b[1]) >> 1, (a[1] + b[0]) >> 1
def shsax(a, b): return (a[0] + b[1]) >> 1, (a[1] - b[0]) >> 1
def smuad(a, b): return _wrap32(a[0] * b[0] + a[1] * b[1])
def smusd(a, b): return _wrap32(a[0] * b[0] - a[1] * b[1])
def smuadx(a, b): return _wrap32(a[0] * b[1] + a[1] * b[0])
def smusdx(a, b): return _wrap32(a[0] * b[1] - a[1] * b[0])


ZERO = (0, 0)


def _cmul_q15(coef, v, inv):
    """The twiddle product and its pack: out1 = (__SMUAD or __SMUSD) >> 16 goes to the low half-word, the high half-word of
    out2 = __SMUSDX or __SMUADX to the high one. Forward: v (co - j si); inverse: v (co + j si)."""
    out1 = (smusd(coef, v) if inv else smuad(coef, v)) >> 16
    out2 = smuadx(coef, v) if inv else smusdx(coef, v)
    return _wrap16(out1 & 0xFFFF), out2 >> 16


def _hi32(a, b):
    """(int32_t) (((q63_t) a * b) >> 32)"""
    return (a * b) >> 32


def _cmul_q31(co, si, r, s, inv):
    """(re, im) of (r + j s) (co -/+ j si) as the radix-4 q31 butterflies write it: high words summed with a 32-bit wrap."""
    if inv:
        return _wrap32(_hi32(r, co) - _hi32(s, si)), _wrap32(_hi32(s, co) + _hi32(r, si))
    return _wrap32(_hi32(r, co) + _hi32(s, si)), _wrap32(_hi32(s, co) - _hi32(r, si))


# ------------------------------------------------------------------ butterfly plans ------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _radix4_plan(L, modifier):
    """The butterflies of arm_radix4_butterfly_* on L points in the reference's loop order, per stage: the four sample indices
    (i0, i0 + n2, i0 + 2 n2, i0 + 3 n2) and the twiddle index ic (C1 = ic, C2 = 2 ic, C3 = 3 ic) of each butterfly. The last stage
    has no twiddles and walks groups of four neighbours."""
    stages = []
    # first stage: i0 = 0 .. n2 - 1, ic += twidCoefModifier per butterfly
    n2 = L >> 2
    i0s, ics, ic = [], [], 0
    for i0 in range(n2):
        i0s.append(i0); ics.append(ic)
        ic += modifier
    stages.append(("first", n2, np.array(i0s), np.array(ics)))
    modifier <<= 2
    # middle stages: for (k = L / 4; k > 4; k >>= 2), each group j with its own twiddles, then i0 = j, j + n1, ...
    k = L >> 2
    while k > 4:
        n1, n2 = n2, n2 >> 2
        i0s, ics, ic = [], [], 0
        for j in range(n2):
            for i0 in range(j, L, n1):
                i0s.append(i0); ics.append(ic)
            ic += modifier
        stages.append(("middle", n2, np.array(i0s), np.array(ics)))
        modifier <<= 2
        k >>= 2
    stages.append(("last", 1, np.arange(0, L, 4), None))
    return stages


def _bitrev_perm(N):
    bits = N.bit_length() - 1
    return np.array([int(format(i, "0%db" % bits)[::-1], 2) for i in range(N)])


# ------------------------------------------------------------------ q15 ------------------------------------------------------------------
def _radix4_q15(x, y, L, tw, modifier, inv):
    """arm_radix4_butterfly_q15 / arm_radix4_butterfly_inverse_q15 (DSP branch) in place on x, y: [batch][L] int64."""
    co, si = tw[0::2].astype(np.int64), tw[1::2].astype(np.int64)
    for kind, n2, i0, ic in _radix4_plan(L, modifier):
        if kind == "last":
            ia, ib, icc, idd = i0, i0 + 1, i0 + 2, i0 + 3
            a, b, c, d = (x[:, ia], y[:, ia]), (x[:, ib], y[:, ib]), (x[:, icc], y[:, icc]), (x[:, idd], y[:, idd])
            R = qadd16(a, c); T = qadd16(b, d)
            o0 = shadd16(R, T); o1 = shsub16(R, T)
            S = qsub16(a, c); U = qsub16(b, d)
            o2, o3 = (shasx(S, U), shsax(S, U)) if inv else (shsax(S, U), shasx(S, U))
            for idx, o in ((ia, o0), (ib, o1), (icc, o2), (idd, o3)):
                x[:, idx], y[:, idx] = o
            continue
        i1, i2, i3 = i0 + n2, i0 + 2 * n2, i0 + 3 * n2
        C1, C2, C3 = (co[ic], si[ic]), (co[2 * ic], si[2 * ic]), (co[3 * ic], si[3 * ic])
        a, b, c, d = (x[:, i0], y[:, i0]), (x[:, i1], y[:, i1]), (x[:, i2], y[:, i2]), (x[:, i3], y[:, i3])
        if kind == "first":
            # two __SHADD16 (v, 0) per input: >> 2; saturating sums; the sum output halved once
            a, b, c, d = [shadd16(shadd16(v, ZERO), ZERO) for v in (a, b, c, d)]
            R = qadd16(a, c); S = qsub16(a, c); T = qadd16(b, d)
            o0 = shadd16(R, T)
            R = qsub16(R, T)
            T = qsub16(b, d)
            R2, S2 = (qsax(S, T), qasx(S, T)) if inv else (qasx(S, T), qsax(S, T))
        else:
            # saturating sums, every output halved twice
            R = qadd16(a, c); S = qsub16(a, c); T = qadd16(b, d)
            o0 = shadd16(shadd16(R, T), ZERO)
            R = shsub16(R, T)
            T = qsub16(b, d)
            R2, S2 = (shsax(S, T), shasx(S, T)) if inv else (shasx(S, T), shsax(S, T))
        o1 = _cmul_q15(C2, R, inv)
        o2 = _cmul_q15(C1, S2, inv)
        o3 = _cmul_q15(C3, R2, inv)
        for idx, o in ((i0, o0), (i1, o1), (i2, o2), (i3, o3)):
            x[:, idx], y[:, idx] = o


def cfft_q15(data, ifft=0):
    """arm_cfft_q15 (DSP branch) with bitReverseFlag = 1 on data [..., 2 N] int16 (interleaved re, im); returns a new array."""
    data = np.asarray(data, np.int16)
    N = data.shape[-1] // 2
    assert N in SIZES, N
    inv = bool(ifft)
    z = data.reshape(-1, N, 2).astype(np.int64)
    x, y = z[:, :, 0].copy(), z[:, :, 1].copy()
    tw = twiddle_q15(N)
    if N & 0x55555555:                                            # N = 4^m
        _radix4_q15(x, y, N, tw, 1, inv)
    else:
        # arm_cfft_radix4by2_{,inverse_}q15: halve both, saturating difference, twiddle (step 1)
        n2 = N >> 1
        coef = (tw[0:2 * n2:2].astype(np.int64), tw[1:2 * n2:2].astype(np.int64))
        T = shadd16((x[:, :n2], y[:, :n2]), ZERO)
        S = shadd16((x[:, n2:], y[:, n2:]), ZERO)
        R = qsub16(T, S)
        top = shadd16(T, S)
        bottom = _cmul_q15(coef, R, inv)
        x[:, :n2], y[:, :n2] = top
        x[:, n2:], y[:, n2:] = bottom
        for h in (slice(0, n2), slice(n2, N)):
            xh, yh = x[:, h].copy(), y[:, h].copy()
            _radix4_q15(xh, yh, n2, tw, 2, inv)
            x[:, h], y[:, h] = xh, yh
        # p <<= 1 in a q31_t, stored back into a q15_t: wraps
        x, y = _wrap16(x << 1), _wrap16(y << 1)
    p = _bitrev_perm(N)
    out = np.stack([x[:, p], y[:, p]], -1)
    return out.reshape(data.shape).astype(np.int16)


# ------------------------------------------------------------------ q31 ------------------------------------------------------------------
def _radix4_q31(x, y, L, tw, modifier, inv):
    """arm_radix4_butterfly_q31 / arm_radix4_butterfly_inverse_q31 in place on x, y: [batch][L] int64."""
    co, si = tw[0::2].astype(np.int64), tw[1::2].astype(np.int64)
    for kind, n2, i0, ia1 in _radix4_plan(L, modifier):
        if kind == "last":
            ia, ib, icc, idd = i0, i0 + 1, i0 + 2, i0 + 3
            xa, ya, xb, yb, xc, yc, xd, yd = x[:, ia], y[:, ia], x[:, ib], y[:, ib], x[:, icc], y[:, icc], x[:, idd], y[:, idd]
            o0 = _wrap32(xa + xb + xc + xd), _wrap32(ya + yb + yc + yd)
            o1 = _wrap32(xa - xb + xc - xd), _wrap32(ya - yb + yc - yd)
            plus = _wrap32(xa + yb - xc - yd), _wrap32(ya - xb - yc + xd)
            minus = _wrap32(xa - yb - xc + yd), _wrap32(ya + xb - yc - xd)
            o2, o3 = (minus, plus) if inv else (plus, minus)
            for idx, o in ((ia, o0), (ib, o1), (icc, o2), (idd, o3)):
                x[:, idx], y[:, idx] = o
            continue
        i1, i2, i3 = i0 + n2, i0 + 2 * n2, i0 + 3 * n2
        ia2, ia3 = 2 * ia1, 3 * ia1
        xa, ya, xb, yb, xc, yc, xd, yd = x[:, i0], y[:, i0], x[:, i1], y[:, i1], x[:, i2], y[:, i2], x[:, i3], y[:, i3]
        if kind == "first":
            xa, ya, xb, yb, xc, yc, xd, yd = [v >> 4 for v in (xa, ya, xb, yb, xc, yc, xd, yd)]   # 4 guard bits
        r1, r2 = _wrap32(xa + xc), _wrap32(xa - xc)
        s1, s2 = _wrap32(ya + yc), _wrap32(ya - yc)
        t1 = _wrap32(xb + xd)
        o0x = _wrap32(r1 + t1)
        r1 = _wrap32(r1 - t1)
        t2 = _wrap32(yb + yd)
        o0y = _wrap32(s1 + t2)
        s1 = _wrap32(s1 - t2)
        t1, t2 = _wrap32(yb - yd), _wrap32(xb - xd)
        o1 = _cmul_q31(co[ia2], si[ia2], r1, s1, inv)
        if inv:
            r1, r2, s1, s2 = _wrap32(r2 - t1), _wrap32(r2 + t1), _wrap32(s2 + t2), _wrap32(s2 - t2)
        else:
            r1, r2, s1, s2 = _wrap32(r2 + t1), _wrap32(r2 - t1), _wrap32(s2 - t2), _wrap32(s2 + t2)
        o2 = _cmul_q31(co[ia1], si[ia1], r1, s1, inv)
        o3 = _cmul_q31(co[ia3], si[ia3], r2, s2, inv)
        if kind == "first":
            o0 = o0x, o0y
            o1, o2, o3 = [(_wrap32(o[0] << 1), _wrap32(o[1] << 1)) for o in (o1, o2, o3)]
        else:
            o0 = o0x >> 2, o0y >> 2
            o1, o2, o3 = [(o[0] >> 1, o[1] >> 1) for o in (o1, o2, o3)]
        for idx, o in ((i0, o0), (i1, o1), (i2, o2), (i3, o3)):
            x[:, idx], y[:, idx] = o


def _mult_r(x, y):
    """mult_32x32_keep32_R: (q31_t) (((q63_t) x * y + 0x80000000) >> 32)"""
    return _wrap32((x * y + 0x80000000) >> 32)


def _mult_acc_r(a, x, y):
    """multAcc_32x32_keep32_R: (q31_t) ((((q63_t) a) << 32) + ((q63_t) x * y) + 0x80000000) >> 32)"""
    return _wrap32(((a << 32) + x * y + 0x80000000) >> 32)


def _mult_sub_r(a, x, y):
    """multSub_32x32_keep32_R: (q31_t) ((((q63_t) a) << 32) - ((q63_t) x * y) + 0x80000000) >> 32)"""
    return _wrap32(((a << 32) - x * y + 0x80000000) >> 32)


def cfft_q31(data, ifft=0):
    """arm_cfft_q31 with bitReverseFlag = 1 on data [..., 2 N] int32 (interleaved re, im); returns a new array."""
    data = np.asarray(data, np.int32)
    N = data.shape[-1] // 2
    assert N in SIZES, N
    inv = bool(ifft)
    z = data.reshape(-1, N, 2).astype(np.int64)
    x, y = z[:, :, 0].copy(), z[:, :, 1].copy()
    tw = twiddle_q31(N)
    if N & 0x55555555:
        _radix4_q31(x, y, N, tw, 1, inv)
    else:
        # arm_cfft_radix4by2_{,inverse_}q31: inputs >> 2, rounded products, << 1
        n2 = N >> 1
        cos_v, sin_v = tw[0:2 * n2:2].astype(np.int64), tw[1:2 * n2:2].astype(np.int64)
        xi, yi, xl, yl = x[:, :n2] >> 2, y[:, :n2] >> 2, x[:, n2:] >> 2, y[:, n2:] >> 2
        xt, yt = _wrap32(xi - xl), _wrap32(yi - yl)
        x[:, :n2], y[:, :n2] = _wrap32(xi + xl), _wrap32(yl + yi)
        p0, p1 = _mult_r(xt, cos_v), _mult_r(yt, cos_v)
        if inv:
            p0, p1 = _mult_sub_r(p0, yt, sin_v), _mult_acc_r(p1, xt, sin_v)
        else:
            p0, p1 = _mult_acc_r(p0, yt, sin_v), _mult_sub_r(p1, xt, sin_v)
        x[:, n2:], y[:, n2:] = _wrap32(p0 << 1), _wrap32(p1 << 1)
        for h in (slice(0, n2), slice(n2, N)):
            xh, yh = x[:, h].copy(), y[:, h].copy()
            _radix4_q31(xh, yh, n2, tw, 2, inv)
            x[:, h], y[:, h] = xh, yh
        x, y = _wrap32(x << 1), _wrap32(y << 1)
    p = _bitrev_perm(N)
    out = np.stack([x[:, p], y[:, p]], -1)
    return out.reshape(data.shape).astype(np.int32)


def cfft(kind, data, ifft=0):
    return (cfft_q15 if kind == "q15" else cfft_q31)(data, ifft)
