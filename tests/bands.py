"""Exponent-window bands of one birth-death chain, restated on the host (test helper).

The streaming solver (`solve_shared_t`, `solve_row` in csrc/wva_device.cuh) takes a different path for a state
depending on which exponent window its `p` and the running sum fall in (DESIGN.md §3.1, §3.2).  `chain_bands`
re-runs pass 1 of a chain in float64 with the service rates the oracle computes (so the same bits as the reference)
and reports where the chain goes relative to those windows; `row_bands` does the same for the grid's row solve.
Window tests compare the high 32 bits of a double, exactly as the device does.
"""
from __future__ import annotations

import math
import struct

import numpy as np

f32 = np.float32


def hi(x: float) -> int:
    """High 32 bits of a double (sign, exponent, top of the mantissa)."""
    return struct.unpack("<Q", struct.pack("<d", x))[0] >> 32


def HI(e: int) -> int:
    return (1023 + e) << 20


def exp2(x: float) -> int:
    """E(x) = floor(log2 x) for a positive double; 1024 for inf, -1075 for 0."""
    if x == 0.0:
        return -1075
    if math.isinf(x):
        return 1024
    return math.frexp(x)[1] - 1


K_P_LO = HI(-280)
K_RATE_LO, K_RATE_HI = HI(-60), HI(60)
K_PN_SPAN = 960 << 20


def f32_bits(x) -> int:
    return int(np.asarray(x, np.float32).view(np.uint32))


def rate_below(lam, m) -> bool:
    """lambda clearly below m (16 float32 ulps of margin), as wva_device.cuh's rate_below."""
    return f32_bits(lam) + 16 < f32_bits(m) and float(lam) > 0.0 and float(m) > 0.0


def in_window(x: float, lo: int, hi_: int) -> bool:
    return lo <= hi(x) < hi_


def block_exponents(serv_rate, N, lam, p_hi_exp=880):
    """e_lo / e_hi of one step's factor lambda / servRate and the 4- and 16-step block windows (exponents), as the
    solver derives them from the float32 exponents of lambda, max(servRate) and min(servRate)."""
    s = np.asarray(serv_rate[:N], np.float32)
    smax, smin = f32(s.max()), f32(s.min())
    if not (smin > 0 and smax >= smin):
        return dict(e_lo=None, e_hi=None, blk4=None, blk16=None)
    El, Ex, En = f32_bits(lam) >> 23, f32_bits(smax) >> 23, f32_bits(smin) >> 23
    e_lo, e_hi = El - Ex - 1, El - En + 1
    out = dict(e_lo=e_lo, e_hi=e_hi)
    for name, k in (("blk4", 3), ("blk16", 15)):
        lo_exp, hi_exp = -279 - k * min(e_lo, 0), p_hi_exp - k * max(e_hi, 0)
        out[name] = (lo_exp, hi_exp) if (lo_exp < hi_exp and lo_exp > -1000 and hi_exp > -1000) else None
    return out


def chain_bands(serv_rate, N: int, K: int, lam) -> dict:
    """Pass 1 of MM1ModelStateDependent (p[n+1] = p[n] * lambda / servRate[min(n, N-1)]) for a float32 lambda, with
    the solver's exact early termination, and the bands it touches:

    e_p1, e_peak, e_sum      E(p[1]), E(max p), E(sum); e_peak / e_sum = 1024 when the chain overflows (the reference
                             rescales it)
    j_end                    first state the solver does not visit (K + 1 when the chain runs to the end)
    n_raised                 states in [max(thr, 2^-280), 2^(E(sum) - 960)), the pass-2 band that takes div.rn.f64
                             when E(sum) > 680
    below_lo, subnormal, zero  p fell below 2^-280 / into subnormals / to 0 before the chain could terminate
    rates_ok                 lambda, servRate[0] and servRate[N-1] in [2^-60, 2^60)
    e_lo, e_hi, blk4, blk16  see block_exponents
    n_above                  states with p >= 2^880
    block_straddle           1 to 3 states reach 2^880 and a 4-step block of the head (blocks start at states 1, 5,
                             9, ...) begins and ends below 2^880 around all of them: only the 3 e_hi margin of the
                             block window makes the solver see the peak (and bail)
    """
    s = [float(x) for x in np.asarray(serv_rate[:N], np.float32)]
    lamf = f32(lam)
    lam_d = float(lamf)
    suffix_min = np.minimum.accumulate(np.asarray(serv_rate[:N], np.float32)[::-1])[::-1]
    out = dict(N=N, K=K, lam=lamf)
    out["rates_ok"] = all(in_window(x, K_RATE_LO, K_RATE_HI) for x in (lam_d, s[0], s[N - 1]))
    out.update(block_exponents(serv_rate, N, lamf))
    p = lam_d / s[0]
    p1 = p
    thr_hi = hi(min(1.0, p1) * 2.0 ** -78) if K < (1 << 23) else 0
    lo_eff = max(thr_hi, K_P_LO)
    tail_mono = rate_below(lamf, s[N - 1])
    total = 1.0 + p
    peak = max(1.0, p)
    ps = [p]
    below_lo = subnormal = zero = overflow = False
    n, j_end = 1, K + 1
    while n < K:
        hp = hi(p)
        if hp < lo_eff:
            past_mode = tail_mono if n >= N - 1 else rate_below(lamf, suffix_min[n])
            if hp < thr_hi and past_mode:
                j_end = n + 1
                break
            if p == 0.0:
                zero = True
                j_end = n + 1
                break
            below_lo |= hp < K_P_LO
            subnormal |= p < 2.0 ** -1022
        p = p * lam_d / s[min(n, N - 1)]
        total += p
        ps.append(p)
        n += 1
        if math.isinf(p) or math.isinf(total):
            overflow = True
            break
        peak = max(peak, p)
    out.update(e_p1=exp2(p1), e_peak=1024 if overflow else exp2(peak), e_sum=1024 if overflow else exp2(total),
               j_end=j_end, overflow=overflow, below_lo=below_lo, subnormal=subnormal, zero=zero)
    n_raised = 0
    if not overflow and hi(total) > K_P_LO + K_PN_SPAN:
        lo2 = hi(total) - K_PN_SPAN
        n_raised = sum(1 for q in ps[: j_end - 1] if max(thr_hi, K_P_LO) <= hi(q) < lo2)
    out["n_raised"] = n_raised
    above = [i + 1 for i, q in enumerate(ps) if hi(q) >= HI(880)]
    out["n_above"] = len(above)
    out["block_straddle"] = False
    if 1 <= len(above) <= 3 and above[-1] < N - 1 + 4:
        n0 = 1 + 4 * ((above[0] - 2) // 4)   # the block start before the first state above
        out["block_straddle"] = (n0 < above[0] and n0 + 4 > above[-1] and n0 + 4 <= len(ps)
                                 and hi(ps[n0 - 1]) < HI(880) and hi(ps[n0 + 3]) < HI(880))
    return out


def row_bands(serv_rate, length: int, lam) -> dict:
    """The grid's row chain (solve_row): the head of a `length`-entry table with an unbounded batch.  Reports E(sum),
    E(peak), the state the chain ends at and whether solve_row would share it with the row's cells (the chain ends
    before the table does, on the fast path, with a sum below 2^620)."""
    s = [float(x) for x in np.asarray(serv_rate[:length], np.float32)]
    lamf = f32(lam)
    lam_d = float(lamf)
    nh = length - 1
    suffix_min = np.minimum.accumulate(np.asarray(serv_rate[:length], np.float32)[::-1])[::-1]
    out = dict(length=length, lam=lamf, shared=False, e_sum=None, e_peak=None, j_last=None)
    if not (in_window(lam_d, K_RATE_LO, K_RATE_HI) and in_window(s[0], K_RATE_LO, K_RATE_HI)) or nh < 2:
        return out
    p = lam_d / s[0]
    thr_hi = hi(min(1.0, p) * 2.0 ** -78)
    lo_eff = max(thr_hi, K_P_LO)
    total, peak, n = 1.0 + p, max(1.0, p), 1
    ps = [p]
    while n < nh and lo_eff <= hi(p) < HI(880):
        p = p * lam_d / s[n]
        total += p
        peak = max(peak, p)
        ps.append(p)
        n += 1
    out.update(e_sum=exp2(total), e_peak=exp2(peak), j_last=n)
    if n >= nh:
        return out
    negligible = hi(p) < thr_hi and rate_below(lamf, suffix_min[n])
    if not negligible and p != 0.0:
        return out
    out["sum_ok"] = HI(0) <= hi(total) < HI(620)
    out["shared"] = out["sum_ok"] and all(q == 0.0 or K_P_LO <= hi(q) < HI(880) for q in ps)
    return out
