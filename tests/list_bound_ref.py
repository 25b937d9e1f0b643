"""Exact host reference of the neighbour lists' rebuild decision (collide.cu, decide_kernel; step_kernel.cuh, step_uav).

Every stepping launch publishes the float bits of the largest squared displacement |x_end - x_start|^2 of any UAV it stepped,
rounded up, through atomicMax.  The first kernel of every collision pass turns that word into d = sqrt_ru(float(bits)), adds it
into D = add_ru(D, d) and keeps the lists while mul_ru(2, D) <= skin; a rebuild resets D to 0.  The host forces a rebuild
(api.cu, begin_pass) before the first pass and after anything but exactly one stepping launch.

The directed roundings are computed exactly with fractions.Fraction (CPython's float(Fraction) rounds correctly), so this is
the decision bit for bit, not an approximation of it."""
import math
import struct
from fractions import Fraction

import numpy as np

UNBOUNDED = 0xFFFFFFFF  # the word a forced pass, a respawn or a restore writes: a NaN pattern larger than any other
NAN_BITS = 0x7FFFFFFF  # what fabsf(__double2float_ru(NaN)) leaves on the device (the canonical NaN, sign cleared)
INF_BITS = 0x7F800000
F32_MAX = float(np.finfo(np.float32).max)
F64_MAX = float(np.finfo(np.float64).max)


def f32_bits(f):
    return struct.unpack("<I", struct.pack("<f", f))[0]


def bits_f32(b):
    """float32 of the bits, widened to a Python float (exactly)."""
    return struct.unpack("<f", struct.pack("<I", int(b) & 0xFFFFFFFF))[0]


def _nearest_f64(q):
    """Fraction -> double, rounded to nearest (overflow to +-inf as the hardware does)."""
    try:
        return float(q)
    except OverflowError:
        return math.inf if q > 0 else -math.inf


def f32_ru(q):
    """The smallest float32 >= q (a Fraction or a float), as a Python float: __double2float_ru for a double argument."""
    if isinstance(q, float):
        if math.isnan(q) or math.isinf(q):
            return q
        q = Fraction(q)
    if q > Fraction(F32_MAX):
        return math.inf
    if q < -Fraction(F32_MAX):
        return -F32_MAX
    # nearest double, then nearest float32: one of the two float32 that bracket q, whatever the double rounding did
    c = np.float32(float(q))
    if Fraction(float(c)) < q:
        c = np.nextafter(c, np.float32(np.inf))
    return float(c)


def sqrt_ru(x):
    """__dsqrt_ru: the smallest double >= sqrt(x); NaN for NaN and negative x."""
    if math.isnan(x) or x < 0:
        return math.nan
    if math.isinf(x) or x == 0:
        return x
    r = math.sqrt(x)  # correctly rounded to nearest: one of the two doubles that bracket sqrt(x)
    if Fraction(r) ** 2 < Fraction(x):
        r = math.nextafter(r, math.inf)
    return r


def _ru(exact, nearest):
    if nearest == -math.inf:  # a finite result below -DBL_MAX rounds up to -DBL_MAX
        return -F64_MAX
    if not math.isinf(nearest) and Fraction(nearest) < exact:
        return math.nextafter(nearest, math.inf)
    return nearest


def add_ru(a, b):
    """__dadd_ru"""
    if not (math.isfinite(a) and math.isfinite(b)):
        return a + b
    exact = Fraction(a) + Fraction(b)
    return _ru(exact, _nearest_f64(exact))


def mul_ru(a, b):
    """__dmul_ru"""
    if not (math.isfinite(a) and math.isfinite(b)):
        return a * b
    exact = Fraction(a) * Fraction(b)
    return _ru(exact, _nearest_f64(exact))


def fma_f64(a, b, c):
    """fma(a, b, c) in double: the exact a * b + c, rounded once to nearest."""
    if not (math.isfinite(a) and math.isfinite(b) and math.isfinite(c)):
        return a * b + c  # inf / NaN: the single rounding makes no difference
    return _nearest_f64(Fraction(a) * Fraction(b) + Fraction(c))


def disp_bits_one(dx, dy, dz):
    """Bits of one UAV's contribution: fabsf(__double2float_ru(fma(dx, dx, fma(dy, dy, dz * dz))))."""
    d2 = fma_f64(dx, dx, fma_f64(dy, dy, dz * dz))
    if math.isnan(d2):
        return NAN_BITS
    return f32_bits(abs(f32_ru(d2)))


def disp_bits(x0, x1, moving=None):
    """The word one stepping launch publishes: the largest bits over the UAVs it stepped (`moving`: bool mask, None = all) from
    positions x0 before and x1 after the launch, [n][3] float64.  Only the UAVs within a few float32 ulps of the float64 maximum
    are evaluated exactly, so a million UAVs stay cheap."""
    x0 = np.asarray(x0, dtype=np.float64).reshape(-1, 3)
    x1 = np.asarray(x1, dtype=np.float64).reshape(-1, 3)
    if moving is not None:
        x0, x1 = x0[moving], x1[moving]
    if len(x0) == 0:
        return 0
    dd = x1 - x0  # the kernel's double subtractions
    with np.errstate(over="ignore", invalid="ignore"):
        approx = dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1] + dd[:, 2] * dd[:, 2]
    if np.isnan(approx).any():
        return NAN_BITS
    top = float(approx.max())
    if math.isinf(top):
        cand = np.flatnonzero(np.isinf(approx) | (approx >= F32_MAX * (1 - 1e-6)))
    else:
        # the float64 sum is within a few double ulps of the fma chain; a float32 ulp is 2^29 times coarser
        cand = np.flatnonzero(approx >= top * (1 - 1e-6))
    return max(disp_bits_one(*map(float, dd[i])) for i in cand)


class ListBound:
    """decide_kernel's state for one handle: D (sum of the per-launch bounds since the last rebuild) and whether lists exist."""

    def __init__(self, skin):
        self.skin = float(skin)
        self.D = 0.0
        self.valid = False

    def decide(self, bits, force=False, always=False):
        """One pass with displacement word `bits`; True iff it rebuilds."""
        d = sqrt_ru(bits_f32(bits))
        D = add_ru(self.D, d)
        rebuild = always or force or not self.valid or not (mul_ru(2.0, D) <= self.skin)
        if rebuild:
            D = 0.0
            self.valid = True
        self.D = D
        return rebuild


class HostSide:
    """api.cu's bookkeeping around the word: a pass after anything but exactly one stepping launch since the last pass (or after
    positions were written otherwise: set_state(x=...), respawn, the first pass) is forced — the host writes UNBOUNDED into the
    word, which decodes to NaN and fails the bound."""

    def __init__(self, skin):
        self.bound = ListBound(skin)
        self.bits = 0
        self.launches = 0
        self.touched = True

    def launch(self, bits):
        self.bits = max(self.bits, int(bits))
        self.launches += 1

    def touch(self):
        self.touched = True

    def collide(self, peer_bits=()):
        """One pass; `peer_bits`: the words the other ranks sent through the hand-shake.  True iff it rebuilds."""
        forced = self.touched or self.launches != 1
        bits = UNBOUNDED if forced else self.bits
        for b in peer_bits:
            bits = max(bits, int(b))
        self.bits, self.launches, self.touched = 0, 0, False
        return self.bound.decide(bits, force=forced)

    def word(self):
        """The word this rank would send through the hand-shake at its next pass."""
        return UNBOUNDED if (self.touched or self.launches != 1) else self.bits
