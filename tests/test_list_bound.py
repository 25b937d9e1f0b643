"""The host reference of the neighbour lists' rebuild decision (list_bound_ref.py) checked on its own, without a GPU: its
directed roundings against np.nextafter and exact rational arithmetic, at exact squares, values that are exactly a float32,
overflow past FLT_MAX, subnormals and NaN; and hand-worked decisions where 2 D lands exactly on the skin and one ulp either side.
test_list_bound_gpu.py then holds the device to this reference pass by pass."""
import math
from fractions import Fraction

import numpy as np
import pytest

import list_bound_ref as R

F32_TINY = float(np.float32(2.0 ** -149))  # smallest float32 subnormal


def rng_doubles(seed, n, lo=-30, hi=30):
    g = np.random.default_rng(seed)
    return list(g.uniform(1.0, 2.0, n) * np.exp2(g.integers(lo, hi, n)))


def up32(x):
    """float32 neighbour above x (as a Python float)"""
    return float(np.nextafter(np.float32(x), np.float32(np.inf)))


def down32(x):
    return float(np.nextafter(np.float32(x), np.float32(-np.inf)))


def test_f32_round_up_against_nextafter():
    values = rng_doubles(1, 3000, -140, 120)
    values += [float(np.float32(v)) for v in values[:500]]  # exactly a float32: stays itself
    values += [math.nextafter(float(np.float32(v)), math.inf) for v in values[:300]]  # one double ulp above a float32
    values += [math.nextafter(float(np.float32(v)), 0.0) for v in values[:300]]  # one double ulp below
    values += [0.0, F32_TINY, F32_TINY / 2, F32_TINY * 1.5, 1e-46, R.F32_MAX, math.nextafter(R.F32_MAX, math.inf), 1e39, 1e300]
    for x in values:
        c = R.f32_ru(x)
        if x > R.F32_MAX:
            assert c == math.inf, x
            continue
        assert float(np.float32(c)) == c and c >= x, x  # a float32, not below x
        assert down32(c) < x, x  # and the smallest such
        if float(np.float32(x)) == x:
            assert c == x
    assert R.f32_ru(math.inf) == math.inf and math.isnan(R.f32_ru(math.nan))
    assert R.f32_ru(-1e39) == -R.F32_MAX


def test_f32_round_up_of_fractions_between_two_float32():
    """Rationals a hair above a float32 (the double nearest to them IS that float32): rounded up to the next one."""
    for f in (1.0, 3.0, 0.25, R.F32_MAX / 2, F32_TINY, float(np.float32(1e-40)), 2.0 ** 100):
        q = Fraction(f) + Fraction(1, 2 ** 1200)
        assert float(q) == f
        assert R.f32_ru(q) == up32(f)
        assert R.f32_ru(Fraction(f)) == f
        assert R.f32_ru(Fraction(f) - Fraction(1, 2 ** 1200)) == f
    assert R.f32_ru(Fraction(R.F32_MAX) + Fraction(1, 2 ** 1200)) == math.inf


def _two_sum_error(a, b):
    """Knuth's TwoSum: the exact a + b - fl(a + b), as a double"""
    s = a + b
    bv = s - a
    av = s - bv
    return (a - av) + (b - bv)


def test_add_round_up_against_two_sum():
    xs = rng_doubles(2, 2000)
    ys = rng_doubles(3, 2000)
    g = np.random.default_rng(4)
    for a, b in zip(xs, ys):
        if g.random() < 0.3:
            b = -b
        s = a + b
        want = math.nextafter(s, math.inf) if _two_sum_error(a, b) > 0 else s
        assert R.add_ru(a, b) == want, (a, b)
    assert R.add_ru(0.1, 0.5) == math.nextafter(0.1 + 0.5, math.inf)  # 0.1 + 0.5 = 0.6000000000000000055...: nearest is below
    assert R.add_ru(1.0, 2.0 ** -80) == math.nextafter(1.0, 2.0)
    assert R.add_ru(1.0, -(2.0 ** -80)) == 1.0
    assert R.add_ru(R.F64_MAX, R.F64_MAX) == math.inf
    assert R.add_ru(-R.F64_MAX, -R.F64_MAX) == -R.F64_MAX
    assert math.isnan(R.add_ru(0.0, math.nan)) and R.add_ru(1.0, math.inf) == math.inf


def test_mul_and_sqrt_round_up_against_exact_rationals():
    xs = rng_doubles(5, 1500, -500, 500)
    ys = rng_doubles(6, 1500, -500, 500)
    for a, b in zip(xs, ys):
        for f, exact in ((R.mul_ru(a, b), Fraction(a) * Fraction(b)), (R.mul_ru(2.0, a), 2 * Fraction(a))):
            if exact > Fraction(R.F64_MAX):
                assert f == math.inf
                continue
            assert Fraction(f) >= exact and Fraction(math.nextafter(f, -math.inf)) < exact, (a, b)
        r = R.sqrt_ru(a)
        assert Fraction(r) ** 2 >= Fraction(a) and Fraction(math.nextafter(r, 0.0)) ** 2 < Fraction(a), a
    assert R.mul_ru(2.0, 0.3) == 2.0 * 0.3  # doubling is exact
    assert R.mul_ru(0.1, 3.0) == 0.1 * 3.0  # the nearest product already lies above 0.3000000000000000166...
    for k in (1.0, 2.0, 3.0, 2.0 ** -537, 12345.0, 1.5 * 2.0 ** 300):  # exact squares stay exact
        assert R.sqrt_ru(k * k) == k
    assert R.sqrt_ru(2.0) == math.sqrt(2.0)  # the nearest double lies above sqrt(2) ...
    assert R.sqrt_ru(3.0) == math.nextafter(math.sqrt(3.0), math.inf)  # ... and below sqrt(3)
    assert R.sqrt_ru(0.0) == 0.0 and R.sqrt_ru(math.inf) == math.inf
    assert math.isnan(R.sqrt_ru(math.nan)) and math.isnan(R.sqrt_ru(-1.0))


def test_fma_rounds_once():
    a = 1.0 + 2.0 ** -27  # a * a = 1 + 2^-26 + 2^-54
    c = 2.0 ** -53
    assert a * a + c == 1.0 + 2.0 ** -26  # two roundings: the 2^-54 is lost, then a tie goes to even
    assert R.fma_f64(a, a, c) == 1.0 + 2.0 ** -26 + 2.0 ** -52  # one rounding keeps 1.5 * 2^-53
    g = np.random.default_rng(7)
    for a, b, c in zip(rng_doubles(8, 500), rng_doubles(9, 500), rng_doubles(10, 500)):
        c = -c if g.random() < 0.5 else c
        f = R.fma_f64(a, b, c)
        exact = Fraction(a) * Fraction(b) + Fraction(c)
        lo, hi = Fraction(math.nextafter(f, -math.inf)), Fraction(math.nextafter(f, math.inf))
        assert abs(Fraction(f) - exact) <= min(Fraction(f) - lo, hi - Fraction(f)) / 2


def test_displacement_bits_of_one_uav():
    bits = R.disp_bits_one
    assert bits(0.0, 0.0, 0.0) == 0
    assert bits(3.0, 4.0, 0.0) == R.f32_bits(25.0)  # exact square, exactly a float32
    assert bits(0.0, 0.0, -0.5) == R.f32_bits(0.25)
    assert bits(0.1, 0.0, 0.0) == R.f32_bits(R.f32_ru(0.1 * 0.1))
    assert R.bits_f32(bits(0.1, 0.0, 0.0)) >= 0.1 * 0.1
    # d2 exactly a float32 plus a hair: the next float32
    d = 1.0 + 2.0 ** -30  # d^2 = 1 + 2^-29 + 2^-60, above the float32 1.0 by less than its ulp
    assert bits(d, 0.0, 0.0) == R.f32_bits(up32(1.0))
    assert bits(1e20, 0.0, 0.0) == R.INF_BITS  # 1e40 > FLT_MAX
    assert bits(1e200, 0.0, 0.0) == R.INF_BITS  # inf already in double
    assert bits(math.inf, 0.0, 0.0) == R.INF_BITS
    assert bits(math.nan, 0.0, 0.0) == R.NAN_BITS
    assert bits(1e-23, 0.0, 0.0) == 1  # 1e-46: below the smallest float32 subnormal, rounded up to it
    assert bits(2.0 ** -80, 0.0, 0.0) == 1  # 2^-160, exact in double
    assert bits(2.0 ** -70, 0.0, 0.0) == R.f32_bits(2.0 ** -140)  # a subnormal float32, exact


def test_displacement_word_over_a_swarm():
    g = np.random.default_rng(11)
    n = 20000
    x0 = g.uniform(-100, 100, (n, 3))
    x1 = x0 + g.normal(0, 0.02, (n, 3))
    want = max(R.disp_bits_one(*map(float, x1[i] - x0[i])) for i in range(n))
    assert R.disp_bits(x0, x1) == want
    moving = np.ones(n, dtype=bool)
    top = int(np.argmax(((x1 - x0) ** 2).sum(1)))
    moving[top] = False
    assert R.disp_bits(x0, x1, moving) < want
    assert R.disp_bits(x0, x0) == 0
    x1[5, 2] = np.nan
    assert R.disp_bits(x0, x1) == R.NAN_BITS
    x1[5, 2] = 1e30
    assert R.disp_bits(x0, x1) == R.INF_BITS
    # two UAVs whose float64 squared norms differ below a float32 ulp: the maximum is taken over the exact bits
    x0 = np.zeros((3, 3))
    x1 = np.array([[1.0 + 2.0 ** -30, 0, 0], [1.0, 0, 0], [0, 0.5, 0]])
    assert R.disp_bits(x0, x1) == R.f32_bits(up32(1.0))


def test_decision_at_the_skin_and_one_ulp_either_side():
    bits = R.f32_bits(0.25)  # d = 0.5 exactly
    for skin, rebuild in ((1.0, False), (math.nextafter(1.0, 0.0), True), (math.nextafter(1.0, 2.0), False)):
        b = R.ListBound(skin)
        assert b.decide(0) is True  # no lists yet
        assert b.decide(bits) is rebuild, skin
    # D = add_ru(0.1, 0.5) lies one ulp above the nearest 0.1 + 0.5: a round-to-nearest sum would keep these lists
    s = 2.0 * (0.1 + 0.5)
    b = R.ListBound(s)
    b.decide(0)
    b.D = 0.1
    assert b.decide(bits) is True
    b = R.ListBound(2.0 * math.nextafter(0.1 + 0.5, 1.0))
    b.decide(0)
    b.D = 0.1
    assert b.decide(bits) is False
    # d = sqrt_ru of a float32 that is not a square: rounded up, so 2 d can exceed a skin that 2 * sqrt(x) (nearest) meets
    f = float(np.float32(0.3))
    d_near = math.sqrt(f)
    assert R.sqrt_ru(f) == math.nextafter(d_near, 1.0)
    b = R.ListBound(2.0 * d_near)
    b.decide(0)
    assert b.decide(R.f32_bits(f)) is True
    # accumulation: four passes of d = 0.25 reach 2 D = 2 exactly, on the skin; a fifth pass is over it
    b = R.ListBound(2.0)
    b.decide(0)
    assert [b.decide(R.f32_bits(0.0625)) for _ in range(5)] == [False, False, False, False, True]
    assert b.D == 0.0
    # NaN, inf and the unbounded word always rebuild; a zero word never does
    for w in (R.NAN_BITS, R.INF_BITS, R.UNBOUNDED):
        b = R.ListBound(1.0)
        b.decide(0)
        assert b.decide(w) is True and b.D == 0.0
    b = R.ListBound(1e-300)
    b.decide(0)
    assert not any(b.decide(0) for _ in range(10))
    assert R.ListBound(1.0).decide(0, force=False, always=True) and R.ListBound(1.0).decide(0)


def test_host_forced_passes():
    h = R.HostSide(1.0)
    assert h.collide() is True  # the first pass
    small = R.f32_bits(1e-6)
    h.launch(small)
    assert h.collide() is False
    assert h.collide() is True  # a pass without a step
    h.launch(small)
    assert h.collide() is False
    h.launch(small)
    h.launch(small)
    assert h.collide() is True  # two launches between passes
    h.launch(small)
    assert h.collide() is False
    h.launch(small)
    h.touch()
    assert h.word() == R.UNBOUNDED
    assert h.collide() is True  # positions written behind the stepping kernel
    h.launch(small)
    assert h.word() == small
    assert h.collide(peer_bits=[R.UNBOUNDED]) is True  # a peer's word
    h.launch(small)
    assert h.collide(peer_bits=[0, small]) is False


@pytest.mark.parametrize("cell", [3.5, 6.0, 12.0])
def test_skin_of_a_cell(cell):
    """api.cu, set_collision_geometry: R_list just under cell / 2, the skin just under R_list - sqrt(3)."""
    r_list = 0.5 * cell * (1.0 - 1e-6)
    skin = (r_list - 1.7320508075688775) * (1.0 - 1e-6)
    assert 0 < skin < r_list - math.sqrt(3.0)
    b = R.ListBound(skin)
    b.decide(0)
    # the largest per-pass displacement that keeps one list-only pass: 2 sqrt_ru(float32) <= skin
    f = np.float32((skin / 2) ** 2)
    while 2 * R.sqrt_ru(float(f)) > skin:
        f = np.nextafter(f, np.float32(0))
    assert b.decide(R.f32_bits(float(f))) is False
    b = R.ListBound(skin)
    b.decide(0)
    assert b.decide(R.f32_bits(up32(float(f)))) is True
