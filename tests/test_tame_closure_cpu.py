"""CPU: the closure argument behind the kernels' tame mode (te_math.cuh, idm_update<TAME = true>), checked on the
oracle alone - the oracle is the reference's arithmetic, so this needs no GPU.  For operands inside the tame domain
(finite |x| < 2^40, speeds zero or in [2^-100, cap], leader finite or +inf) one IDM update must give a tame car again:
finite position, speed zero or in [2^-100, cap] and never above max(v, v0 + a rate).  The cap comes from the library's
own host routine (te_tame_speed_cap), which also has to reject archetypes outside the supported ranges."""
import ctypes as C

import numpy as np

from oracle import oracle as orc
from traffic_env_b200 import _lib

ARCH = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 2.0, 1.0, 0.0], np.float32)


def speed_cap(arch, rate=0.5, length=250.0):
    L = _lib.load()
    a = np.ascontiguousarray(arch, np.float32)
    cap = C.c_float(-1.0)
    _lib.check(L.te_tame_speed_cap(a.ctypes.data, float(rate), float(length), C.byref(cap)))
    return float(cap.value)


def test_speed_cap_of_the_reference_archetype_and_rejections():
    assert speed_cap(ARCH) == float(np.float32(2.0 * (13.89 + 3.0 * 0.5)))
    slow = ARCH.copy(); slow[1] = 20.0                       # cars arrive faster than the dynamics ever get
    assert speed_cap(slow) == 40.0
    slow[1] = 40.0                                           # ... so fast that the quotient bound fails: not tame
    assert speed_cap(slow) == 0.0
    for idx, bad in ((5, 0.0), (5, np.inf), (3, np.nan), (8, 0.0), (6, -1.0), (7, 1e9), (4, 100.0), (1, -3.0)):
        a = ARCH.copy(); a[idx] = bad
        assert speed_cap(a) == 0.0, (idx, bad)
    assert speed_cap(ARCH, rate=0.0) == 0.0 and speed_cap(ARCH, length=np.inf) == 0.0
    # a fast archetype: the quotient bound of the closure argument no longer holds (dv could overflow a float) -> not tame
    fast = ARCH.copy(); fast[5] = 3000.0
    assert speed_cap(fast) == 0.0


def test_tame_operands_stay_tame_on_the_oracle():
    cap = np.float32(speed_cap(ARCH))
    lo = np.float32(2.0 ** -100)
    rng = np.random.RandomState(2024)
    n = 1_500_000
    v = np.exp(rng.uniform(np.log(float(lo)), np.log(float(cap)), n)).astype(np.float32).clip(lo, cap)
    v[: n // 2] = rng.uniform(0, float(cap), n // 2).astype(np.float32)
    v[n // 2: n // 2 + 10000] = 0.0
    v[n // 2 + 10000: n // 2 + 20000] = lo
    v[n // 2 + 20000: n // 2 + 30000] = cap
    vl = np.where(rng.rand(n) < 0.3, 0, rng.uniform(0, float(cap), n)).astype(np.float32)
    x = (rng.uniform(-1, 1, n) * np.exp(rng.uniform(np.log(1e-3), np.log(2.0 ** 39), n))).astype(np.float32)
    x[: n // 2] = rng.uniform(-50, 600, n // 2).astype(np.float32)
    ll = np.where(rng.rand(n) < 0.3, 0, 4).astype(np.float32)
    gap = np.exp(rng.uniform(np.log(1e-9), np.log(2.0 ** 39), n)) * np.where(rng.rand(n) < 0.15, -1, 1)
    gap[: n // 4] = rng.uniform(-2, 60, n // 4)
    xl = (x.astype(np.float64) + ll + gap).astype(np.float32)
    xl[1000:30000] = np.inf
    # the worst case: gap exactly -RN_f32(1e-8) and its float neighbours at the speed cap behind a standing leader
    e8 = np.float32(1e-8)
    w = slice(40000, 43000)
    x[w], ll[w], v[w], vl[w] = 0.0, 0.0, cap, 0.0
    xl[w] = np.tile(np.array([-e8, np.nextafter(-e8, np.float32(0)), np.nextafter(-e8, np.float32(-1))], np.float32), 1000)
    v[41500:43000] = rng.uniform(0, float(cap), 1500).astype(np.float32)
    xl = np.where(np.isfinite(xl) & (np.abs(xl) >= 2.0 ** 40), np.float32(2.0 ** 39), xl).astype(np.float32)
    ox, ov = orc.sim_bulk(0.5, xl, vl, ll, x, v, ARCH)
    assert np.isfinite(ox).all() and (np.abs(ox) < 2.0 ** 40 + 2.0 ** 21).all()
    assert ((ov == 0) | ((ov >= lo) & (ov <= cap))).all() and not np.signbit(ov).any()
    assert (ov <= np.maximum(v, np.float32(13.89 + 3.0 * 0.5)) * np.float32(1 + 1e-6)).all()
    assert (ox >= x).all()                                   # the gated position update never moves a car backwards


def test_outside_the_domain_the_reference_itself_leaves_it():
    """Why the cap exists: far above it the float dv = a (1 - p - q^2) overflows and the gated position update makes x NaN."""
    e8 = np.float32(1e-8)
    z = np.zeros(1, np.float32)
    ox, ov = orc.sim_bulk(0.5, np.array([-e8], np.float32), z, z, z.copy(), np.array([1000.0], np.float32), ARCH)
    assert np.isnan(ox).all()
