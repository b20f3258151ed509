"""GPU: device arithmetic against the host, bit for bit (through the C-ABI test hooks)."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def _lib():
    from traffic_env_b200 import _lib
    return _lib.load(), _lib


def gpu_powf(x, y):
    L, m = _lib()
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty_like(x)
    m.check(L.te_test_powf(0, x.ctypes.data, float(y), out.ctypes.data, x.size))
    return out


def gpu_idm(rate, arch, xl, vl, ll, x, v):
    L, m = _lib()
    arrs = [np.ascontiguousarray(a, np.float32) for a in (xl, vl, ll, x, v)]
    a = np.ascontiguousarray(arch, np.float32)
    xo, vo = np.empty_like(arrs[0]), np.empty_like(arrs[0])
    m.check(L.te_test_idm(0, float(rate), a.ctypes.data, *[t.ctypes.data for t in arrs], xo.ctypes.data,
                          vo.ctypes.data, arrs[0].size))
    return xo, vo


def same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return ((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b)))


@pytest.mark.parametrize("y", [4.0, 2.5, 1.0, 0.37])
def test_powf_matches_host_libm(y):
    """numba lowers float32 ** float32 to libm powf; the device restates glibc's algorithm."""
    rng = np.random.RandomState(5)
    x = np.concatenate([
        rng.uniform(0, 2, 3_000_000).astype(np.float32),
        (np.abs(rng.standard_normal(500_000)) * 1e-3).astype(np.float32),
        rng.randint(0, 0x7f800000, 2_000_000, dtype=np.int64).astype(np.uint32).view(np.float32),
        np.arange(0, 0x00800000, 4099, dtype=np.uint32).view(np.float32),  # subnormals
        np.array([0, 1e-45, 1e-40, 1.17549435e-38, 1, np.inf, np.nan, 3e38, 0.79985, 13.88 / 13.89], np.float32)])
    got, want = gpu_powf(x, y), orc.powf_bulk(x, y)
    bad = ~same_bits(got, want)
    assert not bad.any(), "first mismatch x=%r got=%r want=%r" % (x[bad][0], got[bad][0], want[bad][0])


def test_powf_all_velocity_ratios():
    """Every float32 in [0, 1.25] that v / v0 can take on a coarse lattice plus its neighbours."""
    base = np.arange(0, np.float32(1.25).view(np.uint32), 257, dtype=np.uint32)
    x = np.concatenate([base, base + 1, base + 2]).view(np.float32)
    got, want = gpu_powf(x, 4.0), orc.powf_bulk(x, 4.0)
    assert same_bits(got, want).all()


def test_idm_update_matches_oracle():
    rng = np.random.RandomState(11)
    n = 2_000_000
    arch = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 2.0, 1.0, 0.0], np.float32)
    x = rng.uniform(-50, 260, n).astype(np.float32)
    gap = np.where(rng.rand(n) < 0.3, rng.uniform(0, 8, n), rng.uniform(0, 300, n))
    xl = (x + gap + 4).astype(np.float32)
    v = np.where(rng.rand(n) < 0.2, 0, rng.uniform(0, 15, n)).astype(np.float32)
    vl = np.where(rng.rand(n) < 0.3, 0, rng.uniform(0, 15, n)).astype(np.float32)
    ll = np.where(rng.rand(n) < 0.2, 0, 4).astype(np.float32)
    # virtual leaders: red light at the road end and free road (+inf), plus collisions (negative gap)
    xl[:50000] = 250.0
    xl[50000:100000] = np.inf
    vl[:100000] = 0
    ll[:100000] = 0
    xl[100000:110000] = x[100000:110000] - 1.0
    v[110000:111000] = 1e-30
    v[111000:112000] = 1e-42
    gx, gv = gpu_idm(0.5, arch, xl, vl, ll, x, v)
    ox, ov = orc.sim_bulk(0.5, xl, vl, ll, x, v, arch)
    bx, bv = ~same_bits(gx, ox), ~same_bits(gv, ov)
    assert not bx.any() and not bv.any(), "x mismatches %d, v mismatches %d" % (bx.sum(), bv.sum())


def test_idm_other_rate_and_archetype():
    rng = np.random.RandomState(12)
    n = 300_000
    arch = np.array([0.0, 8.0, 5.5, 1.7, 3.0, 20.0, 2.3, 1.4, 2.0, 0.0], np.float32)
    x = rng.uniform(0, 500, n).astype(np.float32)
    xl = (x + rng.uniform(0, 100, n)).astype(np.float32)
    v = rng.uniform(0, 25, n).astype(np.float32)
    vl = rng.uniform(0, 25, n).astype(np.float32)
    ll = np.full(n, 5.5, np.float32)
    gx, gv = gpu_idm(0.25, arch, xl, vl, ll, x, v)
    ox, ov = orc.sim_bulk(0.25, xl, vl, ll, x, v, arch)
    assert same_bits(gx, ox).all() and same_bits(gv, ov).all()


def test_philox_block_matches_oracle():
    L, m = _lib()
    rng = np.random.RandomState(3)
    for _ in range(64):
        ctr = rng.randint(0, 2**32, 4, dtype=np.int64).astype(np.uint32)
        key = rng.randint(0, 2**32, 2, dtype=np.int64).astype(np.uint32)
        out = np.empty(4, np.uint32)
        m.check(L.te_test_philox(0, ctr.ctypes.data, key.ctypes.data, out.ctypes.data))
        assert list(out) == orc.philox4x32_10(ctr, key)
    # known-answer vector of the Random123 distribution (philox4x32-10, all-zero counter and key)
    z = np.zeros(4, np.uint32)
    out = np.empty(4, np.uint32)
    m.check(L.te_test_philox(0, z.ctypes.data, z[:2].ctypes.data, out.ctypes.data))
    assert [hex(int(v)) for v in out] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]


def test_idm_adversarial_operands():
    """The branch-free fast path and its generic fallback against the oracle on operands chosen to hit the
    acceptance tests of the division, the underflow / subnormal branches of powf and non-finite state."""
    rng = np.random.RandomState(21)
    n = 6_000_000
    arch = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 2.0, 1.0, 0.0], np.float32)
    x = rng.uniform(-300, 600, n).astype(np.float32)
    v = np.abs(rng.standard_normal(n) * 8).astype(np.float32)
    vl = np.abs(rng.standard_normal(n) * 8).astype(np.float32)
    ll = np.full(n, 4.0, np.float32)
    # gaps over 30 orders of magnitude, both signs, and exact cancellations s + 1e-8 ~ 0
    mag = np.exp(rng.uniform(np.log(1e-12), np.log(1e12), n))
    s = (mag * rng.choice([-1.0, 1.0], n, p=[0.2, 0.8])).astype(np.float32)
    xl = (x.astype(np.float64) + 4.0 + s).astype(np.float32)
    k = n // 10
    xl[:k] = x[:k] + np.float32(4.0)                      # s == 0 exactly
    xl[k:2 * k] = (x[k:2 * k] + np.float32(4.0)) + np.float32(-1e-8)
    v[2 * k:3 * k] = np.exp(rng.uniform(np.log(1e-45), np.log(1e-3), k)).astype(np.float32)   # creeping / subnormal speeds
    v[3 * k:3 * k + 1000] = 0.0
    v[3 * k + 1000:3 * k + 2000] = np.float32(13.89)      # ratio exactly 1
    v[3 * k + 2000:3 * k + 3000] = np.float32(1e30)       # overflowing power
    v[3 * k + 3000:3 * k + 4000] = np.float32(3e38)       # v * T overflows: s_star = inf
    vl[3 * k + 3000:3 * k + 3500] = np.float32(3e38)      # ... with v - vl == 0 (t3 stays finite)
    xl[3 * k + 3000:3 * k + 3250] = np.inf                # ... behind a free road: inf / inf
    special = np.array([np.nan, np.inf, -np.inf, 3e38, -3e38, 0.0, -0.0], np.float32)
    idx = rng.randint(4 * k, n, size=30000)
    x[idx[:10000]] = rng.choice(special, 10000)
    v[idx[10000:20000]] = rng.choice(special, 10000)
    xl[idx[20000:]] = rng.choice(special, 10000)
    gx, gv = gpu_idm(0.5, arch, xl, vl, ll, x, v)
    ox, ov = orc.sim_bulk(0.5, xl, vl, ll, x, v, arch)
    bx, bv = ~same_bits(gx, ox), ~same_bits(gv, ov)
    assert not bx.any() and not bv.any(), "x mismatches %d (first at %s), v mismatches %d" % (
        bx.sum(), np.nonzero(bx)[0][:3], bv.sum())


def test_powf4_filter_exhaustive():
    """Proof by exhaustion of the delta == 4 shortcut: over EVERY non-negative finite float r, whenever the filter
    accepts RN_f32((r*r)*(r*r)) it equals the glibc algorithm's result (which test_powf_* tie to the host libm)."""
    L, m = _lib()
    out = np.zeros(4, np.uint64)
    m.check(L.te_test_powf4_exhaustive(0, 1 << 20, out.ctypes.data))
    differ, max_dist, declined, accepted_but_wrong = (int(v) for v in out)
    assert accepted_but_wrong == 0
    assert 0 < differ < 1_000_000 and max_dist < (1 << 20)     # the shortcut is not vacuous and the margin holds
    # results outside the normal float range (r < 2^-31.5 or r >= 2^32) are declined by construction; of the rest ~0.4 %
    assert declined < 0.76 * 0x7f800000


def test_idm_with_and_without_powf4_shortcut_agree():
    """Same operands through a handle-independent hook with the shortcut disabled (environment switch)."""
    import os
    rng = np.random.RandomState(33)
    n = 1_000_000
    arch = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 2.0, 1.0, 0.0], np.float32)
    x = rng.uniform(0, 250, n).astype(np.float32)
    xl = (x + rng.uniform(4, 120, n)).astype(np.float32)
    v = rng.uniform(0, 15, n).astype(np.float32)
    vl = rng.uniform(0, 15, n).astype(np.float32)
    ll = np.full(n, 4, np.float32)
    a = gpu_idm(0.5, arch, xl, vl, ll, x, v)
    os.environ["TE_NO_POWF4_SHORTCUT"] = "1"
    try:
        b = gpu_idm(0.5, arch, xl, vl, ll, x, v)
    finally:
        del os.environ["TE_NO_POWF4_SHORTCUT"]
    assert same_bits(a[0], b[0]).all() and same_bits(a[1], b[1]).all()


def test_idm_pow2_forms_agree_with_conversions_and_oracle():
    """T and rate powers of two: v * T and rate * v are taken as double products of the widened v (no conversion).
    Same operands with the shortcut disabled (environment switch) and against the oracle, for the reference's
    archetype and for another power-of-two pair, over speeds from subnormal to overflowing."""
    import os
    rng = np.random.RandomState(44)
    n = 1_500_000
    for rate, T in ((0.5, 2.0), (0.25, 4.0), (1.0, 0.5)):
        arch = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, T, 1.0, 0.0], np.float32)
        x = rng.uniform(-100, 400, n).astype(np.float32)
        xl = (x + np.exp(rng.uniform(np.log(1e-6), np.log(1e4), n))).astype(np.float32)
        v = np.exp(rng.uniform(np.log(1e-45), np.log(3e38), n)).astype(np.float32)
        v[: n // 2] = rng.uniform(0, 20, n // 2).astype(np.float32)
        v[n // 2: n // 2 + 5000] = 0.0
        vl = rng.uniform(0, 20, n).astype(np.float32)
        ll = np.full(n, 4, np.float32)
        a = gpu_idm(rate, arch, xl, vl, ll, x, v)
        os.environ["TE_NO_POW2_SHORTCUT"] = "1"
        try:
            b = gpu_idm(rate, arch, xl, vl, ll, x, v)
        finally:
            del os.environ["TE_NO_POW2_SHORTCUT"]
        ox, ov = orc.sim_bulk(rate, xl, vl, ll, x, v, arch)
        assert same_bits(a[0], b[0]).all() and same_bits(a[1], b[1]).all()
        assert same_bits(a[0], ox).all() and same_bits(a[1], ov).all()


def gpu_idm_tame(rate, arch, xl, vl, ll, x, v):
    L, m = _lib()
    arrs = [np.ascontiguousarray(a, np.float32) for a in (xl, vl, ll, x, v)]
    a = np.ascontiguousarray(arch, np.float32)
    xo, vo = np.empty_like(arrs[0]), np.empty_like(arrs[0])
    m.check(L.te_test_idm_tame(0, float(rate), a.ctypes.data, *[t.ctypes.data for t in arrs], xo.ctypes.data,
                               vo.ctypes.data, arrs[0].size))
    return xo, vo


def test_idm_unchecked_form_on_tame_operands():
    """The form the step kernels run while the handle is tame (idm_update<true>: no validity predicate, no generic
    fallback) against the checked form and the oracle, over the whole tame domain and its edges: speeds of 0, 2^-100,
    the handle's speed cap (twice the fastest speed of the dynamics) and log-uniform in between, positions up to 2^40 in magnitude, gaps from overlapping (negative) through
    zero and the -1e-8 neighbourhood to 2^40 and the free road (+inf leader), leader lengths 0 and up to 2^19; and that
    the results are tame again (closed domain: what the kernel relies on tick after tick)."""
    rng = np.random.RandomState(77)
    n = 3_000_000
    arch = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 2.0, 1.0, 0.0], np.float32)
    lo, hi = np.float32(2.0 ** -100), np.float32(2.0 * (13.89 + 3.0 * 0.5))     # tame_archetype's cap
    v = np.exp(rng.uniform(np.log(float(lo)), np.log(float(hi)), n)).astype(np.float32)
    v = np.clip(v, lo, hi)
    v[: n // 2] = rng.uniform(0, 30, n // 2).astype(np.float32)
    v[n // 2: n // 2 + 20000] = 0.0
    v[n // 2 + 20000: n // 2 + 30000] = lo
    v[n // 2 + 30000: n // 2 + 40000] = hi
    v[n // 2 + 40000: n // 2 + 60000] = np.float32(13.89) * (1 + rng.randint(-3, 4, 20000) * np.float32(2.0 ** -23))
    vl = np.where(rng.rand(n) < 0.3, 0, np.exp(rng.uniform(np.log(float(lo)), np.log(float(hi)), n))).astype(np.float32)
    vl[: n // 2] = np.where(rng.rand(n // 2) < 0.3, 0, rng.uniform(0, 30, n // 2)).astype(np.float32)
    x = (rng.uniform(-1, 1, n) * np.exp(rng.uniform(np.log(1e-3), np.log(2.0 ** 39), n))).astype(np.float32)
    x[: n // 2] = rng.uniform(-50, 600, n // 2).astype(np.float32)
    ll = np.where(rng.rand(n) < 0.3, 0, 4).astype(np.float32)
    ll[-5000:] = np.float32(2.0 ** 19)
    gap = np.exp(rng.uniform(np.log(1e-9), np.log(2.0 ** 39), n)) * np.where(rng.rand(n) < 0.15, -1, 1)
    gap[: n // 4] = rng.uniform(-2, 60, n // 4)
    xl = (x.astype(np.float64) + ll + gap).astype(np.float32)
    k = 200000
    xl[k: k + 50000] = np.inf                                   # free road
    xl[k + 50000: k + 100000] = x[k + 50000: k + 100000] + ll[k + 50000: k + 100000]      # gap exactly zero (when exact)
    v[k + 100000: k + 150000] = np.where(rng.rand(50000) < 0.5, hi, v[k + 100000: k + 150000])   # largest s_star there
    vl[k + 100000: k + 150000] = np.where(rng.rand(50000) < 0.5, 0, vl[k + 100000: k + 150000])
    near = (x[k + 100000: k + 150000].astype(np.float64) + ll[k + 100000: k + 150000] - 1e-8)
    xl[k + 100000: k + 150000] = near.astype(np.float32)        # s + 1e-8 as close to zero as floats allow
    # the worst case of the closure argument: gap exactly -RN_f32(1e-8) (|s + 1e-8| = 6.08e-17, the largest quotient) and
    # its float neighbours, at the speed cap behind a standing leader (the largest s_star)
    w = slice(k + 150000, k + 153000)
    x[w], ll[w], v[w], vl[w] = 0.0, 0.0, hi, 0.0
    e8 = np.float32(1e-8)
    xl[w] = np.tile(np.array([-e8, np.nextafter(-e8, np.float32(0)), np.nextafter(-e8, np.float32(-1))], np.float32), 1000)
    v[k + 151500: k + 153000] = rng.uniform(0, float(hi), 1500).astype(np.float32)
    xl = np.where(np.isfinite(xl) & (np.abs(xl) >= 2.0 ** 40), np.float32(2.0 ** 39), xl).astype(np.float32)
    ux, uv = gpu_idm_tame(0.5, arch, xl, vl, ll, x, v)
    cx, cv = gpu_idm(0.5, arch, xl, vl, ll, x, v)
    ox, ov = orc.sim_bulk(0.5, xl, vl, ll, x, v, arch)
    assert same_bits(cx, ox).all() and same_bits(cv, ov).all()
    bx, bv = ~same_bits(ux, ox), ~same_bits(uv, ov)
    assert not bx.any() and not bv.any(), "x mismatches %d, v mismatches %d" % (bx.sum(), bv.sum())
    assert np.isfinite(ux).all() and (np.abs(ux) < 2.0 ** 40 + 2.0 ** 21).all()
    assert ((uv == 0) | ((uv >= lo) & (uv <= hi))).all() and not np.signbit(uv).any()
    assert (uv <= np.maximum(v, np.float32(13.89 + 3.0 * 0.5)) * np.float32(1 + 1e-6)).all()


def test_idm_tame_hook_refuses_an_archetype_without_the_tame_form():
    """te_test_idm_tame runs the compile-time-archetype form, which is only right where the step kernels would run it:
    T = 3 is not a power of two, so the hook refuses instead of returning wrong numbers."""
    from traffic_env_b200._lib import TrafficB200Error
    arch = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 3.0, 1.0, 0.0], np.float32)
    z = np.zeros(16, np.float32)
    with pytest.raises(TrafficB200Error, match="te_test_idm_tame"):
        gpu_idm_tame(0.5, arch, z + 40.0, z, z + 4.0, z, z + 5.0)
