"""The exactly-rounded helpers of vhr_common.cuh, run on the device through tests/csrc/exact_helpers_harness.cu and compared with plain
IEEE arithmetic: sqrt_exact on every bit pattern, the three shared-reciprocal divisions on a boundary grid, on every divisor significand
at the edges of their fast range and on random bit patterns, the fixed-point filter coordinate of bilinear_setup on every float it
takes, and wrap_repeat / wrap_texel on every int."""
import time

import numpy as np
import pytest
import torch

import exact_helpers_lib as E
import helpers as Hh

pytestmark = pytest.mark.gpu
f32 = np.float32
FLT_MAX = float(np.finfo(f32).max)


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _empty(n, dtype):
    return torch.empty(n, dtype=dtype, device="cuda")


def _sweep(name, *args):
    rep = E.new_report()
    t0 = time.perf_counter()
    E.call(name, *args, rep)
    n, checked, recs = E.read_report(rep)
    print(f"[sweep] {name}{args[:1] if name != 'eh_div_sweep' else ''}: {checked} inputs checked in {time.perf_counter() - t0:.2f} s, {n} mismatches")
    return n, checked, recs


def _same_bits(x, y):
    x, y = np.asarray(x, f32), np.asarray(y, f32)
    return (x.view(np.uint32) == y.view(np.uint32)) | (np.isnan(x) & np.isnan(y))


def _hex(x):
    return f"{float(x)!r} ({int(np.asarray(x, f32).view(np.uint32)):#010x})"


# ---------------------------------------------------------------------------------------------------------------------------------
# sqrt_exact
# ---------------------------------------------------------------------------------------------------------------------------------
def test_sqrt_exact_every_bit_pattern():
    n, checked, recs = _sweep("eh_sqrt_sweep")
    assert checked == 1 << 32
    assert n == 0, [(_hex(np.uint32(x).view(f32)), hex(g), hex(w)) for x, g, w, _ in recs[:8]]


def test_fsqrt_rn_is_numpy_sqrt():
    """Ties the sweep's reference to IEEE: __fsqrt_rn against numpy's float32 sqrt on 2^24 patterns, 2^16 per exponent and sign."""
    rng = np.random.default_rng(11)
    bits = (np.arange(1 << 24, dtype=np.uint32) << np.uint32(8)) | rng.integers(0, 256, 1 << 24, dtype=np.uint32)
    x = bits.view(f32)
    ieee, exact = _empty(x.size, torch.float32), _empty(x.size, torch.float32)
    E.call("eh_sqrt_eval", _t(x), ieee, exact, x.size)
    with np.errstate(invalid="ignore"):
        want = np.sqrt(x)
    for got, what in ((ieee.cpu().numpy(), "__fsqrt_rn"), (exact.cpu().numpy(), "sqrt_exact")):
        ok = _same_bits(got, want)
        bad = np.flatnonzero(~ok)[:8]
        assert ok.all(), (what, [(_hex(x[i]), _hex(got[i]), _hex(want[i])) for i in bad])


# ---------------------------------------------------------------------------------------------------------------------------------
# div_exact, div_exact_flag, div_exact_flag_bounded
# ---------------------------------------------------------------------------------------------------------------------------------
def _in_range(x):
    ax = np.abs(x)
    return (ax >= f32(2.0 ** -40)) & (ax < f32(2.0 ** 40))


def _finite_nonzero(x):
    return (x != 0) & (np.abs(x) <= FLT_MAX)


def _rare_expected(a, w):
    """div_exact_flag's contract: `rare` exactly when both operands are finite and nonzero and one of them lies outside [2^-40, 2^40)."""
    return _finite_nonzero(a) & _finite_nonzero(w) & (~_in_range(a) | ~_in_range(w))


def _rare_expected_bounded(w):
    """div_exact_flag_bounded's (dividend +0 or in range): `rare` exactly when the divisor is finite, nonzero and outside the range."""
    return _finite_nonzero(w) & ~_in_range(w)


def _div_device(a, w):
    n = a.size
    q, qf, qb = (_empty(n, torch.float32) for _ in range(3))
    rf, rb = _empty(n, torch.uint8), _empty(n, torch.uint8)
    E.call("eh_div_eval", _t(a), _t(w), n, q, qf, rf, qb, rb)
    return q.cpu().numpy(), qf.cpu().numpy(), rf.cpu().numpy().astype(bool), qb.cpu().numpy(), rb.cpu().numpy().astype(bool)


def _check_div(a, w, what):
    q, qf, rf, qb, rb = _div_device(a, w)
    with np.errstate(all="ignore"):
        want = a / w
    rare, rare_b = _rare_expected(a, w), _rare_expected_bounded(w)
    bounded = (a.view(np.uint32) == 0) | _in_range(a)          # div_exact_flag_bounded's precondition: +0 or in range
    problems = []
    for name, bad in (("div_exact", ~_same_bits(q, want)),
                      ("div_exact_flag: quotient without rare", ~rf & ~_same_bits(qf, want)),
                      ("div_exact_flag: rare", rf != rare),
                      ("div_exact_flag_bounded: quotient without rare", bounded & ~rb & ~_same_bits(qb, want)),
                      ("div_exact_flag_bounded: rare", bounded & (rb != rare_b))):
        if bad.any():
            i = np.flatnonzero(bad)
            got = {"div_exact": q, "div_exact_flag: quotient without rare": qf, "div_exact_flag_bounded: quotient without rare": qb}.get(name)
            problems.append(f"{name}: {i.size} of {a.size} pairs, e.g. " + "; ".join(
                f"{_hex(a[k])} / {_hex(w[k])} = {_hex(want[k])}" + (f" got {_hex(got[k])}" if got is not None else f" rare expected {(rare_b if 'bounded' in name else rare)[k]}")
                for k in i[:6]))
    print(f"[div] {what}: {a.size} pairs, {int(rare.sum())} expected rare, {len(problems)} contract violations")
    assert not problems, f"{what}:\n" + "\n".join(problems)


def _boundary_values():
    one_ulp = lambda x: [np.nextafter(f32(x), f32(0)), f32(x), np.nextafter(f32(x), f32(np.inf))]
    v = [0.0, np.uint32(1).view(f32), np.uint32(0x007FFFFF).view(f32), np.finfo(f32).tiny, *one_ulp(2.0 ** -40), *one_ulp(2.0 ** 40),
         1.0, 3.0, f32(1) / f32(3), 2.0 ** 126, *one_ulp(3.0e38), FLT_MAX, np.inf, np.nan]
    v = np.array(v, f32)
    return np.concatenate([v, -v])


def test_div_boundary_grid():
    v = _boundary_values()
    a, w = np.repeat(v, v.size), np.tile(v, v.size)
    _check_div(a, w, "boundary grid")


def test_div_every_divisor_significand():
    """Every divisor significand at exponents at the edges of the fast range ([2^-40, 2^40)) and in its middle, over 4096 dividend
    significands at exponents covering the quotient range (subnormal to FLT_MAX), against __fdiv_rn on the device."""
    w_exps = np.array([-41, -40, 0, 39, 40], np.int32) + 127
    a_exps = np.array([0, 1, -41 + 127, -40 + 127, -20 + 127, 127, 20 + 127, 39 + 127, 40 + 127, 254], np.int32)
    n_sig = 4096
    n, checked, recs = _sweep("eh_div_sweep", _t(w_exps), w_exps.size, _t(a_exps), a_exps.size, n_sig)
    assert checked == (1 << 23) * w_exps.size * a_exps.size * n_sig
    fn = {0: "div_exact", 1: "div_exact_flag", 2: "div_exact_flag_bounded"}
    assert n == 0, [f"{fn[k & 3]}{' (flag)' if k & 16 else ''}: {_hex(np.uint32(a).view(f32))} / {_hex(np.uint32(w).view(f32))} "
                    f"got {_hex(np.uint32(g).view(f32))}" for a, w, g, k in recs[:8]]


def test_div_random_bit_patterns():
    rng = np.random.default_rng(7)
    for chunk in range(4):
        a = rng.integers(0, 1 << 32, 1 << 24, dtype=np.uint64).astype(np.uint32).view(f32)
        w = rng.integers(0, 1 << 32, 1 << 24, dtype=np.uint64).astype(np.uint32).view(f32)
        _check_div(a, w, f"random bit patterns, chunk {chunk}")


# ---------------------------------------------------------------------------------------------------------------------------------
# bilinear_setup, wrap_repeat, wrap_texel
# ---------------------------------------------------------------------------------------------------------------------------------
BILINEAR_SIZES = (1, 2, 3, 59, 1920, 4096)


@pytest.mark.parametrize("n", BILINEAR_SIZES)
def test_bilinear_setup_fixed_point_branch_every_float(n):
    bad, checked, recs = _sweep("eh_bilinear_sweep", n)
    assert checked > (1 << 30)
    assert bad == 0, [(_hex(np.uint32(u).view(f32)), hex(g), hex(w)) for u, _, g, w in recs[:8]]


@pytest.mark.parametrize("n", BILINEAR_SIZES)
def test_bilinear_setup_vs_numpy_oracle(n):
    """2^24 random coordinates of the fixed-point range: taps and weight against the oracle's formula restated in numpy."""
    rng = np.random.default_rng(n)
    bits = rng.integers(0, 1 << 32, 1 << 25, dtype=np.uint64).astype(np.uint32).view(f32)
    lim = 16384.0 / n
    u = np.concatenate([bits, rng.uniform(-lim, lim, 1 << 24).astype(f32)])
    t = ((u * f32(n)).astype(f32) - f32(0.5)).astype(f32)
    u = u[np.abs(t) < 16384][: 1 << 24]
    assert u.size == 1 << 24
    i0, i1, a = _empty(u.size, torch.int32), _empty(u.size, torch.int32), _empty(u.size, torch.float32)
    E.call("eh_bilinear_eval", _t(u), n, u.size, i0, i1, a)
    fl, wa, _ = Hh.oracle_bilinear_setup(u, n)
    assert np.array_equal(i0.cpu().numpy(), np.mod(fl, n)) and np.array_equal(i1.cpu().numpy(), np.mod(fl + 1, n))
    assert np.array_equal(a.cpu().numpy().view(np.uint32), wa.view(np.uint32))


@pytest.mark.parametrize("n", (1, 2, 3, 7, 59, 1920, 4096, 16384))
def test_wrap_every_int(n):
    bad, checked, recs = _sweep("eh_wrap_sweep", n)
    assert checked == 1 << 32
    modes = {0: "REPEAT", 1: "MIRRORED_REPEAT", 2: "CLAMP_TO_EDGE", 3: "CLAMP_TO_BORDER", 4: "wrap_repeat"}
    assert bad == 0, [(np.uint32(i).view(np.int32).item(), modes[m], np.uint32(g).view(np.int32).item()) for i, _, m, g in recs[:8]]
