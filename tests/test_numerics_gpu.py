"""The search's numeric building blocks against high-precision host references.

The end-to-end parity tests compare whole searches; they cannot see a primitive that got slightly worse
on inputs their positions do not reach.  tests/csrc/numerics_probe.cu includes the engine's own headers and applies
each device function elementwise (or per warp), so every bound below is a bound on the code the kernels
run: exp_nonpos (the exact path's exp), the certified select's float32 exp / reciprocal / fixed-point
sums and the error budget they add up to against kCertEps, the order-preserving keys and warp
reductions, and the Gumbel noise of gmz_fill_gumbel and the persistent self-play kernel."""
import ctypes as C
import math
import os
import shutil
import subprocess
from decimal import Decimal, localcontext
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "datou_gomoku_muzero_b200", "csrc")
PROBE_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "numerics_probe.cu")

M64 = (1 << 64) - 1
GOLD, K1, K2 = 0x9E3779B97F4A7C15, 0xBF58476D1CE4E5B9, 0x94D049BB133111EB
U24 = 2.0 ** -24                   # unit roundoff of float32
# exp_approx(d) = ex2.approx(fl(fl(d) * fl(log2 e))): the two roundings of the argument and the rounded constant
# move the exponent by |d| (2^-24 + 2^-24 + |fl(log2 e)/log2 e - 1|), on top of ex2.approx's own relative error.
LOG2E_F32 = float(np.float32(1.4426950408889634))
EXP_APPROX_A = 2.0 ** -22
EXP_APPROX_B = 1.001 * (2 * U24 + abs(LOG2E_F32 / 1.4426950408889634 - 1.0))
CERT_D_MAX = 87.4                  # below -87.34 exp_approx flushes to +0: such a candidate's probability is < 2^-126


# ------------------------------------------------------------------------------------------------ host restatements
def mix64(z):
    z ^= z >> 30; z = (z * K1) & M64
    z ^= z >> 27; z = (z * K2) & M64
    return z ^ (z >> 31)


def _unxorshift(z, s):
    x = z
    for _ in range(64 // s + 1):
        x = z ^ (x >> s)
    return x


def unmix64(z):
    z = _unxorshift(z, 31); z = (z * pow(K2, -1, 1 << 64)) & M64
    z = _unxorshift(z, 27); z = (z * pow(K1, -1, 1 << 64)) & M64
    return _unxorshift(z, 30)


def gumbel_u(seed, counter):
    """The counter -> u mapping of gumbel_at (gmz_play.cuh) in Python floats (IEEE double, round to nearest even)."""
    z = mix64((mix64(seed ^ GOLD) + counter * GOLD) & M64)
    return min((float(z >> 11) + 0.5) * 2.0 ** -53, 1.0 - 2.0 ** -53)


def counter_for(seed, z):
    """The counter whose draw under `seed` is mix64(...) == z (mix64 is a bijection)."""
    return ((unmix64(z) - mix64(seed ^ GOLD)) * pow(GOLD, -1, 1 << 64)) & M64


def f64_key_host(x):
    b = np.asarray(x, np.float64).view(np.uint64)
    return b ^ np.where(b >> np.uint64(63), np.uint64(M64), np.uint64(1 << 63))


def f64_unkey_host(k):
    k = np.asarray(k, np.uint64)
    return (k ^ np.where(k >> np.uint64(63), np.uint64(1 << 63), np.uint64(M64))).view(np.float64)


def _decimal_exp(x, prec=50):
    with localcontext() as ctx:
        ctx.prec = prec
        return Decimal(x).exp()


def _ulp_of_exact(e):
    """ulp of the binade the exact value e > 0 lies in (2^-1074 in the subnormal range)."""
    ex = math.frexp(float(e))[1]
    if Decimal(2) ** (ex - 1) > e:          # float(e) rounded up into the next binade
        ex -= 1
    return Fraction(2) ** max(ex - 53, -1074)


# ------------------------------------------------------------------------------------------------ the probe
@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    from datou_gomoku_muzero_b200 import _build
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = str(tmp_path_factory.mktemp("numerics_probe") / "numerics_probe.so")
    subprocess.check_call([nvcc, *_build.NVCC_FLAGS, "-I", CSRC, "-I", os.path.join(ROOT, "include"), "-shared",
                           PROBE_SRC, "-o", so])
    lib = C.CDLL(so)
    P = C.c_void_p
    for name, n in (("probe_exp_nonpos", 2), ("probe_exp_approx", 2), ("probe_rcp", 3), ("probe_warp_sum_fx", 2),
                    ("probe_warp_sum_f64", 2), ("probe_warp_ext", 4), ("probe_keys", 6)):
        getattr(lib, name).argtypes = [P] * n + [C.c_int]
        getattr(lib, name).restype = C.c_int
    lib.probe_cert_eps.restype = C.c_double
    lib.probe_cert_eps.argtypes = []
    return lib


def _call(fn, args, n):
    rc = fn(*[a.ctypes.data for a in args], n)
    assert rc == 0, f"probe returned {rc}"


def _probe_exp_nonpos(probe, x):
    x = np.ascontiguousarray(x, np.float64); y = np.empty_like(x)
    _call(probe.probe_exp_nonpos, [x, y], len(x))
    return y


def _probe_exp_approx(probe, d):
    d = np.ascontiguousarray(d, np.float64); y = np.empty(len(d), np.float32)
    _call(probe.probe_exp_approx, [d, y], len(d))
    return y


def _probe_rcp(probe, x):
    x = np.ascontiguousarray(x, np.float64); ra = np.empty(len(x), np.float32); rn = np.empty(len(x), np.float64)
    _call(probe.probe_rcp, [x, ra, rn], len(x))
    return ra, rn


def _probe_warp_sum_fx(probe, v):
    v = np.ascontiguousarray(v, np.float32).reshape(-1); y = np.empty_like(v)
    _call(probe.probe_warp_sum_fx, [v, y], len(v))
    return y.reshape(-1, 32)


def _probe_warp_sum_f64(probe, v):
    v = np.ascontiguousarray(v, np.float64).reshape(-1); y = np.empty_like(v)
    _call(probe.probe_warp_sum_f64, [v, y], len(v))
    return y.reshape(-1, 32)


# ------------------------------------------------------------------------------------------------ exp_nonpos
def _exp_nonpos_inputs():
    rs = np.random.RandomState(11)
    ln2 = math.log(2.0)
    parts = [np.linspace(-745.2, 0.0, 20001), -rs.uniform(0, 745.2, 20000), -rs.uniform(0, 1, 5000),
             -10.0 ** rs.uniform(-300, 0, 2000), np.linspace(-745.2, -708.3, 3000)]
    # Cody-Waite: k = rint(x log2 e) switches at x = (k + 1/2) ln 2
    edges = [(k + 0.5) * ln2 for k in range(-1075, 0) if (k + 0.5) * ln2 >= -700.5]
    edges += [-700.0, -708.3964185322641, -709.782712893384, -744.4400719213812, -745.1332191019411]
    near = []
    for e in edges:
        v = e
        for _ in range(4):
            near.append(v); v = np.nextafter(v, -np.inf)
        v = np.nextafter(e, np.inf)
        for _ in range(3):
            near.append(v); v = np.nextafter(v, np.inf)
    parts.append(np.array(near))
    parts.append(np.array([-0.0, 0.0, -5e-324, -2.2250738585072014e-308, -1e-300, -745.2, -np.inf]))
    return np.concatenate(parts)


@pytest.mark.gpu
def test_exp_nonpos_within_one_ulp_and_monotone(probe):
    x = _exp_nonpos_inputs()
    x = x[x <= 0.0]
    y = _probe_exp_nonpos(probe, x)
    worst, worst_x = 0.0, None
    for xi, yi in zip(x.tolist(), y.tolist()):
        if xi == -math.inf:
            assert yi == 0.0
            continue
        e = _decimal_exp(xi)
        err = abs(Fraction(yi) - Fraction(e)) / _ulp_of_exact(e)
        if err > worst:
            worst, worst_x = float(err), xi
    print(f"exp_nonpos: max error {worst:.3f} ulp at x = {worst_x!r}")
    assert worst <= 1.0, (worst, worst_x)
    # monotone non-increasing as x decreases, never negative
    o = np.argsort(x, kind="stable")
    assert np.all(np.diff(y[o]) >= 0.0) and np.all(y >= 0.0)
    # a pure function of x: equal inputs on different lanes give equal bits
    perm = np.random.RandomState(3).permutation(len(x))
    y2 = _probe_exp_nonpos(probe, x[perm])
    assert np.array_equal(y2.view(np.uint64), y[perm].view(np.uint64))


# ------------------------------------------------------------------------------------------------ exp_approx
@pytest.fixture(scope="module")
def exp_approx_meas(probe):
    """(d, y, relative error) of exp_approx over d in [-88, 0]; rel = nan where the exact value is below 2^-126."""
    rs = np.random.RandomState(12)
    d = np.concatenate([-rs.uniform(0, 88, 60000), -rs.uniform(0, 1, 10000), -10.0 ** rs.uniform(-12, 0, 2000),
                        np.linspace(-88, 0, 8801), [0.0, -0.0, -87.33654475055310, -87.33654475055311]])
    y = _probe_exp_approx(probe, d)
    rel = np.full(len(d), np.nan)
    tiny = Fraction(2) ** -126
    with localcontext() as ctx:
        ctx.prec = 40
        for i, (di, yi) in enumerate(zip(d.tolist(), y.tolist())):
            e = Fraction(Decimal(di).exp())
            if e >= tiny:
                rel[i] = float(abs(Fraction(yi) - e) / e)
    return d, y, rel


@pytest.mark.gpu
def test_exp_approx_error_envelope(exp_approx_meas):
    d, y, rel = exp_approx_meas
    ad = np.abs(d)
    env = EXP_APPROX_A + EXP_APPROX_B * ad
    normal = ~np.isnan(rel) & (np.exp(d) >= 2.0 ** -126 * (1 + 2 * env))
    for lo, hi in ((0, 1), (1, 10), (10, 30), (30, 60), (60, 88)):
        m = normal & (ad >= lo) & (ad < hi)
        print(f"exp_approx: |d| in [{lo},{hi}): max rel err {rel[m].max():.3e}, envelope {env[m].max():.3e}")
    bad = normal & (rel > env)
    assert not bad.any(), list(zip(d[bad][:5], rel[bad][:5], env[bad][:5]))
    # results below 2^-126 flush to +0 -- never a subnormal, never -0 or negative
    yb = y.view(np.uint32)
    assert np.all((yb == 0) | (y >= 2.0 ** -126))
    assert np.all(y[np.exp(d) < 2.0 ** -126 * (1 - 2 * env)] == 0.0)
    assert y[d == 0.0].tolist() == [1.0] * int((d == 0.0).sum())
    o = np.argsort(d, kind="stable")
    assert np.all(np.diff(y[o].astype(np.float64)) >= 0.0)


# ------------------------------------------------------------------------------------------------ reciprocals
@pytest.fixture(scope="module")
def rcp_meas(probe):
    rs = np.random.RandomState(13)
    x = np.concatenate([np.arange(1, 32769, dtype=np.float64), 10.0 ** rs.uniform(-3, np.log10(4e4), 50000),
                        rs.uniform(1e-3, 4e4, 50000)])
    ra, rn = _probe_rcp(probe, x)
    ea = max(abs(Fraction(a) * Fraction(float(np.float32(xi))) - 1) for a, xi in zip(ra.tolist(), x.tolist()))
    en = max(abs(Fraction(b) * Fraction(xi) - 1) for b, xi in zip(rn.tolist(), x.tolist()))
    return float(ea), float(en)


@pytest.mark.gpu
def test_rcp_approx_and_newton(rcp_meas):
    ea, en = rcp_meas
    print(f"rcp_approx: max rel err {ea:.3e} (vs 1/float32(x));  rcp_newton: max rel err {en:.3e}")
    assert ea <= 2.0 ** -23
    # (float32 rounding of x + rcp.approx) ~ 1.5 * 2^-23, squared by the Newton step: ~3.2e-14
    assert en <= 4e-14


# ------------------------------------------------------------------------------------------------ warp sums
def _fx_host(v):
    """warp_sum_fx restated: round-half-even to 2^-23 fixed point, exact integer sum, one float32 rounding."""
    q = np.rint(v.astype(np.float64) * 2.0 ** 23).astype(np.int64)
    tot = q.sum(axis=1)
    assert np.all(tot < 2 ** 32), "the 32-bit REDUX would wrap"
    return (tot.astype(np.float64).astype(np.float32) * np.float32(2.0 ** -23)).astype(np.float32)


def _fx_inputs():
    rs = np.random.RandomState(14)
    W = 4096
    # U at NC = 3: every lane a float32 sum of <= 12 exp terms in [0, 1], the best unvisited action's term == 1
    terms = rs.uniform(0, 1, (W, 32, 12)) ** rs.choice([1.0, 4.0, 40.0], (W, 32, 1))
    terms[rs.uniform(size=terms.shape) < 0.3] = 0.0
    terms[:, :, 0][rs.uniform(size=(W, 32)) < 0.05] = 2.0 ** -30
    terms[np.arange(W), rs.randint(0, 32, W), 0] = 1.0
    lanes = np.zeros((W, 32), np.float32)
    for j in range(12):
        lanes = (lanes + terms[:, :, j].astype(np.float32)).astype(np.float32)
    u_shape = lanes
    # the softmax denominator: lane 0 = ef * U (U <= 361), lanes 1..31 = ef <= 1 (a hair above when xs - mx > 0)
    den = rs.uniform(0, 1, (W, 32)).astype(np.float32) ** rs.choice([1.0, 8.0], (W, 1)).astype(np.float32)
    den[:, 0] = (rs.uniform(0, 1, W) * rs.uniform(1, 361, W)).astype(np.float32)
    eps = np.float32(1 + 2.0 ** -20)
    extremes = np.array([[361 * eps] + [eps] * 31, [361.0] + [1.0] * 31, [1.0] + [0.0] * 31,
                         [1.0] + [2.0 ** -24] * 31, [1.0] + [2.0 ** -24 * 3] * 31, [12.0] * 32], np.float32)
    return u_shape, np.concatenate([den, extremes])


@pytest.fixture(scope="module")
def fx_meas(probe):
    out = {}
    for name, v in zip(("U", "denominator"), _fx_inputs()):
        y = _probe_warp_sum_fx(probe, v)
        assert np.all(y == y[:, :1]), "lanes disagree"
        assert np.array_equal(y[:, 0].view(np.uint32), _fx_host(v).view(np.uint32))
        exact = [sum(map(Fraction, row.tolist())) for row in v]
        err = np.array([float(abs(Fraction(a) - s)) for a, s in zip(y[:, 0].tolist(), exact)])
        S = np.array([float(s) for s in exact])
        out[name] = (S, err)
    return out


@pytest.mark.gpu
def test_warp_sum_fx_error(fx_meas):
    for name, (S, err) in fx_meas.items():
        small = S < 2.0
        print(f"warp_sum_fx ({name}): max abs err {err.max():.3e} (total < 2: {err[small].max() if small.any() else 0:.3e});"
              f" max rel err on totals >= 1: {(err / S)[S >= 1].max():.3e}")
        # 2^-23 fixed point: <= 2^-24 per lane; the integer total then rounds once to float32 (exact below 2^24, i.e. total < 2)
        assert np.all(err <= 32 * U24 + U24 * S)
        assert np.all(err[small] <= 32 * U24)


@pytest.mark.gpu
def test_warp_sum_f64_lanes_agree_and_error(probe):
    rs = np.random.RandomState(15)
    W = 2048
    v = rs.choice([-1.0, 1.0], (W, 32)) * 10.0 ** rs.uniform(-20, 20, (W, 32))
    v[: W // 4] = rs.normal(0, 1, (W // 4, 32))
    v[W // 4: W // 2, ::2] = -v[W // 4: W // 2, 1::2] * (1 + 2.0 ** -40)      # heavy cancellation
    y = _probe_warp_sum_f64(probe, v)
    assert np.array_equal(y.view(np.uint64), np.repeat(y[:, :1], 32, 1).view(np.uint64)), "lanes disagree"
    h = v.copy()                                      # the xor butterfly restated in float64
    for o in (16, 8, 4, 2, 1):
        h = h + h[:, np.arange(32) ^ o]
    assert np.array_equal(y.view(np.uint64), h.view(np.uint64))
    worst = 0.0
    for row, s in zip(v, y[:, 0].tolist()):
        exact = sum(map(Fraction, row.tolist()))
        bound = 5 * 2.0 ** -53 * sum(abs(Fraction(t)) for t in row.tolist())
        worst = max(worst, float(abs(Fraction(s) - exact) / bound))
    print(f"warp_sum_f64: max |err| / (2^-53 sum|x|) = {5 * worst:.3f}")
    assert worst <= 1.0


# ------------------------------------------------------------------------------------------------ keys and warp max / min
def _special_doubles():
    f = np.finfo(np.float64)
    return np.array([0.0, -0.0, 5e-324, -5e-324, f.tiny, -f.tiny, f.max, -f.max, np.inf, -np.inf, 1.0, -1.0])


@pytest.mark.gpu
def test_keys_are_order_preserving_bijections(probe):
    rs = np.random.RandomState(16)
    L = 20000
    bits = rs.randint(0, 2 ** 63, L, dtype=np.int64).astype(np.uint64) | (rs.randint(0, 2, L).astype(np.uint64) << np.uint64(63))
    x = np.concatenate([_special_doubles(), bits.view(np.float64), rs.normal(0, 1, 1000)])
    x = x[~np.isnan(x)][:L]
    f = np.finfo(np.float32)
    spf = np.array([0.0, -0.0, 1e-45, -1e-45, f.tiny, -f.tiny, f.max, -f.max, np.inf, -np.inf, 1.0, -1.0], np.float32)
    xf = np.concatenate([spf, rs.randint(0, 2 ** 32, 2 * L, dtype=np.int64).astype(np.uint32).view(np.float32)])
    xf = xf[~np.isnan(xf)][:L]
    x, xf = np.ascontiguousarray(x), np.ascontiguousarray(xf)
    k, back = np.empty(len(x), np.uint64), np.empty(len(x), np.float64)
    kf, backf = np.empty(len(x), np.uint32), np.empty(len(x), np.float32)
    _call(probe.probe_keys, [x, k, back, xf, kf, backf], len(x))
    assert np.array_equal(k, f64_key_host(x))
    assert np.array_equal(back.view(np.uint64), x.view(np.uint64))
    assert np.array_equal(backf.view(np.uint32), xf.view(np.uint32))
    # order: by value, and -0 < +0
    for vals, keys in ((x, k.astype(object)), (xf.astype(np.float64), kf.astype(object))):
        order = sorted(range(len(vals)), key=lambda i: (vals[i], not math.copysign(1.0, vals[i]) < 0))
        ks = [keys[i] for i in order]
        vs = [(vals[i], math.copysign(1.0, vals[i])) for i in order]
        for (va, ka), (vb, kb) in zip(zip(vs, ks), zip(vs[1:], ks[1:])):
            assert (ka < kb) if va != vb else (ka == kb)


@pytest.mark.gpu
def test_warp_max_min_match_host_restatement(probe):
    rs = np.random.RandomState(17)
    sp = _special_doubles()
    W = 1024
    v = rs.normal(0, 1, (W, 32)) * 10.0 ** rs.randint(-300, 300, (W, 1))
    v[: W // 2] = rs.choice(sp, (W // 2, 32))
    v[W // 2: W // 2 + 64] = rs.choice([0.0, -0.0], (64, 32))
    v[W // 2 + 64] = -0.0
    v[W // 2 + 65] = [0.0] + [-0.0] * 31
    v[W // 2 + 66] = -np.inf
    v[W // 2 + 67, :] = 1.0
    v[W // 2 + 67, 31] = np.nextafter(1.0, 2.0)
    v = np.ascontiguousarray(v)
    mx, mn = np.empty_like(v), np.empty_like(v)
    mk = np.empty(v.shape, np.uint64)
    _call(probe.probe_warp_ext, [v, mx, mn, mk], v.size)
    hk = f64_key_host(v).max(axis=1)
    hmx = f64_unkey_host(hk)
    hmn = -f64_unkey_host(f64_key_host(-v).max(axis=1))
    assert np.array_equal(mk, np.repeat(hk[:, None], 32, 1))
    assert np.array_equal(mx.view(np.uint64), np.repeat(hmx[:, None], 32, 1).view(np.uint64))
    assert np.array_equal(mn.view(np.uint64), np.repeat(hmn[:, None], 32, 1).view(np.uint64))
    assert np.all(mx[:, 0] == v.max(axis=1)) and np.all(mn[:, 0] == v.min(axis=1))
    # -0 < +0: a warp of both signed zeros has max +0 and min -0
    z = W // 2 + 65
    assert mx[z, 0] == 0.0 and not np.signbit(mx[z, 0]) and np.signbit(mn[z, 0])
    assert np.signbit(mx[z - 1, 0]) and np.signbit(mn[z - 1, 0])


# ------------------------------------------------------------------------------------------------ the certificate's budget
@pytest.mark.gpu
def test_certified_select_error_budget(probe, exp_approx_meas, rcp_meas, fx_meas):
    """kCertEps against the error of a probability on the certified path (select_interior in gmz_tree.cuh):
    pf = ef * rcp_approx(warp_sum_fx(ef, or ef * U for the unvisited candidate)), ef = exp_approx(xs - mx).
    The near-tie test `sb - s > kCertEps (pb + pf)` is sound when |err(sb - s)| <= err(pb) + err(pf) stays below the
    margin; asserted with a factor 2 to spare."""
    eps = probe.probe_cert_eps()
    d, _, rel = exp_approx_meas
    ok = ~np.isnan(rel)
    assert np.all(rel[ok] <= EXP_APPROX_A + EXP_APPROX_B * np.abs(d[ok]))
    e_rcp, e_newton = rcp_meas

    def env(x):
        return EXP_APPROX_A + EXP_APPROX_B * x

    # A sum of exp terms sum_i e^{d_i} (1 + delta_i), delta_i <= env(|d_i|), with one term at d = 0 (the maximum) and
    # at most n others: its relative error is at most env(W), W the largest e^d-weighted mean of |d| -- attained with
    # all n other terms at one common |d| (stationarity gives |d| = 1 + W for every term).  n = 361 unvisited actions
    # (U) + 31 visited children bounds both U and the denominator.
    n = 392
    x = np.linspace(0.0, 100.0, 1000001)
    W = float(np.max(n * x * np.exp(-x) / (1 + n * np.exp(-x))))
    gamma11 = 11 * U24 / (1 - 11 * U24)
    fx_rel = 32 * U24 + U24                       # on totals >= 1: 2^-24 per lane + the float32 rounding of the total
    for S, err in fx_meas.values():
        assert np.all(err[S >= 1] / S[S >= 1] <= fx_rel)
    e_U = env(W) + gamma11 + fx_rel               # U: exp terms, per-lane float32 sums of <= 12 terms, fixed point
    e_den = env(W) + (e_U + U24) + fx_rel         # ef terms; the unvisited one ef * U (one product rounding); fixed point
    # pf: its own exp at |d| <= CERT_D_MAX, the denominator, rcp_approx of it, the product; the visit terms
    # n / (1 + sumN) share one rcp_newton, whose error is relative to their difference (bounded through pb + pf)
    e_p = env(CERT_D_MAX) + e_den + e_rcp + U24 + 2 * e_newton
    print(f"certified select: W = {W:.3f}, exp_approx at |d| = {CERT_D_MAX}: {env(CERT_D_MAX):.3e}, U: {e_U:.3e}, "
          f"denominator: {e_den:.3e}, per probability: {e_p:.3e}; kCertEps = {eps:.2e} = {eps / e_p:.2f} x that")
    rs = np.random.RandomState(18)
    pb, pf = rs.uniform(0, 1, 10000), rs.uniform(0, 1, 10000)
    assert np.all(2 * (e_p * pb + e_p * pf) < eps * (pb + pf))
    assert 2 * e_p < eps


# ------------------------------------------------------------------------------------------------ Gumbel noise
def test_mix64_inverse_reaches_every_edge_draw():
    """Host side of the edge-draw tests: unmix64 inverts mix64, and the counters built with it hit z >> 11 = v."""
    for z in (0, 1, 12345, GOLD, M64, 1 << 63):
        assert mix64(unmix64(z)) == z and unmix64(mix64(z)) == z
    assert counter_for(7, M64) == 5309084603200359959
    assert mix64((mix64(7 ^ GOLD) + 5309084603200359959 * GOLD) & M64) >> 11 == 2 ** 53 - 1
    # (2^53 - 1) + 0.5 rounds to even, i.e. to 2^53: u would be exactly 1 without the clamp
    assert (float(2 ** 53 - 1) + 0.5) * 2.0 ** -53 == 1.0
    assert gumbel_u(7, 5309084603200359959) == 1.0 - 2.0 ** -53
    # the play-kernel seed: noise counter 0 (game 0, first search, action 0) is that draw
    assert unmix64(unmix64(M64)) ^ GOLD == 2518503608491339079
    assert mix64((mix64(2518503608491339079 ^ GOLD) + 0) & M64) == M64
    # no other draw reaches 1 - 2^-53: (v + 0.5) rounds to an even v or v + 1 once v >= 2^52
    for v in (2 ** 53 - 2, 2 ** 53 - 3, 2 ** 52, 2 ** 52 + 1):
        assert (float(v) + 0.5) * 2.0 ** -53 < 1.0 - 2.0 ** -53


def _gumbel_ref(u):
    with localcontext() as ctx:
        ctx.prec = 50
        return -(-(Decimal(u).ln())).ln()


def _fill_gumbel(n, seed, offset):
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    eng = SearchEngine(1, board_size=6, num_simulations=8)
    out = torch.empty(n, dtype=torch.float64, device=eng.device)
    eng.fill_gumbel(out, seed, offset)
    return out.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("seed,offset,n", [(0, 0, 1000), (77, 12345, 777), (2 ** 64 - 1, 2 ** 64 - 300, 600),
                                           (7, 2 ** 63 - 128, 257)])
def test_fill_gumbel_counter_mapping_and_accuracy(seed, offset, n):
    g = _fill_gumbel(n, seed, offset)
    assert np.all(np.isfinite(g))
    worst = 0.0
    for i, gi in enumerate(g.tolist()):
        ref = _gumbel_ref(gumbel_u(seed, (offset + i) & M64))        # the counter wraps modulo 2^64
        err = abs(Decimal(gi) - ref) / max(Decimal(1), abs(ref))
        worst = max(worst, float(err))
    print(f"fill_gumbel seed {seed} offset {offset}: max |err| / max(1, |g|) = {worst:.3e} = 2^{math.log2(worst or 2.0**-99):.1f}")
    assert worst <= 2.0 ** -50


@pytest.mark.gpu
def test_fill_gumbel_edge_draws_are_finite():
    seed = 7
    for v in (0, 1, 2 ** 52 - 1, 2 ** 52, 2 ** 53 - 2, 2 ** 53 - 1):
        z = (v << 11) | 0x5A5
        c = counter_for(seed, z)
        g = float(_fill_gumbel(1, seed, c)[0])
        assert math.isfinite(g), (v, g)
        ref = _gumbel_ref(gumbel_u(seed, c))
        assert abs(Decimal(g) - ref) <= Decimal(2.0 ** -50) * max(Decimal(1), abs(ref)), (v, g, ref)


@pytest.mark.gpu
def test_fill_gumbel_distribution():
    from scipy import stats
    g = _fill_gumbel(1 << 20, 20260101, 0)
    p = stats.kstest(g, "gumbel_r").pvalue
    print(f"K-S p-value of 2^20 draws against Gumbel(0, 1): {p:.4f}")
    assert p > 1e-3


@pytest.mark.gpu
def test_selfplay_game_through_the_u_equals_one_draw_matches_oracle():
    """noise_seed 2518503608491339079 puts the u = 1 draw at noise counter 0: game 0's first search, action 0.
    The persistent kernel's game must stay finite and equal the oracle's game fed the same noise."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    from oracle import oracle
    from test_selfplay_gpu import _noise_for_game
    N, S, G, seed, nseed = 9, 64, 2, 5, 2518503608491339079
    A = N * N
    eng = SearchEngine(G, board_size=N, num_simulations=S)
    sp = SelfPlayEngine(eng, "e0", seed=seed, noise_seed=nseed)
    traj = TrajectoryStore(eng, extra_slots=4)
    first = []
    for _ in range(8):
        sp.play(moves_per_game=A // 3, traj=traj, restart=True)
        first = [r for r in traj.harvest() if r["game"] == 0][:1]
        if first:
            break
    assert first and first[0]["start_move_count"] == 0
    first = first[0]
    gum = _noise_for_game(eng, 0, first["length"], nseed)
    assert np.all(np.isfinite(gum))
    assert abs(Decimal(gum[0, 0]) - _gumbel_ref(1.0 - 2.0 ** -53)) <= Decimal(2.0 ** -50) * 37
    cfg = oracle.make_config(board_size=N, num_simulations=S, eval_seed=seed, mode=0)
    o = oracle.selfplay_game(cfg, np.concatenate([gum, np.zeros((1, A))]))
    assert o["T"] == first["length"]
    assert np.array_equal(o["actions"], first["actions"]) and o["winner"] == first["winner"]
    assert np.array_equal(o["values"], first["values"])
    np.testing.assert_allclose(first["policies"], o["policies"], rtol=1e-12, atol=1e-15)
