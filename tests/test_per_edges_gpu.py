"""Edges of the PER SumTree kernels (csrc/gmz_per.cu) that test_per_gpu.py does not reach: update calls longer than one
kernel chunk (PER_MAX_CHUNK = 2048), whole-warp groups on one node, trees deeper than 20 levels, adds longer than the
ring, sampling batches above 1024 with zero leaves and extreme priorities, float drift after long update sequences,
the update_priorities formula, and out-of-range tree indices and capacities.

Two references:
  * oracle.SumTree (sequential add / update / sample, pinned to the reference KAT by test_oracle_golden.py), bit for bit;
  * exact restatements -- integer multiples of 2^-1074, Fractions, double-double sums -- for what the oracle cannot
    check because it shares the kernels' formulation: that a sampled leaf contains its draw, how far the IS weights are
    from the exact ratio, and how far the tree's sums have drifted from the sums of their leaves.
"""
import ctypes as C
import math
from fractions import Fraction
from itertools import accumulate

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CHUNK = 2048                 # PER_MAX_CHUNK in gmz_per.cu
GUARD = 64                   # float64 guard elements on each side of a guarded tree
GUARD_BITS = 0x7FF4DEADBEEF1234


def _rb():
    from datou_gomoku_muzero_b200 import replay_buffer as rb
    return rb


def _oracle():
    from oracle import oracle as O
    return O


def _internal_levels(cap):
    """Internal nodes 0 .. cap-2 grouped by depth, deepest level first (a level's children are done before it)."""
    levels, d = [], 0
    while (1 << d) - 1 < cap - 1:
        levels.append(np.arange((1 << d) - 1, min((1 << (d + 1)) - 1, cap - 1)))
        d += 1
    return levels[::-1]


def _seed_tree(cap, rs, zero_frac=0.05):
    """A populated tree: leaves |N(0,1)| over six decades (some exactly zero), every internal node the float64 sum of its
    children.  Update semantics only add to what is there, so any such state is a fair start for both trees."""
    t = np.zeros(2 * cap - 1)
    leaves = np.abs(rs.randn(cap)) * 10.0 ** rs.uniform(-3, 3, cap)
    leaves[rs.random_sample(cap) < zero_frac] = 0.0
    t[cap - 1:] = leaves
    for ks in _internal_levels(cap):
        t[ks] = t[2 * ks + 1] + t[2 * ks + 2]
    return t


def _pair(cap, t):
    """(device SumTree, oracle SumTree) holding the same tree `t`."""
    import torch
    gt, ot = _rb().SumTree(cap), _oracle().SumTree(cap)
    gt.tree.copy_(torch.from_numpy(t))
    ot.tree[:] = t
    return gt, ot


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def _guarded(st):
    """Re-seat st.tree as a view into a larger float64 buffer whose GUARD elements before and after hold GUARD_BITS."""
    import torch
    n = st.tree.numel()
    big = torch.full((n + 2 * GUARD,), GUARD_BITS, dtype=torch.int64, device=st.device)
    st.tree = big.view(torch.float64)[GUARD:GUARD + n]
    return big


def _guards_intact(big):
    g = big.cpu().numpy()
    return bool((g[:GUARD] == GUARD_BITS).all() and (g[-GUARD:] == GUARD_BITS).all())


# ---------------------------------------------------------------------------------------------------------- updates
def _update_batch(cap, n, rs):
    """n leaf indices with the patterns the update kernel groups by: repeats of one leaf on both sides of every chunk
    boundary, one leaf in all 32 lanes of a warp group, an aligned block of 32 consecutive leaves (one complete 5-level
    subtree: lanes pair up, then quads, ... up to one 32-lane group on every ancestor above it), a block that straddles
    two subtrees (and, when the capacity is not a power of two, the two leaf levels), plus uniform random leaves."""
    first = cap - 1
    idx = rs.randint(0, cap, n) + first
    groups = n // 32
    for g in {1, groups // 2, CHUNK // 32 - 1}:                     # whole warp on one leaf; one group ends a chunk
        if g < groups:
            idx[32 * g:32 * g + 32] = idx[32 * g]
    if cap >= 64:
        aligned = ((first + 1 + 31) // 32) * 32 - 1                 # (k + 1) % 32 == 0: a complete 32-leaf subtree
        deep = (1 << int(math.log2(2 * cap - 1))) - 1               # first leaf of the deepest level
        straddle = max(first, min(deep - 16, 2 * cap - 33)) if deep > first else aligned + 16
        for g, start in zip((2, 3, groups - 1, CHUNK // 32 + 2), (aligned, straddle) * 2):
            if g < groups and start + 31 <= 2 * cap - 2:
                idx[32 * g:32 * g + 32] = np.arange(start, start + 32)
    for b in range(CHUNK, n, CHUNK):                                # L x L | L L across each chunk boundary
        for j in (b - 2, b, b + 1):
            if j < n:
                idx[j] = idx[b - 2]
    pr = np.abs(rs.randn(n)) * 10.0 ** rs.uniform(-3, 3, n)
    pr[rs.random_sample(n) < 0.03] = 0.0
    return idx, pr


@pytest.mark.parametrize("cap", [1, 2, 3, 37, 4096, 4097, (1 << 22) + 3])
def test_chunked_updates_match_sequential_updates(cap):
    """gmz_per_update with more updates than one chunk holds, so the batch spans 2 .. 5 launches; 2^22 + 3 leaves put the
    deepest leaves at depth 23, so warps past 20 do work.  The tree must equal the oracle's after every call."""
    import torch
    rs = np.random.RandomState(cap % 100_003)
    gt, ot = _pair(cap, _seed_tree(cap, rs))
    for n in (2047, 2048, 2049, 2 * CHUNK + 33, 10_000):
        idx, pr = _update_batch(cap, n, rs)
        if n % 2:
            gt.update_many(idx, pr)                                 # host indices
        else:
            gt.update_many(torch.from_numpy(idx).cuda(), torch.from_numpy(pr).cuda())
        ot.update_batch(idx, pr, 1.0)
        assert _same_bits(gt.tree.cpu().numpy(), ot.tree), (cap, n)


@pytest.mark.parametrize("cap", [1, 2, 37, 64, 1000])
def test_adds_longer_than_the_ring_match_sequential_adds(cap):
    """SumTree.add_many with more priorities than the ring holds (the ring wraps more than once in one call; gmz_per_add
    hands such batches to gmz_per_update), between small and ring-sized calls that take the other paths."""
    rs = np.random.RandomState(1000 + cap)
    gt, ot = _rb().SumTree(cap), _oracle().SumTree(cap)
    sizes = [cap + 1, 7, 3 * cap + 5] + ([64] if cap >= 64 else []) + [2049, 63] + ([cap] if cap >= 64 else []) + [5000, 1]
    for n in sizes:
        pr = np.abs(rs.randn(n)) * 10.0 ** rs.uniform(-3, 3, n)
        gt.add_many(pr)
        for x in pr:
            ot.add(float(x))
        assert (gt.write_ptr, gt.count) == (ot.write_ptr, ot.count), (cap, n)
        assert _same_bits(gt.tree.cpu().numpy(), ot.tree), (cap, n)


# --------------------------------------------------------------------------------------------------------- sampling
def _exact(x):
    """A finite float64 as the integer number of 2^-1074 it holds (exact)."""
    num, den = float(x).as_integer_ratio()
    return num * ((1 << 1074) // den)


def _descent_order(cap):
    """Leaf tree indices left to right, the order get_leaf's descent sees them: with a capacity that is not a power of
    two the deepest level (the last ring positions) lies under the leftmost internal nodes, the level above to its right."""
    deep = (1 << int(math.log2(2 * cap - 1))) - 1
    return np.concatenate([np.arange(deep, 2 * cap - 1), np.arange(cap - 1, deep)])


def _f32(q):
    """A non-negative Fraction rounded once to float32 (nearest, ties to even).  Through float64 that is right unless the
    float64 value sits exactly on a float32 midpoint; then the Fraction decides."""
    d = float(q)
    f = np.float32(d)
    if float(f) != d:
        g = np.nextafter(f, np.float32(np.inf) if d > float(f) else np.float32(0))
        if float(f) + float(g) == 2 * d and Fraction(d) != q:
            hi_, lo_ = (g, f) if float(g) > float(f) else (f, g)
            f = hi_ if q > Fraction(d) else lo_
    return f


def _ulps(a, b):
    """Distance in float32 steps between non-negative float32 arrays."""
    return np.abs(np.asarray(a, np.float32).view(np.int32).astype(np.int64) -
                  np.asarray(b, np.float32).view(np.int32).astype(np.int64))


def check_sample(tree, cap, count, u, beta, idx, pr, w):
    """High-precision checks of one gmz_per_sample result (the oracle pins the bits; this pins what they mean).
    Returns (largest weight error in float32 ulps, draws that sit within the rounding allowance of a boundary)."""
    B = len(u)
    order = _descent_order(cap)
    rank = np.empty(2 * cap - 1, np.int64)
    rank[order] = np.arange(cap)
    ex = [_exact(x) for x in tree]
    hi = list(accumulate(ex[k] for k in order))                    # exact cumulative leaf sums, left to right
    lo = [0] + hi[:-1]
    # how far any stored internal sum is from the exact sum of its leaves
    sums = ex[:]
    for ks in _internal_levels(cap):
        for k in ks:
            sums[k] = sums[2 * k + 1] + sums[2 * k + 2]
    delta = max((abs(sums[k] - ex[k]) for k in range(cap - 1)), default=0)
    total = tree[0]
    depth = int(math.log2(2 * cap - 1))
    # the descent compares against stored sums and subtracts with rounding: per level at most delta + ulp(total)
    tol = (depth + 1) * (delta + _exact(math.ulp(total)))
    segment = total / B
    i = np.arange(B, dtype=np.float64)
    lo_s, hi_s = segment * i, segment * (i + 1)
    v = lo_s + (hi_s - lo_s) * u                                     # the draw, in the kernel's float64 operations
    assert (idx >= cap - 1).all() and (idx <= 2 * cap - 2).all(), "sampled a non-leaf"
    assert _same_bits(pr, tree[idx]), "priority is not the sampled leaf's"
    near = 0
    for b in range(B):
        j, V = int(rank[idx[b]]), _exact(v[b])
        inside = (lo[j] < V <= hi[j]) or (j == 0 and V == 0)
        if not inside:
            # a draw within the descent's rounding of a leaf boundary may take either neighbour (or a zero leaf there)
            assert lo[j] - tol <= V <= hi[j] + tol, (b, j, V, lo[j], hi[j], tol)
            near += 1
    # IS weights: (count * p / total)^-beta / max  ==  (p_min / p)^beta exactly, with p_min the smallest sampled priority
    if beta == 0:
        assert (w == 1.0).all()
        return 0.0, near
    pmin = pr.min()
    with np.errstate(divide="ignore", over="ignore"):
        overflow = not np.isfinite(np.float32(np.power(np.float64(count) * (pmin / total), -beta)))
    if overflow:
        # the largest float32 weight is inf: inf / inf = NaN where the weight overflowed, every other weight / inf = 0
        with np.errstate(divide="ignore", over="ignore"):
            big = ~np.isfinite(np.power(np.float64(count) * (pr / total), -beta).astype(np.float32))
        assert np.isnan(w[big]).all() and (w[~big] == 0).all()
        return 0.0, near
    # The kernel rounds the weight and the max to float32 once each (2^-24 relative apiece), so its quotient is within
    # 2 ulps of the exact ratio before the final rounding; rounding is monotone, so the result is at most 2 float32 steps
    # from the exact ratio rounded once.  beta = 1: the ratio as a Fraction; beta = 0.4: in float64.
    assert np.isfinite(w).all()
    if beta == 1:
        ref = np.array([_f32(Fraction(float(pmin)) / Fraction(float(p))) for p in pr], np.float32)
    else:
        with np.errstate(under="ignore"):
            ref = ((pmin / pr) ** beta).astype(np.float32)
    worst = int(_ulps(w, ref).max())
    assert worst <= 2, (worst, int(np.argmax(_ulps(w, ref))))
    return worst, near


def _sample_scenes(cap, rs):
    """(name, leaf priorities or None for the unfilled tail, count) of each tree the sampling test draws from."""
    pos = np.arange(cap)
    base = np.abs(rs.randn(cap)) * 10.0 ** rs.uniform(-2, 2, cap)
    zeros = base.copy()
    zeros[(pos % 97 == 13) | ((pos > cap // 3) & (pos < cap // 3 + 40))] = 0.0      # zero leaves in the middle
    tail = cap * 3 // 5
    return [("zero leaves", zeros, cap),
            ("count < capacity", base[:tail], tail),                 # the rest of the ring: zero leaves
            ("1e-300 .. 1e300", 10.0 ** rs.uniform(-300, 300, cap), cap),
            ("all 1.0", np.ones(cap), cap),
            ("all 0.1", np.full(cap, 0.1), cap)]


@pytest.mark.parametrize("cap", [4096, 5000])
def test_sampling_edges_match_oracle_and_exact_draws(cap):
    """gmz_per_sample at B up to 4097 (a thread draws several samples; the max runs over all of them), on a power-of-two
    capacity and on one whose leaves sit on two levels, with zero leaves, an unfilled ring, extreme and equal priorities,
    u = 0 and u = 1 - 2^-53, and beta 0, 0.4 and 1."""
    rs = np.random.RandomState(cap)
    worst, near, draws = 0.0, 0, 0
    for name, pri, count in _sample_scenes(cap, rs):
        gt, ot = _rb().SumTree(cap), _oracle().SumTree(cap)
        gt.add_many(pri)
        for x in pri:
            ot.add(float(x))
        tree = gt.tree.cpu().numpy()
        assert _same_bits(tree, ot.tree) and gt.count == ot.count == count, name
        for B in (1, 1023, 1024, 1025, 2048, 4097):
            u = rs.random_sample(B)
            u[0], u[-1] = 0.0, np.nextafter(1.0, 0.0)
            pick = rs.random_sample(B) < 0.1
            u[pick] = np.where(rs.random_sample(int(pick.sum())) < 0.5, 0.0, np.nextafter(1.0, 0.0))
            for beta in (0.0, 0.4, 1.0):
                gi, gp, gw = gt.sample(u, beta)
                oi, op, ow = ot.sample(B, u, beta)
                assert np.array_equal(gi, oi), (name, B, beta)
                assert _same_bits(gp, op), (name, B, beta)
                assert gw.dtype == np.float32 and np.array_equal(gw, ow, equal_nan=True), (name, B, beta)
                assert np.array_equal(np.isinf(gw), np.isinf(ow)), (name, B, beta)
                wu, nb = check_sample(tree, cap, count, u, beta, gi, gp, gw)
                worst, near, draws = max(worst, wu), near + nb, draws + B
    print(f"cap {cap}: {draws} draws, largest IS-weight error {worst:.3f} float32 ulp, {near} draws within the "
          f"rounding allowance of a leaf boundary")


# ------------------------------------------------------------------------------------------------------------ drift
def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def test_tree_drift_after_long_update_sequences_is_bounded():
    """20 rounds of sample(360) + update_priorities on a 1M-leaf tree filled by add_many.  Every node -- the root
    against math.fsum, the others against double-double sums of their leaves -- is within k * ulp(M) of the exact sum
    of its leaves, where k counts the updates that reached it (each brings one rounded change and one rounded +=) and
    M bounds every value it can have held (the sum of each leaf's largest priority)."""
    import torch
    cap, B = 1_000_000, 360
    rs = np.random.RandomState(7)
    gt = _rb().SumTree(cap)
    pri = np.abs(rs.randn(cap)) + 1e-6
    gt.add_many(pri)
    writes = np.ones(cap, np.int64)
    leafmax = pri.copy()
    for _ in range(20):
        idx, _, _ = gt.sample_device(torch.from_numpy(rs.random_sample(B)).cuda(), 0.4)
        td = rs.randn(B).astype(np.float32) * np.float32(rs.choice([1e-3, 1.0, 30.0]))
        newp = (np.abs(td) + np.float32(1e-6)).astype(np.float64)
        gt.update_many(idx, torch.from_numpy(newp).cuda())
        pos = idx.cpu().numpy() - (cap - 1)
        np.add.at(writes, pos, 1)
        np.maximum.at(leafmax, pos, newp)
    t = gt.tree.cpu().numpy()
    root_err, k_root, ratio = check_drift(t, cap, writes, leafmax)
    print(f"1M tree after 20 rounds: |root - fsum| = {root_err:.3e} = {root_err / math.ulp(t[0]):.0f} ulp(root) "
          f"(bound {k_root} ulp); largest node error / bound = {ratio:.2e}")


def check_drift(t, cap, writes, leafmax):
    """Every internal node of tree `t` within k * ulp(M) of the exact sum of its leaves (see the test above).
    Returns (|root - fsum(leaves)|, k at the root, largest error / bound over the internal nodes)."""
    n = 2 * cap - 1
    hi, lo = np.zeros(n), np.zeros(n)
    hi[cap - 1:] = t[cap - 1:]
    k = np.zeros(n, np.int64)
    k[cap - 1:] = writes
    m = np.zeros(n)
    m[cap - 1:] = leafmax
    for ks in _internal_levels(cap):
        l, r = 2 * ks + 1, 2 * ks + 2
        s, e = _two_sum(hi[l], hi[r])
        hi[ks], lo[ks] = _two_sum(s, e + lo[l] + lo[r])
        k[ks] = k[l] + k[r]
        m[ks] = m[l] + m[r]
    inner = np.arange(cap - 1)
    err = np.abs((t[inner] - hi[inner]) - lo[inner])
    bound = k[inner] * np.spacing(m[inner] * (1 + 2.0 ** -40))
    assert (err <= bound).all(), int(np.argmax(err / bound))
    root_fsum = math.fsum(t[cap - 1:])
    assert abs(root_fsum - (hi[0] + lo[0])) <= math.ulp(root_fsum)
    root_err = abs(t[0] - root_fsum)
    assert root_err <= k[0] * math.ulp(m[0]), (root_err, k[0])
    return root_err, int(k[0]), float((err / bound).max())


# -------------------------------------------------------------------------------------------------- update_priorities
TD = np.array([0.0, -0.0, 1e-45, -1e-45, 2.0 ** -140, -1.1754942e-38, 1.1754944e-38, 1.5, -7.25, 3.0e38, -1e-6, 1e-6],
              np.float32)


def _expected_priorities(td, eps):
    """|td| + eps rounded once to float32 (float64 holds both operands' sum to within a rounding that cannot move the
    float32 result: 53 >= 2 * 24 + 2), widened; eps is a Python float, so NumPy's float32 arithmetic rounds it first."""
    return np.float32(np.abs(td).astype(np.float64) + np.float64(np.float32(eps))).astype(np.float64)


@pytest.mark.parametrize("eps", [1e-6, 0.0])
def test_update_priorities_follow_the_reference_formula(eps):
    """InMemoryReplayBuffer / DeviceReplayBuffer.update_priorities with td exactly 0, float32 subnormals and eps = 0:
    the leaves written, the whole tree (oracle) and max_priority."""
    import torch
    from datou_gomoku_muzero_b200.config import config
    rb, O = _rb(), _oracle()
    cap = 64
    rs = np.random.RandomState(3)
    idx = rs.randint(0, cap, len(TD)) + cap - 1
    idx[4] = idx[2]                                                  # a repeated leaf: the later write wins
    want = _expected_priorities(TD, eps)
    saved = config.ENABLE_PER, config.PER_EPSILON
    config.ENABLE_PER, config.PER_EPSILON = True, eps
    try:
        ot = O.SumTree(cap)
        for _ in range(cap):
            ot.add(1.0)
        ot.update_batch(idx, want, 1.0)
        want_max = max(1.0, float(want.max()))

        buf = rb.InMemoryReplayBuffer(cap)
        buf.add_many(list(range(cap)))
        buf.update_priorities(list(idx), TD)
        assert _same_bits(buf.sum_tree.tree.cpu().numpy(), ot.tree)
        assert float(buf.max_priority) == want_max
        buf.add("next")                                              # the next slice enters at max_priority
        assert float(buf.sum_tree.tree[cap - 1]) == want_max

        dbuf = rb.DeviceReplayBuffer(cap, board_size=6)
        dbuf.sum_tree.add_many(torch.ones(cap, dtype=torch.float64, device=dbuf.device))
        dbuf.update_priorities(torch.from_numpy(idx).to(dbuf.device), torch.from_numpy(TD).to(dbuf.device))
        assert _same_bits(dbuf.sum_tree.tree.cpu().numpy(), ot.tree)
        assert float(dbuf.max_priority) == want_max
    finally:
        config.ENABLE_PER, config.PER_EPSILON = saved


# ------------------------------------------------------------------------------------------- out-of-range arguments
def _bad_indices(cap):
    return [-1, -7, 2 * cap - 1, 2 * cap + 40]


@pytest.mark.parametrize("cap", [1, 37, 4097])
def test_device_indices_outside_the_tree_write_nothing(cap):
    """Device-tensor indices are not read back on the host, so the kernel skips those outside [0, 2*capacity - 1): the
    guard regions around the tree keep their bits and the tree equals the oracle's after only the in-range updates.
    Through SumTree.update_many directly and through DeviceReplayBuffer.update_priorities."""
    import torch
    from datou_gomoku_muzero_b200.config import config
    rb = _rb()
    rs = np.random.RandomState(20 + cap)
    t = _seed_tree(cap, rs)
    gt, ot = _pair(cap, t)
    big = _guarded(gt)
    gt.tree.copy_(torch.from_numpy(t))
    idx = rs.randint(0, cap, 100) + cap - 1
    bad = _bad_indices(cap)
    for lane, b in zip((0, 5, 31, 32, 63, 96, 97, 99), bad * 2):      # first / last lanes, the partial last group
        idx[lane] = b
    idx[40:72] = bad[0]                                               # a whole group of one out-of-range index
    idx[70] = bad[2]
    pr = np.abs(rs.randn(100)) + 0.5
    ok = (idx >= 0) & (idx < 2 * cap - 1)
    gt.update_many(torch.from_numpy(idx).cuda(), torch.from_numpy(pr).cuda())
    ot.update_batch(idx[ok], pr[ok], 1.0)
    assert _guards_intact(big)
    assert _same_bits(gt.tree.cpu().numpy(), ot.tree)

    saved = config.ENABLE_PER
    config.ENABLE_PER = True
    try:
        dbuf = rb.DeviceReplayBuffer(cap, board_size=6)
        dbig = _guarded(dbuf.sum_tree)
        dbuf.sum_tree.tree.copy_(torch.from_numpy(ot.tree))
        td = rs.randn(100).astype(np.float32)
        dbuf.update_priorities(torch.from_numpy(idx).cuda(), torch.from_numpy(td).cuda())
        p = (np.abs(td) + np.float32(config.PER_EPSILON)).astype(np.float64)
        ot.update_batch(idx[ok], p[ok], 1.0)
        assert _guards_intact(dbig)
        assert _same_bits(dbuf.sum_tree.tree.cpu().numpy(), ot.tree)
    finally:
        config.ENABLE_PER = saved


def test_host_indices_outside_the_tree_raise_index_error():
    """Indices from host memory are checked before anything reaches the device, as the reference's SumTree.update
    raises IndexError: nothing is written (guards, tree and max_priority keep their values).  Internal-node indices
    stay accepted, as the reference accepts them."""
    import torch
    from datou_gomoku_muzero_b200.config import config
    rb = _rb()
    cap = 37
    rs = np.random.RandomState(5)
    t = _seed_tree(cap, rs)
    gt, ot = _pair(cap, t)
    big = _guarded(gt)
    gt.tree.copy_(torch.from_numpy(t))
    for b in _bad_indices(cap):
        with pytest.raises(IndexError):
            gt.update_many(np.array([cap - 1, b], np.int64), np.array([3.0, 4.0]))
        with pytest.raises(IndexError):
            gt.update_many([cap, b, cap + 1], [1.0, 2.0, 5.0])
        with pytest.raises(IndexError):
            gt.update(b, 2.0)
    assert _guards_intact(big)
    assert _same_bits(gt.tree.cpu().numpy(), t)

    for k in (0, cap - 2, (cap - 2) // 2):                           # internal nodes, one per call
        gt.update_many([k], [123.5])
        ot.update(k, 123.5)
        assert _same_bits(gt.tree.cpu().numpy(), ot.tree), k
    assert _guards_intact(big)

    saved = config.ENABLE_PER
    config.ENABLE_PER = True
    try:
        buf = rb.InMemoryReplayBuffer(cap)
        buf.add_many(list(range(cap)))
        before = buf.sum_tree.tree.cpu().numpy()
        bbig = _guarded(buf.sum_tree)
        buf.sum_tree.tree.copy_(torch.from_numpy(before))
        for b in _bad_indices(cap):
            with pytest.raises(IndexError):
                buf.update_priorities([cap - 1, b], np.array([50.0, 60.0], np.float32))
        assert buf.max_priority == 1.0
        assert _guards_intact(bbig) and _same_bits(buf.sum_tree.tree.cpu().numpy(), before)
    finally:
        config.ENABLE_PER = saved


def test_capacity_above_2_pow_32_is_refused():
    """k_per_update's 32 warps cover tree depths 0..31, so the deepest leaf may be at depth 32: capacity <= 2^32.  All
    three entry points refuse more before looking at the batch size, so even an empty call reports it."""
    import torch
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    P = lambda x: C.c_void_p(x.data_ptr())                           # noqa: E731
    dev = torch.device("cuda")
    tree, u, pr = (torch.zeros(8, dtype=torch.float64, device=dev) for _ in range(3))
    idx = torch.zeros(8, dtype=torch.int64, device=dev)
    w = torch.zeros(8, dtype=torch.float32, device=dev)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    calls = {"gmz_per_update": lambda cap: lib.gmz_per_update(P(tree), cap, P(idx), P(pr), 0, st),
             "gmz_per_add": lambda cap: lib.gmz_per_add(P(tree), cap, 0, P(pr), 0, P(idx), st),
             "gmz_per_sample": lambda cap: lib.gmz_per_sample(P(tree), cap, cap, P(u), 0, 0.4, P(idx), P(pr), P(w), st)}
    for name, call in calls.items():
        assert call(1 << 32) == 0, name
        for cap in ((1 << 32) + 1, 1 << 40):
            assert call(cap) != 0, (name, cap)
            msg = lib.gmz_last_error()
            assert name.encode() in msg and b"capacity" in msg, (name, msg)
    torch.cuda.synchronize()
