"""The MSM's large-input paths on skewed, repeated and identity inputs (run on the B200 box: pytest -m gpu).

The engine chooses its most involved code only for large inputs: the radix-partition sort and its direct-to-global placement of overflowing
bins, 1 - 4 batched-affine levels, the dense copy of the x coordinates, the hot-bucket fix-up, streamed pieces of host-buffer calls.  Each
test here reaches one of these regimes with its automatic choice (or with a forced window size where only that reaches the path), asserts
from the engine's reported shape that it did, and compares the result with (sum_i k_i s_i) * G: the bases are drawn from a pool of points
k_j * G, their negations and duplicates, with identity bases mixed in (test_msm_scale_inputs.py).  No CPU MSM runs at these sizes."""
import numpy as np
import pytest
from conftest import same_affine
from test_msm_scale_inputs import SCALARS_MONTGOMERY, checksum, make_bases, make_scalars, scalar_modulus

from oracle import oracle as A
from oracle import pyref as B

pytestmark = pytest.mark.gpu

NAMES = {A.BN254_G1: "g1", A.GRUMPKIN: "grumpkin", A.BN254_G2: "g2"}


@pytest.fixture(scope="module")
def k():
    import kogarashi_b200 as kk
    kk.init()
    yield kk
    kk.set_param("window_bits", 0)
    kk.set_param("oneshot_split", 0)


# ---- what the engine ran, from its reported shape ------------------------------------------------------------------------------------
SMEM_OPTIN = 227 * 1024   # shared memory one block of a B200 may opt in to (cudaDevAttrMaxSharedMemoryPerBlockOptin)


def sort_plan(n, c, W, nseg):
    """LaunchSort::plan (kernels_sort.cu) restated: (coarse bins per segment, shared-memory capacity of a bin in k_sort_buckets), or None
    when the plan is refused and the counting sort runs instead."""
    if c < 2:
        return None
    bits, per_seg = c - 1, n * W // nseg
    lb = 0
    while lb < bits and (per_seg >> lb) > 16384:
        lb += 1
    if lb > 11:
        lb = 11
        while lb < bits and (per_seg >> lb) > 32768:
            lb += 1
    if bits > lb + 8:
        lb = bits - 8
    if lb > 12:
        return None
    nbins, tile = 1 << lb, 32768 if lb > 11 else 16384
    expect = per_seg >> lb
    cap = min(40960, max(4096, expect + expect // 4 + 1024))
    if nseg * nbins * 4 > SMEM_OPTIN - 1024 or (3 * nbins + 1) * 4 + tile * 5 > SMEM_OPTIN - 1024:
        return None
    return nbins, cap


def regime(k, curve, n, table=False):
    """The last MSM on device 0, made in one piece: its shape (c, W, n) as the engine reports it, and the sort, the number of batched-affine
    levels and the dense-x setting that the automatic choices of enqueue_msm (msm.cu) make for that shape."""
    shape = k.last_timing(0)[1]
    c, W, Bk = shape["c"], shape["W"], shape["B"]
    assert shape["n"] == n, shape
    M = n * W                                   # (scalar, window) entries
    G = Bk if table else W * Bk                 # buckets: one set shared by the windows of a precomputed table
    plan = sort_plan(n, c, W, 1 if table else W)
    sort = "radix" if M >= 1 << 21 and plan else "window_major" if M * 4 > 96 << 20 else "counting"
    levels = 0
    if curve != A.BN254_G2:                     # Fq2 coordinates take no batched-affine levels
        per = M / G
        levels = 0 if M < 8_000_000 or per < 16 else 1 if M < 12_000_000 else 2 if M < 30_000_000 else 4 if per >= 128 else 3
    dense_x = levels > 0 and not table and (1 << 20) < n <= (1 << 24)
    r = dict(c=c, W=W, n=n, M=M, sort=sort, levels=levels, dense_x=dense_x, plan=plan)
    print(f"[regime] {NAMES[curve]}{' table' if table else ''}: c={c} W={W} n={n} entries={M} sort={sort} levels={levels} dense_x={dense_x}")
    return r


def assert_regime(r, want, what):
    got = {key: r[key] for key in want}
    assert got == want, f"{what}: expected {want}, the reported shape c={r['c']} W={r['W']} n={r['n']} ({r['M']} entries) gives {got}"


# ---- 1. automatic regimes, registered bases ------------------------------------------------------------------------------------------
# Host scalars reach the engine in one piece below 2^22 pairs; the 2^23-point case passes them in device memory (a host-buffer call of that
# size is streamed in pieces, each with its own shape), which is also how the bench's headline path calls the engine.
AUTO = [
    (100_003, dict(sort="counting", levels=0, dense_x=False), ()),
    ((1 << 18) + 4321, dict(sort="radix", levels=0, dense_x=False), ()),
    ((1 << 19) + 777, dict(sort="radix", levels=1, dense_x=False), ()),
    (1 << 20, dict(sort="radix", levels=2, dense_x=False), ()),
    ((1 << 20) + 1, dict(sort="radix", levels=2, dense_x=True), ()),
    ((1 << 21) + 3, dict(sort="radix", levels=3, dense_x=True), ("small", "canonical_unreduced")),
    ((1 << 23) + 5, dict(sort="radix", levels=4, dense_x=True), ("uniform", "rm1")),
]
LARGEST = AUTO[-1][0]


def _auto_id(case):
    n, want, _ = case
    return f"{n}-{want['sort']}-l{want['levels']}{'-densex' if want['dense_x'] else ''}"


def _device_commit(curve, bases, sc):
    from kogarashi_b200.nova import DeviceVec
    v = DeviceVec(A.SCALAR_FIELD[curve], sc)
    try:
        return v.commit(bases)
    finally:
        v.free()


@pytest.mark.parametrize("case", AUTO, ids=_auto_id)
@pytest.mark.parametrize("curve", [A.BN254_G1, A.GRUMPKIN], ids=["g1", "grumpkin"])
def test_auto_regimes_checksum(k, curve, case):
    n, want, extra = case
    pts, inf, ks = make_bases(curve, n, seed=n)
    bases = k.Bases(curve, pts, inf)
    del pts
    try:
        for j, mix in enumerate(("nova", "one_bucket") + extra):
            sc, fmt, sc_mont = make_scalars(curve, mix, n, seed=10 * n + j)
            if n >= 1 << 22:
                assert fmt == SCALARS_MONTGOMERY
                got = _device_commit(curve, bases, sc)
            else:
                got = k.to_affine(curve, k.msm_curve_addition(bases, sc, scalar_fmt=fmt))
            assert_regime(regime(k, curve, n), want, mix)
            assert same_affine(got, checksum(curve, ks, sc_mont)), (NAMES[curve], n, mix)
    finally:
        bases.free()


# ---- 2. the same inputs through every entry point ------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [A.BN254_G1, A.GRUMPKIN], ids=["g1", "grumpkin"])
def test_entry_points_checksum(k, curve):
    """kgr_msm (host scalars, streamed in pieces at this size), kgr_msm_device on a torch tensor, kgr_pedersen_commit_vec on a DeviceVec,
    kgr_msm_oneshot (automatic pieces and three), kgr_msm_batch with two large jobs and a small one: the same element for Nova-shaped scalars."""
    import torch
    n = LARGEST
    pts, inf, ks = make_bases(curve, n, seed=n + 1)
    sc, _, _ = make_scalars(curve, "nova", n, seed=7)
    exp = checksum(curve, ks, sc)
    bases = k.Bases(curve, pts, inf)
    try:
        assert same_affine(k.to_affine(curve, k.msm_curve_addition(bases, sc)), exp), "kgr_msm"
        d_sc = torch.from_numpy(sc.view(np.int64)).cuda()
        torch.cuda.synchronize()
        assert same_affine(k.to_affine(curve, k.msm_device(bases, d_sc.data_ptr(), n)), exp), "kgr_msm_device"
        assert_regime(regime(k, curve, n), dict(sort="radix", levels=4, dense_x=True), "kgr_msm_device")
        del d_sc
        assert same_affine(_device_commit(curve, bases, sc), exp), "kgr_pedersen_commit_vec"
        for pieces in (0, 3):
            k.set_param("oneshot_split", pieces)
            assert same_affine(k.to_affine(curve, k.msm_curve_addition(pts, sc, curve=curve, inf=inf)), exp), ("kgr_msm_oneshot", pieces)
        k.set_param("oneshot_split", 0)
        sc2, _, _ = make_scalars(curve, "one_bucket", n, seed=8)
        m = 1000
        sc3, _, _ = make_scalars(curve, "small", m, seed=9)
        small = k.Bases(curve, pts[:m], inf[:m])
        try:
            got = k.msm_batch([(bases, sc), (bases, sc2), (small, sc3)])
        finally:
            small.free()
        for g, want, what in zip(got, (exp, checksum(curve, ks, sc2), checksum(curve, ks[:m], sc3)), ("nova", "one_bucket", "small")):
            assert same_affine(k.to_affine(curve, g), want), ("kgr_msm_batch", what)
    finally:
        k.set_param("oneshot_split", 0)
        bases.free()


def _same_digit_scalar(c, p):
    """A scalar whose signed c-bit digits are all the same d < 2^(c-1) (no carries) in every window it reaches: with a precomputed table,
    whose windows share one bucket set, every one of its n * (windows) entries lands in the same bucket."""
    d = (0x2B5 % (1 << (c - 1))) | 1
    s, w = 0, 0
    while (w + 1) * c < p.bit_length() - 1:
        s += d << (w * c)
        w += 1
    return s, w


@pytest.mark.parametrize("curve", [A.BN254_G1, A.GRUMPKIN], ids=["g1", "grumpkin"])
def test_precomputed_table_checksum_2p20(k, curve):
    """precompute(0) at 2^20 with Nova-shaped scalars, one bucket per window, and one bucket for the whole call: the longest hot bucket the
    fix-up meets, cut into more pieces than k_fixup_long's capped number of slices holds at their nominal length (FL_SLICE * FL_MAX_SLICES),
    so every slice sums many more pieces than that."""
    n = 1 << 20
    pts, inf, ks = make_bases(curve, n, seed=n + 2)
    bases = k.Bases(curve, pts, inf).precompute(0)
    del pts
    try:
        for j, mix in enumerate(("nova", "one_bucket")):
            sc, _, _ = make_scalars(curve, mix, n, seed=20 + j)
            got = k.to_affine(curve, k.msm_curve_addition(bases, sc))
            r = regime(k, curve, n, table=True)
            assert_regime(r, dict(sort="radix", levels=2, dense_x=False), mix)
            assert same_affine(got, checksum(curve, ks, sc)), mix
        p = scalar_modulus(curve)
        s, windows = _same_digit_scalar(r["c"], p)
        assert windows >= r["W"] - 2
        sc = np.tile(np.array(B.int_to_limbs(B.to_mont(s, p)), dtype=np.uint64), (n, 1))
        got = k.to_affine(curve, k.msm_curve_addition(bases, sc))
        assert_regime(regime(k, curve, n, table=True), dict(sort="radix", levels=2, dense_x=False), "same digit")
        assert same_affine(got, checksum(curve, ks, sc)), "same digit in every window"
    finally:
        bases.free()


# ---- 3. the sort's fall-backs under skew (forced window sizes) -----------------------------------------------------------------------
FORCED = [
    # more than 4096 coarse bins per window: the plan is refused; above 96 MB of digits the window-major counting sort runs, below the plain one
    (A.BN254_G1, (1 << 21) + 4096, 22, "nova", dict(sort="window_major", levels=0)),
    (A.GRUMPKIN, 1 << 20, 22, "one_bucket", dict(sort="counting", levels=0)),
    # a hot bin larger than the shared-memory buffer of k_sort_buckets: placed straight into global memory (with four affine levels at c = 12)
    (A.BN254_G1, (1 << 21) + 99, 12, "nova", dict(sort="radix", levels=4)),
    (A.GRUMPKIN, 1 << 21, 20, "one_bucket", dict(sort="radix", levels=0)),
]


@pytest.mark.parametrize("curve,n,c,mix,want", FORCED, ids=[f"{NAMES[f[0]]}-{f[1]}-c{f[2]}-{f[3]}-{f[4]['sort']}" for f in FORCED])
def test_sort_fallbacks_under_skew(k, curve, n, c, mix, want):
    pts, inf, ks = make_bases(curve, n, seed=n + c)
    bases = k.Bases(curve, pts, inf)
    del pts
    sc, _, _ = make_scalars(curve, mix, n, seed=c)
    k.set_param("window_bits", c)
    try:
        got = k.to_affine(curve, k.msm_curve_addition(bases, sc))
        r = regime(k, curve, n)
    finally:
        k.set_param("window_bits", 0)
        bases.free()
    assert r["c"] == c
    assert_regime(r, want, f"window_bits {c}")
    if want["sort"] == "radix":
        # every scalar 1 (nova) or every scalar (one_bucket) puts its entry into the same bucket of window 0: that bin alone exceeds the buffer
        one = A.field_op(A.SCALAR_FIELD[curve], "to_mont", np.array([1, 0, 0, 0], dtype=np.uint64))
        hot = int((sc == one).all(axis=1).sum()) if mix == "nova" else n
        assert hot > r["plan"][1], (hot, r["plan"])
    assert same_affine(got, checksum(curve, ks, sc)), (NAMES[curve], n, c, mix)


# ---- 4. G2 at 2^20 -------------------------------------------------------------------------------------------------------------------
def test_g2_checksum_2p20(k):
    """G2 takes no affine levels, but the radix-partition sort, the hot-bucket fix-up and (host buffers) the streamed pieces."""
    curve, n = A.BN254_G2, 1 << 20
    pts, inf, ks = make_bases(curve, n, seed=n + 3)
    bases = k.Bases(curve, pts, inf)
    try:
        for j, mix in enumerate(("nova", "one_bucket")):
            sc, _, _ = make_scalars(curve, mix, n, seed=30 + j)
            exp = checksum(curve, ks, sc)
            assert same_affine(k.to_affine(curve, k.msm_curve_addition(bases, sc)), exp), (mix, "registered")
            assert_regime(regime(k, curve, n), dict(sort="radix", levels=0), mix)
            assert same_affine(k.to_affine(curve, k.msm_curve_addition(pts, sc, curve=curve, inf=inf)), exp), (mix, "oneshot")
    finally:
        bases.free()
