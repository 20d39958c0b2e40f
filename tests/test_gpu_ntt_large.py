"""The Fr NTT at the domain sizes where it runs three shared-memory passes (2^21 .. 2^28), against the restated reference FFT (oracle FrFft =
groth16/src/fft.rs) bit for bit where the oracle is affordable, and against sums evaluated in Python integers everywhere else.

Covers what only happens past 2^20: the third pass of LaunchNtt::transform_bitrev_input, pass offsets (p_shift) of 14 and more in k_ntt_pass,
twiddle indices of 2^20 and more, the 2^28 domain (omega = the root itself), the device-memory entry point kgr_ntt_device with guard regions
around the caller's buffer, Groth16 H (kgr_groth16_h) and kgr_groth16_prove_r1cs at production domain sizes.

Field elements are Montgomery residues x*R mod r (R = 2^256).  Every transform is linear with canonical constants (powers of omega and of the
coset generator), so applying it to the raw Montgomery integers gives the raw Montgomery integers of the result: the Python checks below work on
raw integers and never convert."""
import ctypes
import random

import numpy as np
import pytest

from oracle import oracle as A
from oracle import pyref as B

pytestmark = pytest.mark.gpu

R = B.FR
# fr.rs:60-65 ROOT_OF_UNITY (the limbs are the canonical value; the library converts them to Montgomery form), 2-adicity S = 28 (fr.rs:53)
ROOT = B.limbs_to_int([0xd34f1ed960c37c9c, 0x3215cf6dd39329c8, 0x98865ea93dd31f74, 0x03ddb9f5166d18b7])
S = 28
GEN = 7  # MULTIPLICATIVE_GENERATOR (fr.rs:18), the coset shift
OPS = ("dft", "idft", "coset_dft", "coset_idft")
GUARD = 64  # sentinel elements on each side of a device buffer
TOP_MASK = (1 << ((R >> 192).bit_length() - 1)) - 1  # a top limb below this keeps four random limbs under r


def seed(tag):
    return bytes((tag + i) % 256 for i in range(16))


def omega(log_n):
    return pow(ROOT, 1 << (S - log_n), R)


def raw_ints(arr):
    """(n, 4) uint64 limbs -> the integers they hold (Montgomery residues, not converted)."""
    return [a | b << 64 | c << 128 | d << 192 for a, b, c, d in np.asarray(arr, dtype=np.uint64).tolist()]


def raw_limbs(v):
    return np.array(B.int_to_limbs(v), dtype=np.uint64)


def horner(coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + c) % R
    return acc


def hadamard(a, b):
    """a o b elementwise, by the oracle's sparse product with diag(a)."""
    m = a.shape[0]
    diag = (np.arange(m + 1, dtype=np.uint32), np.arange(m, dtype=np.uint32), a)
    return A.sparse_prod(A.FIELD_FR, m, diag, b)


def kgr_ntt(log_n, op, values):
    """kgr_ntt through the C ABI, which (unlike Fft) also takes inputs longer than the domain."""
    from kogarashi_b200 import _lib
    from kogarashi_b200.fft import OPS as IDS
    v = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1, 4)
    out = np.zeros((1 << log_n, 4), dtype=np.uint64)
    n_out = ctypes.c_size_t()
    u64 = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))
    _lib.check(_lib.lib().kgr_ntt(log_n, IDS[op], u64(v), v.shape[0], u64(out), ctypes.byref(n_out)))
    return out[: n_out.value]


@pytest.fixture(scope="module")
def k():
    import kogarashi_b200 as kk
    kk.init()
    yield kk
    kk.init()  # destroys the engines and their cached NTT domains, so that later modules do not run with tens of GiB of tables resident


@pytest.fixture(scope="module")
def x21():
    """A random 2^21-element input and the reference's four transforms of it."""
    x = A.random_field(A.FIELD_FR, 1 << 21, seed=seed(21))
    return x, {op: A.fft(21, op, x) for op in OPS}


# ---- 1. three-pass transforms against the reference FFT ---------------------------------------------------------------------------------
@pytest.mark.parametrize("log_n,ops", [(21, OPS), (22, OPS), (23, ("dft", "coset_idft")), (24, ("dft", "coset_idft"))],
                         ids=["21-all", "22-all", "23-dft-coset_idft", "24-dft-coset_idft"])
def test_three_pass_transforms_bit_exact(k, request, log_n, ops):
    f = k.Fft(log_n)
    if log_n == 21:
        x, ref = request.getfixturevalue("x21")
    else:
        x, ref = A.random_field(A.FIELD_FR, 1 << log_n, seed=seed(log_n)), {}
    for op in ops:
        exp, n_exp = ref[op] if op in ref else A.fft(log_n, op, x)
        got = getattr(f, op)(x)
        assert got.shape[0] == n_exp and (got == exp[:n_exp]).all(), (log_n, op)
    if len(ops) == len(OPS):
        assert (f.idft(f.dft(x)) == x).all() and (f.coset_idft(f.coset_dft(x)) == x).all()  # fft.rs:247-270 round trips


def test_three_pass_schedule_is_reached(k):
    """A transform is one bit reversal plus ceil(k / 10) passes: 2^20 is the largest two-pass domain, 2^21 and up take three.  Pins that the
    transforms above run the three-pass schedule."""
    one = A.random_field(A.FIELD_FR, 1, seed=seed(1))
    for log_n, passes in ((20, 2), (21, 3), (24, 3)):
        f = k.Fft(log_n)
        f.dft(one)  # builds the domain tables on first use
        before = k.launch_count()
        f.dft(one)
        assert k.launch_count() - before == 1 + passes, log_n


def test_ragged_and_overlong_inputs_at_2p21(k):
    """Shorter inputs are zero padded and the inverse transforms strip trailing zeros (fft.rs:157-162, poly.rs:61-63); a longer input is
    truncated to the domain, as FrFft::prepare's resize does."""
    log_n, n = 21, 1 << 21
    f = k.Fft(log_n)
    x = A.random_field(A.FIELD_FR, n // 2 + 12345, seed=seed(60))
    x[-1000:] = 0  # trailing zero coefficients: the inverse transforms strip them
    for op in OPS:
        exp, n_exp = A.fft(log_n, op, x)
        got = getattr(f, op)(x)
        assert got.shape[0] == n_exp and (got == exp[:n_exp]).all(), op
    back = f.idft(f.dft(x))
    assert back.shape[0] == x.shape[0] - 1000 and (back == x[: back.shape[0]]).all()
    back = f.coset_idft(f.coset_dft(x))
    assert back.shape[0] == x.shape[0] - 1000 and (back == x[: back.shape[0]]).all()
    long = A.random_field(A.FIELD_FR, n + 777, seed=seed(61))
    for op in ("dft", "coset_dft", "idft"):
        exp, n_exp = A.fft(log_n, op, long)
        got = kgr_ntt(log_n, op, long)
        assert got.shape[0] == n_exp and (got == exp[:n_exp]).all(), op
        assert (got == getattr(f, op)(long[:n])).all(), op


# ---- 2. an independent check in Python integers at 2^21 ---------------------------------------------------------------------------------
def test_domain_constants_and_evaluations_in_python_ints(k, x21):
    """The facts the domain set-up relies on, and the device dft / coset_dft at a few points against Horner evaluations of the input
    polynomial: a check that does not go through the restated reference."""
    assert ROOT < R and pow(ROOT, 1 << S, R) == 1 and pow(ROOT, 1 << (S - 1), R) == R - 1  # a primitive 2^28-th root of unity
    assert pow(GEN, (R - 1) // 2, R) == R - 1  # 7 is a non-residue: the coset 7 * <omega> is disjoint from every 2-power domain
    log_n, n = 21, 1 << 21
    w = omega(log_n)
    assert pow(w, n // 2, R) == R - 1
    x, ref = x21
    f = k.Fft(log_n)
    dft, cdft = f.dft(x), f.coset_dft(x)
    assert (dft == ref["dft"][0]).all() and (cdft == ref["coset_dft"][0]).all()
    coeffs = raw_ints(x)
    rng = random.Random(log_n)
    for i in (1, rng.randrange(2, n - 1), n - 1):
        assert raw_ints(dft[i: i + 1])[0] == horner(coeffs, pow(w, i, R)), i
    i = rng.randrange(n)
    assert raw_ints(cdft[i: i + 1])[0] == horner(coeffs, GEN * pow(w, i, R) % R), i


# ---- 3. the device-memory entry point, with guard regions -------------------------------------------------------------------------------
class Guarded:
    """A torch buffer of n + 2 * GUARD elements: kgr_ntt_device transforms the middle n, the random words on both sides must survive."""

    def __init__(self, n, gen):
        import torch
        self.torch, self.n = torch, n
        self.buf = torch.empty((n + 2 * GUARD, 4), dtype=torch.int64, device="cuda")
        self.buf[:GUARD].random_(-2 ** 63, None, generator=gen)
        self.buf[GUARD + n:].random_(-2 ** 63, None, generator=gen)
        self.head, self.tail = self.buf[:GUARD].clone(), self.buf[GUARD + n:].clone()
        self.mid = self.buf[GUARD: GUARD + n]

    def run(self, f, op):
        self.torch.cuda.synchronize()  # the library's stream does not order itself after torch's
        f.transform_device(op, self.mid.data_ptr())
        assert self.torch.equal(self.buf[:GUARD], self.head), (op, "wrote below the buffer")
        assert self.torch.equal(self.buf[GUARD + self.n:], self.tail), (op, "wrote past the buffer")

    def rows(self, idx):
        t = self.mid[self.torch.tensor(idx, dtype=self.torch.int64, device="cuda")]
        return raw_ints(t.cpu().numpy().view(np.uint64))

    def set_row(self, i, v):
        self.mid[i] = self.torch.from_numpy(raw_limbs(v).view(np.int64)).cuda()


def test_device_entry_point_bit_exact_within_its_elements(k, x21):
    import torch
    x, ref = x21
    n = x.shape[0]
    f = k.Fft(21)
    g = Guarded(n, torch.Generator(device="cuda").manual_seed(21))
    xd = torch.from_numpy(x.view(np.int64)).cuda()
    for op in OPS:
        g.mid.copy_(xd)
        g.run(f, op)
        got = g.mid.cpu().numpy().view(np.uint64)
        assert (got == ref[op][0]).all(), op  # the inverse transforms leave the stripped tail as zeros


def _sparse_check(g, f, log_n, coef, idx, op, point):
    """After `op` on the sparse polynomial sum_j coef[j] X^j, element i holds sum_j coef[j] point(i)^j."""
    g.run(f, op)
    got = g.rows(idx)
    for i, v in zip(idx, got):
        x = point(i)
        assert v == sum(c * pow(x, j, R) for j, c in coef.items()) % R, (log_n, op, i)


def _assert_sparse(g, coef, chunk):
    """The whole middle equals the sparse vector: its rows, and zeros everywhere else (compared on the device)."""
    assert g.rows(sorted(coef)) == [coef[j] for j in sorted(coef)]
    for j in coef:
        g.set_row(j, 0)
    for s in range(0, g.n, chunk):
        assert not bool(g.mid[s: s + chunk].any()), s
    for j, c in coef.items():
        g.set_row(j, c)


def _dense_chunks(n, chunk, seed_):
    """Random reduced residues, generated chunk by chunk from one seeded generator so that they can be generated again to compare."""
    import torch
    gen = torch.Generator(device="cuda").manual_seed(seed_)
    for s in range(0, n, chunk):
        t = torch.empty((chunk, 4), dtype=torch.int64, device="cuda").random_(-2 ** 63, None, generator=gen)
        t[:, 3] &= TOP_MASK
        yield s, t


@pytest.mark.parametrize("log_n", [25, 26, 27, 28])
def test_device_entry_point_up_to_2p28(k, log_n):
    """Sparse inputs at 2^25 .. 2^28: sampled outputs of dft and coset_dft against sums in Python integers, then idft / coset_idft back to
    the input exactly; at 2^28 also a dense round trip of random residues.  The sentinels around the buffer are checked after every op.
    Nothing here goes through host memory: at 2^28 the buffer is 8 GiB and the four domain tables 24 GiB."""
    import torch
    n = 1 << log_n
    k.init()  # drops the domain tables and buffers of the smaller sizes
    torch.cuda.empty_cache()
    need = 3 * 32 * n + 32 * (n + 2 * GUARD) + (2 << 30)  # tables, buffer, a chunk and some slack
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"2^{log_n} needs {need / 2 ** 30:.1f} GiB of free device memory, {free / 2 ** 30:.1f} GiB are free")
    chunk = min(n, 1 << 24)
    f = k.Fft(log_n)
    g = Guarded(n, torch.Generator(device="cuda").manual_seed(log_n))
    try:
        rng = random.Random(log_n)
        degrees = sorted({0, 1, 0x5555555 & (n - 1), n // 2 + 1, n - 1})
        coef = {j: (R - 1 if j == 0 else rng.randrange(1, R)) for j in degrees}
        g.mid.zero_()
        for j, c in coef.items():
            g.set_row(j, c)
        idx = sorted({0, 1, n // 2, n - 1} | {rng.randrange(n) for _ in range(60)})
        w = omega(log_n)
        _sparse_check(g, f, log_n, coef, idx, "dft", lambda i: pow(w, i, R))
        g.run(f, "idft")
        _assert_sparse(g, coef, chunk)
        _sparse_check(g, f, log_n, coef, idx, "coset_dft", lambda i: GEN * pow(w, i, R) % R)
        g.run(f, "coset_idft")
        _assert_sparse(g, coef, chunk)
        if log_n == S:
            for fwd, inv in (("dft", "idft"), ("coset_dft", "coset_idft")):
                for s, t in _dense_chunks(n, chunk, 2828):
                    g.mid[s: s + chunk].copy_(t)
                before = k.launch_count()
                g.run(f, fwd)
                assert k.launch_count() - before == (1 if fwd == "coset_dft" else 0) + 1 + 3  # [coset scale,] bit reversal, three passes
                g.run(f, inv)
                for s, t in _dense_chunks(n, chunk, 2828):
                    assert torch.equal(g.mid[s: s + chunk], t), (fwd, s)
    finally:
        del g
        torch.cuda.empty_cache()
        k.init()


# ---- 4. Groth16 H at three-pass domains -------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def abc21():
    n = 1 << 21
    a = A.random_field(A.FIELD_FR, n, seed=seed(70))
    b = A.random_field(A.FIELD_FR, n, seed=seed(71))
    return a, b, hadamard(a, b)


def test_h_quotient_identity_at_a_random_point(k, abc21):
    """H(tau) (tau^n - 1) == A(tau) B(tau) - C(tau) in Python integers, with A, B, C the interpolants of a, b, c = a o b on the domain:
    A(tau) = (tau^n - 1) / n * sum_i a_i w^i / (tau - w^i)."""
    log_n, n = 21, 1 << 21
    a, b, c = abc21
    q = k.Fft(log_n).h_coefficients(a, b, c)
    assert 0 < q.shape[0] <= n - 1
    w, tau = omega(log_n), random.Random(7 * log_n).randrange(R)
    zt = (pow(tau, n, R) - 1) % R
    assert zt
    pw, x = [0] * n, 1
    for i in range(n):
        pw[i] = x
        x = x * w % R
    d = [(tau - p) % R for p in pw]
    pre, acc = [0] * n, 1  # batch inversion of the tau - w^i
    for i in range(n):
        pre[i] = acc
        acc = acc * d[i] % R
    inv = pow(acc, -1, R)
    lw = [0] * n
    for i in range(n - 1, -1, -1):
        lw[i] = pw[i] * (inv * pre[i] % R) % R
        inv = inv * d[i] % R
    scale = zt * pow(n, -1, R) % R
    ev = lambda v: scale * (sum(s * t for s, t in zip(raw_ints(v), lw)) % R) % R
    at, bt, ct, ht = ev(a), ev(b), ev(c), horner(raw_ints(q), tau)
    m = B.R256 % R  # every value above is the Montgomery integer, i.e. R times the field element
    assert ht * zt % R * m % R == (at * bt - ct * m) % R


def test_domain_cache_and_buffer_reuse_across_sizes(k, abc21):
    """2^21, then 2^10, then 2^21 again in one process: the per-size domain tables and the larger device buffers are reused correctly."""
    a, b, c = abc21
    f21, f10 = k.Fft(21), k.Fft(10)
    q1, d1 = f21.h_coefficients(a, b, c), f21.dft(a)
    a10, b10 = a[:1 << 10], b[:1 << 10]
    c10 = c[:1 << 10]
    exp, n_exp = A.groth16_h(10, a10, b10, c10)
    got = f10.h_coefficients(a10, b10, c10)
    assert got.shape[0] == n_exp and (got == exp[:n_exp]).all()
    assert (f10.dft(a10) == A.fft(10, "dft", a10)[0]).all()
    q2, d2 = f21.h_coefficients(a, b, c), f21.dft(a)
    assert q1.shape == q2.shape and (q1 == q2).all() and (d1 == d2).all()


# ---- 5. kgr_groth16_prove_r1cs at three-pass domains ------------------------------------------------------------------------------------
def _random_csr(rng, m, n_z, pool):
    """0 to 3 terms per row (about a quarter of the rows empty), columns anywhere in z, coefficients drawn from `pool`."""
    row_ptr = np.zeros(m + 1, dtype=np.uint32)
    row_ptr[1:] = np.cumsum(rng.integers(0, 4, m))
    nnz = int(row_ptr[-1])
    return row_ptr, rng.integers(0, n_z, nnz).astype(np.uint32), pool[rng.integers(0, pool.shape[0], nnz)]


@pytest.mark.parametrize("log_n,m", [(21, (1 << 21) - 3), (21, (1 << 20) + 1), (22, 1000)])
def test_prove_r1cs_at_three_pass_domains(k, log_n, m):
    """A random (unsatisfied) R1CS evaluated on the device into bit-reversed positions: q equals the reference H of the host evaluations,
    and kgr_groth16_h of them, length included; the h query equals an MSM of q.  The queries are 64 points, so no large MSM runs."""
    from kogarashi_b200.nova import FIELD_FR, DeviceVec, R1csShape
    n_z, n_inputs = 1024, 4
    rng = np.random.default_rng(log_n * 1000003 + m)
    pool = A.random_field(A.FIELD_FR, 64, seed=seed(80))
    pool[0], pool[1] = raw_limbs(B.to_mont(1, R)), raw_limbs(B.to_mont(R - 1, R))
    mats = [_random_csr(rng, m, n_z, pool) for _ in range(3)]
    z = A.random_field(A.FIELD_FR, n_z, seed=seed(81))
    z[0] = raw_limbs(B.to_mont(1, R))
    evals = [A.sparse_prod(A.FIELD_FR, m, M, z) for M in mats]
    q_ref, n_ref = A.groth16_h(log_n, *evals)
    shape, zd = R1csShape(FIELD_FR, m, n_z, *mats), DeviceVec(FIELD_FR, z)
    h, l, a, b_g1 = (k.Bases.generate(k.BN254_G1, 64, s) for s in (91, 92, 93, 94))
    try:
        res, q, _ = k.groth16_prove_r1cs(log_n, shape, zd, n_inputs, h, l, a, b_g1, None, [])
        assert q.shape[0] == n_ref and (q == q_ref[:n_ref]).all()
        q_host = k.Fft(log_n).h_coefficients(*evals)
        assert q_host.shape == q.shape and (q_host == q).all()
        assert (k.to_affine(k.BN254_G1, res["h"]) == k.to_affine(k.BN254_G1, k.msm_curve_addition(h, q))).all()
    finally:
        for x in (h, l, a, b_g1, shape, zd):
            x.free()
