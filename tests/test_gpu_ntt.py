"""GPU parity tests of the Fr NTT (row N2) against the restated reference FFT (oracle FrFft = groth16/src/fft.rs), bit for bit."""
import numpy as np
import pytest

from oracle import oracle as A

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def k():
    import kogarashi_b200 as kk
    kk.init()
    return kk


@pytest.mark.parametrize("log_n", [1, 2, 3, 5, 8, 10, 11, 13, 16, 20])  # 20: the largest two-pass domain (10 + 10 stages)
def test_transforms_bit_exact(k, log_n):
    n = 1 << log_n
    f = k.Fft(log_n)
    x = A.random_field(A.FIELD_FR, n, seed=bytes(range(log_n, log_n + 16)))
    for op in ("dft", "idft", "coset_dft", "coset_idft"):
        exp, n_exp = A.fft(log_n, op, x)
        got = getattr(f, op)(x)
        assert got.shape[0] == n_exp and (got == exp[:n_exp]).all(), (log_n, op)
    assert (f.idft(f.dft(x)) == x).all() and (f.coset_idft(f.coset_dft(x)) == x).all()     # fft.rs:247-270 round trips


@pytest.mark.parametrize("log_n,m", [(3, 5), (6, 64), (10, 700)])
def test_ragged_inputs_and_stripping(k, log_n, m):
    """Inputs shorter than the domain are zero padded (prepare_fft); inverse transforms strip trailing zeros (Coefficients::new)."""
    f = k.Fft(log_n)
    x = A.random_field(A.FIELD_FR, m, seed=bytes(range(16)))
    for op in ("dft", "coset_dft", "idft"):
        exp, n_exp = A.fft(log_n, op, x)
        got = getattr(f, op)(x)
        assert got.shape[0] == n_exp and (got == exp[:n_exp]).all()
    low = f.dft(x[:3])                                   # a degree-2 polynomial evaluated on the domain ...
    back = f.idft(low)                                   # ... comes back with exactly 3 coefficients
    assert back.shape[0] == 3 and (back == x[:3]).all()
    assert f.idft(np.zeros((4, 4), dtype=np.uint64)).shape[0] == 0


def test_fft_multiplication_matches_naive(k):
    """groth16/src/fft.rs:272-291: product via dft == schoolbook product (oracle field arithmetic)."""
    log_n, d = 6, 20
    f = k.Fft(log_n)
    a = A.random_field(A.FIELD_FR, d, seed=bytes(range(1, 17)))
    b = A.random_field(A.FIELD_FR, d, seed=bytes(range(2, 18)))
    ea, eb = f.dft(a), f.dft(b)
    prod = np.stack([A.field_op(A.FIELD_FR, "mul", ea[i], eb[i]) for i in range(1 << log_n)])
    got = f.idft(prod)
    naive = np.zeros((2 * d - 1, 4), dtype=np.uint64)
    for i in range(d):
        for j in range(d):
            naive[i + j] = A.field_op(A.FIELD_FR, "add", naive[i + j], A.field_op(A.FIELD_FR, "mul", a[i], b[j]))
    assert got.shape[0] == 2 * d - 1 and (got == naive).all()


# 2^21 and 2^22 run three passes per transform; m = n / 2 + 1 is mostly padding
@pytest.mark.parametrize("log_n,m", [(2, 4), (10, 1000), (14, 1 << 14), (21, 1 << 21), (21, (1 << 20) + 1), (22, 1 << 22), (22, (1 << 21) + 1)])
def test_h_coefficients_match_reference_pipeline(k, log_n, m):
    """prover.rs:36-47 on the device == the same pipeline through the restated reference FFT."""
    f = k.Fft(log_n)
    a = A.random_field(A.FIELD_FR, m, seed=bytes(range(3, 19)))
    b = A.random_field(A.FIELD_FR, m, seed=bytes(range(4, 20)))
    # make c = a * b on the domain so that H is a genuine quotient (degree <= n - 2)
    c = A.sparse_prod(A.FIELD_FR, m, (np.arange(m + 1, dtype=np.uint32), np.arange(m, dtype=np.uint32), a), b)  # diag(a) b
    exp, n_exp = A.groth16_h(log_n, a, b, c)
    got = f.h_coefficients(a, b, c)
    assert got.shape[0] == n_exp and (got == exp[:n_exp]).all()
    assert n_exp <= (1 << log_n) - 1


def test_large_transform_through_staged_host_copies():
    """2^19 elements = 16 MiB each way from ordinary numpy memory: the upload and the download go through the pinned staging ring
    (upload_from_host / download_to_host); result bit-exact with the restated reference FFT, ragged input included."""
    import kogarashi_b200 as k
    from kogarashi_b200.fft import Fft
    k.init()
    kk = 19
    n = 1 << kk
    vals = A.random_field(A.FIELD_FR, n - 12345, seed=bytes(range(21, 37)))
    f = Fft(kk)
    got = f.dft(vals)
    exp, _ = A.fft(kk, "dft", vals)
    assert got.shape == exp.shape and (got == exp).all()
    back = f.idft(got)                       # idft strips trailing zeros (poly.rs:61-63): the ragged input comes back at its own length
    assert back.shape[0] == vals.shape[0] and (back == vals).all()
