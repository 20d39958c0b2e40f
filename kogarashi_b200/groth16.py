"""The MSM / FFT part of the reference's Groth16 prover on the GPU engine (SURVEY.md §8f rows N1 + N2 + N3).

Reference: groth16/src/prover.rs:32-92.  `create_proof` runs seven FFTs (:36-47), six G1 MSMs (h, l, a x2, b_g1 x2;
:51-62), two G2 MSMs (b_g2 x2, :64-65) and assembles
    A = r*delta + alpha + a_answer                                          (:75,81-82)
    B = s*delta_g2 + beta_g2 + b2_answer                                    (:76,87-88)
    C = r*s*delta + s*alpha + r*beta + s*a_answer + r*b1_answer + q + l     (:77,84,90-92)
`Groth16G1Prover` computes A and C; `Groth16Prover` adds B with the G2 MSM, i.e. the whole proof.
Here the G1 CRS (`Parameters::{h, l, a, b_g1}`, groth16/src/params.rs:7-29) is registered on the GPU once per prover;
per proof the H coefficients come from the device NTT (kogarashi_b200.fft) and the `a_inputs / a_aux` and
`b_g1_inputs / b_g1_aux` pairs are fused into one MSM each over z = inputs ++ aux (the prover splits them only because
of its slice layout, :58-62).  The blinding terms are a five-point MSM, so no curve arithmetic is done in Python.
`prove_r1cs` starts one step earlier, from the constraint system: the evaluations of :33 are computed on the device from a registered
R1CS shape and the resident assignment z, and every query reads its scalars from z in device memory.
`setup` generates the parameters themselves (groth16/src/zksnark.rs:17-127) on the device from the registered shape; `from_params` hands its
resident queries to a prover without a download or a re-upload.
`Groth16Verifier` checks proofs (groth16/src/verifier.rs, the pairing equation of proof.rs:39-48) on the device, one batched pairing check for
a set of proofs against one key.
"""
import os

import numpy as np

from .fft import Fft
from .msm import (BN254_G1, BN254_G2, SCALARS_CANONICAL, SCALARS_MONTGOMERY, Bases, coord_limbs, groth16_msms, groth16_prove_r1cs, groth16_setup,
                  groth16_verify, msm_batch, msm_curve_addition, proj_add, to_affine)

FR = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001  # bn254/src/fr.rs:11-16


class ProverSubVersionCrsAttack(ValueError):
    """groth16/src/error.rs:3 — `create_proof` refuses a CRS whose delta_g1 or delta_g2 is the identity (prover.rs:67-69)."""


def _vk_points(points, inf, words):
    """vk elements as a (k, words) array + (k,) infinity flags.  The reference encodes the identity as (0, R, is_infinity = true)
    (zkstd/src/macros/curve/weierstrass/group.rs:106-110); (0, 0) — the device's own identity encoding — is accepted as well."""
    pts = np.stack([np.ascontiguousarray(p, dtype=np.uint64).reshape(words) for p in points])
    flags = np.zeros(len(points), dtype=np.uint8) if inf is None else np.ascontiguousarray(inf, dtype=np.uint8).reshape(len(points)).copy()
    flags |= (~pts.any(axis=1)).astype(np.uint8)
    return pts, flags


def _canonical(vals):
    out = np.zeros((len(vals), 4), dtype=np.uint64)
    for i, v in enumerate(vals):
        v %= FR
        for k in range(4):
            out[i, k] = (v >> (64 * k)) & 0xFFFFFFFFFFFFFFFF
    return out


def _mont(vals):
    return _canonical([v * (1 << 256) for v in vals])


class Groth16Params:
    """The parameters of zksnark.rs:17-127 with every query resident on the device (`setup`): `a`, `b_g1`, `b_g2` (None for a G1-only setup),
    `ic`, `l`, `h` are `Bases`; `vk_g1` (3, 9) holds alpha, beta, delta and `vk_g2` (3, 17) beta, gamma, delta as x, y, is_infinity.
    `log_n` is the domain the prover must use.  The h query has m - 1 entries as in the reference, so a proof is only guaranteed to be valid
    for m = 2^log_n.  A prover built with `from_params` takes over a, b_g1, h, l (and b_g2) and frees them; `ic` and the vk stay here."""

    QUERIES = ("a", "b_g1", "b_g2", "ic", "l", "h")

    def __init__(self, log_n, queries, vk_g1, vk_g2):
        self.log_n, self.vk_g1, self.vk_g2 = log_n, vk_g1, vk_g2
        for name in self.QUERIES:
            setattr(self, name, queries.get(name))

    def take(self, *names):
        """Hand the named query handles over to a new owner: they are no longer held (or freed) by these parameters."""
        out = []
        for name in names:
            b = getattr(self, name)
            if b is None:
                raise ValueError(f"the {name} query is not held by these parameters (not generated, or already taken)")
            setattr(self, name, None)
            out.append(b)
        return out

    def download(self):
        """-> {"log_n", "vk_g1", "vk_g2", and per query still held: (points (n, 8) or (n, 16) uint64 Montgomery x || y, is_infinity (n,) uint8)}:
        the host arrays for serialisation and for a verifier (an identity reads (0, 0) with its flag set)."""
        out = dict(log_n=self.log_n, vk_g1=self.vk_g1.copy(), vk_g2=None if self.vk_g2 is None else self.vk_g2.copy())
        for name in self.QUERIES:
            b = getattr(self, name)
            if b is not None:
                pts = b.download() if b.n else np.zeros((0, 2 * coord_limbs(b.curve)), dtype=np.uint64)
                out[name] = (pts, (~pts.any(axis=1)).astype(np.uint8))
        return out

    def free(self):
        for name in self.QUERIES:
            b = getattr(self, name)
            if b is not None:
                b.free()
                setattr(self, name, None)


def setup(shape, n_inputs, toxic=None, g2=True):
    """ZkSnark::setup (groth16/src/zksnark.rs:17-127) on the device: `shape` is the nova.R1csShape of the circuit registered over FIELD_FR with
    columns over z = x ++ w, `n_inputs` = len(x) (the constant one included).  toxic: (alpha, beta, gamma, delta, tau) as Python ints; by default
    each is 64 bytes of os.urandom reduced modulo r, redrawn while zero.  g2=False skips the G2 query.  -> Groth16Params"""
    if toxic is None:
        toxic = []
        while len(toxic) < 5:
            v = int.from_bytes(os.urandom(64), "little") % FR
            if v:
                toxic.append(v)
    toxic = [int(v) % FR for v in toxic]
    if len(toxic) != 5:
        raise ValueError("toxic waste is five field elements: alpha, beta, gamma, delta, tau")
    log_n, queries, vk_g1, vk_g2 = groth16_setup(shape, n_inputs, _mont(toxic), g2)
    return Groth16Params(log_n, queries, vk_g1, vk_g2)


class Groth16G1Prover:
    """Points are (n, 8) uint64 Montgomery arrays with (n,) uint8 infinity flags (CRS entries may be the identity,
    groth16/src/zksnark.rs:62-66,177-185)."""

    def __init__(self, delta_g1, alpha_g1, beta_g1, a, a_inf, b_g1, b_g1_inf, h, h_inf, l, l_inf, precompute=False, vk_inf=None):
        """vk_inf: optional is_infinity flags of (delta_g1, alpha_g1, beta_g1).  An identity delta_g1 raises ProverSubVersionCrsAttack
        before anything is uploaded — the reference returns that error from create_proof (prover.rs:67-69)."""
        self._set_vk(delta_g1, alpha_g1, beta_g1, vk_inf)
        self._set_queries(*(Bases(BN254_G1, p, f) for p, f in ((a, a_inf), (b_g1, b_g1_inf), (h, h_inf), (l, l_inf))), precompute=precompute)

    @classmethod
    def from_params(cls, params, precompute=False):
        """A prover on the resident queries of `params` (groth16.setup): no download, no re-upload.  The prover takes the handles over
        (Groth16Params.take) and frees them once, in `free`."""
        self = cls.__new__(cls)
        self._adopt(params, precompute)
        return self

    def _adopt(self, params, precompute):
        alpha, beta, delta = params.vk_g1
        self._set_vk(delta[:8], alpha[:8], beta[:8], [delta[8], alpha[8], beta[8]])
        self._set_queries(*params.take("a", "b_g1", "h", "l"), precompute=precompute)

    def _set_vk(self, delta_g1, alpha_g1, beta_g1, vk_inf):
        self.vk, self.vk_inf = _vk_points([delta_g1, alpha_g1, beta_g1], vk_inf, 8)
        if self.vk_inf[0]:
            raise ProverSubVersionCrsAttack("vk.delta_g1 is the identity")

    def _set_queries(self, a, b_g1, h, l, precompute):
        self.a, self.b_g1, self.h, self.l = a, b_g1, h, l
        self.vk_bases = Bases(BN254_G1, self.vk, self.vk_inf)
        if precompute:
            for b in (self.a, self.b_g1, self.h, self.l):
                b.precompute(0)

    def _g1_jobs(self, q, inputs, aux, r, scalar_fmt):
        """The G1 queries of prover.rs:51-62 as one batch (independent MSMs overlap on the device) + the blinding of A."""
        z = np.concatenate([np.asarray(inputs, dtype=np.uint64).reshape(-1, 4), np.asarray(aux, dtype=np.uint64).reshape(-1, 4)])
        return z, [(self.a, z, 0, scalar_fmt),                      # a_inputs + a_aux       (:58-59, :80)
                   (self.b_g1, z, 0, scalar_fmt),                   # b_g1_inputs + b_g1_aux (:61-62, :86)
                   (self.h, q, 0, scalar_fmt),                      # :51
                   (self.l, aux, 0, scalar_fmt),                    # :56
                   self._blind_a_job(r)]

    def _blind_a_job(self, r):
        return (self.vk_bases, _canonical([r, 1]), 0, SCALARS_CANONICAL)   # r*delta + alpha (:75)

    def _assemble_g1(self, res, r, s):
        a_answer, b1_answer, q_pt, l_pt, blind_a = res[:5]
        delta, alpha, beta = self.vk
        g_a = proj_add(BN254_G1, blind_a, a_answer)
        aa, ba = to_affine(BN254_G1, a_answer), to_affine(BN254_G1, b1_answer)
        pts = np.stack([aa[:8], ba[:8], delta, alpha, beta])
        inf = np.array([aa[8], ba[8], self.vk_inf[0], self.vk_inf[1], self.vk_inf[2]], dtype=np.uint8)
        blind_c = msm_curve_addition(pts, _canonical([s, r, r * s, s, r]), curve=BN254_G1, inf=inf, scalar_fmt=SCALARS_CANONICAL)
        g_c = proj_add(BN254_G1, proj_add(BN254_G1, blind_c, q_pt), l_pt)
        return to_affine(BN254_G1, g_a), to_affine(BN254_G1, g_c)

    def prove_g1(self, q, inputs, aux, r, s, scalar_fmt=SCALARS_MONTGOMERY):
        """q, inputs, aux: (len, 4) uint64 scalars in `scalar_fmt`; r, s: Python ints (the prover's blinding factors, prover.rs:71-72).
        -> (A, C) as (9,) uint64 affine [x, y, is_infinity] = Proof.a / Proof.c after `.into()` (prover.rs:94-98)."""
        _, jobs = self._g1_jobs(q, inputs, aux, r, scalar_fmt)
        return self._assemble_g1(msm_batch(jobs), r, s)

    def prove_from_evaluations(self, log_n, a_evals, b_evals, c_evals, inputs, aux, r, s):
        """The whole G1 side of create_proof from the R1CS evaluations (prover.rs:33): one kgr_groth16_msms call — H on the device feeding the h
        query directly, the other queries overlapped with it.  All scalars are Montgomery arrays (the reference's in-memory form)."""
        _, jobs = self._g1_jobs(np.zeros((0, 4), dtype=np.uint64), inputs, aux, r, SCALARS_MONTGOMERY)
        del jobs[2]                                                   # the h query is the fused part of the call
        q_pt, q, res = groth16_msms(log_n, a_evals, b_evals, c_evals, self.h, jobs)
        return self._assemble_g1([res[0], res[1], q_pt, res[2], res[3]], r, s) + (q,)

    def prove_r1cs(self, log_n, shape, z, n_inputs, r, s):
        """The G1 side of create_proof from the constraint system (prover.rs:32-98) in one kgr_groth16_prove_r1cs call: `shape` is the
        nova.R1csShape of the circuit registered over FIELD_FR, `z` the nova.DeviceVec of cs.x() ++ cs.w(), the first n_inputs elements the
        instance.  -> (A, C, q) as prove_from_evaluations."""
        res, q, jobs = groth16_prove_r1cs(log_n, shape, z, n_inputs, self.h, self.l, self.a, self.b_g1, None, [self._blind_a_job(r)])
        return self._assemble_g1([res["a"], res["b_g1"], res["h"], res["l"], jobs[0]], r, s) + (q,)

    def commitments(self, q, inputs, aux, r, s):
        """Same as prove_g1 for scalars given as Python integers."""
        return self.prove_g1(_canonical(list(q)), _canonical(list(inputs)), _canonical(list(aux)), r, s, scalar_fmt=SCALARS_CANONICAL)

    def free(self):
        for b in (self.a, self.b_g1, self.h, self.l, self.vk_bases):
            b.free()


class Groth16Prover(Groth16G1Prover):
    """All three proof elements.  G2 points are (n, 16) uint64 = x.c0 x.c1 y.c0 y.c1 Montgomery (bn254/src/g2.rs:15-21)."""

    def __init__(self, delta_g1, alpha_g1, beta_g1, a, a_inf, b_g1, b_g1_inf, h, h_inf, l, l_inf, delta_g2, beta_g2, b_g2, b_g2_inf, precompute=False,
                 vk_inf=None, vk_g2_inf=None):
        """vk_g2_inf: optional is_infinity flags of (delta_g2, beta_g2); an identity delta_g2 raises ProverSubVersionCrsAttack (prover.rs:67-69)."""
        self._set_vk_g2(delta_g2, beta_g2, vk_g2_inf)
        super().__init__(delta_g1, alpha_g1, beta_g1, a, a_inf, b_g1, b_g1_inf, h, h_inf, l, l_inf, precompute=precompute, vk_inf=vk_inf)
        self._set_g2_query(Bases(BN254_G2, b_g2, b_g2_inf), precompute)

    def _adopt(self, params, precompute):
        if params.b_g2 is None:
            raise ValueError("the parameters hold no b_g2 query (setup with g2=False, or already taken)")
        beta, _, delta = params.vk_g2
        self._set_vk_g2(delta[:16], beta[:16], [delta[16], beta[16]])
        super()._adopt(params, precompute)
        self._set_g2_query(*params.take("b_g2"), precompute)

    def _set_vk_g2(self, delta_g2, beta_g2, vk_g2_inf):
        self.vk_g2, self.vk_g2_inf = _vk_points([delta_g2, beta_g2], vk_g2_inf, 16)
        if self.vk_g2_inf[0]:
            raise ProverSubVersionCrsAttack("vk.delta_g2 is the identity")

    def _set_g2_query(self, b_g2, precompute):
        self.b_g2 = b_g2
        self.vk_g2_bases = Bases(BN254_G2, self.vk_g2, self.vk_g2_inf)
        if precompute:
            self.b_g2.precompute(0)

    def prove(self, q, inputs, aux, r, s, scalar_fmt=SCALARS_MONTGOMERY):
        """-> (A, B, C): A, C (9,) uint64 and B (17,) uint64 affine [x, y, is_infinity] = Proof {a, b, c} (prover.rs:94-98).
        All eight MSMs of prover.rs:51-65 (pairs fused) and the two independent blinding sums go to the device as one batch."""
        z, jobs = self._g1_jobs(q, inputs, aux, r, scalar_fmt)
        # the G2 query is the longest job (3x the arithmetic per point): it goes first so that the G1 queries overlap with it
        jobs = [(self.b_g2, z, 0, scalar_fmt)] + jobs + [self._blind_b_job(s)]   # :64-65,:87
        res = msm_batch(jobs)
        g_a, g_c = self._assemble_g1(res[1:6], r, s)
        return g_a, self._assemble_b(res[0], res[6]), g_c

    def _blind_b_job(self, s):
        return (self.vk_g2_bases, _canonical([s, 1]), 0, SCALARS_CANONICAL)   # s*delta_g2 + beta_g2 (:76)

    @staticmethod
    def _assemble_b(b2_answer, blind_b):
        return to_affine(BN254_G2, proj_add(BN254_G2, blind_b, b2_answer))   # :87-88

    def prove_from_evaluations(self, log_n, a_evals, b_evals, c_evals, inputs, aux, r, s):
        """create_proof after witness generation (prover.rs:33-98) as one kgr_groth16_msms call + the dependent blinding sum."""
        z, jobs = self._g1_jobs(np.zeros((0, 4), dtype=np.uint64), inputs, aux, r, SCALARS_MONTGOMERY)
        del jobs[2]
        jobs = [(self.b_g2, z, 0, SCALARS_MONTGOMERY)] + jobs + [self._blind_b_job(s)]
        q_pt, q, res = groth16_msms(log_n, a_evals, b_evals, c_evals, self.h, jobs)
        g_a, g_c = self._assemble_g1([res[1], res[2], q_pt, res[3], res[4]], r, s)
        return g_a, self._assemble_b(res[0], res[5]), g_c, q

    def prove_r1cs(self, log_n, shape, z, n_inputs, r, s):
        """create_proof from the constraint system (prover.rs:32-98): the evaluations, H and all eight query MSMs on the device in one
        kgr_groth16_prove_r1cs call, with the scalars read from the resident z (see Groth16G1Prover.prove_r1cs).  -> (A, B, C, q)"""
        res, q, jobs = groth16_prove_r1cs(log_n, shape, z, n_inputs, self.h, self.l, self.a, self.b_g1, self.b_g2, [self._blind_a_job(r), self._blind_b_job(s)])
        g_a, g_c = self._assemble_g1([res["a"], res["b_g1"], res["h"], res["l"], jobs[0]], r, s)
        return g_a, self._assemble_b(res["b_g2"], jobs[1]), g_c, q

    def proof(self, q, inputs, aux, r, s):
        """Scalars as Python integers."""
        return self.prove(_canonical(list(q)), _canonical(list(inputs)), _canonical(list(aux)), r, s, scalar_fmt=SCALARS_CANONICAL)

    def free(self):
        super().free()
        self.b_g2.free()
        self.vk_g2_bases.free()


class Groth16Verifier:
    """groth16/src/verifier.rs on the device (kgr_groth16_verify).  vk_g1 (3, 9): alpha, beta, delta; vk_g2 (3, 17): beta, gamma, delta (the layout
    of Groth16Params); ic: the ic query as `Bases`, or a host (points (n, 8), is_infinity (n,)) pair that is registered here and freed in `free`."""

    def __init__(self, vk_g1, vk_g2, ic):
        self.vk_g1 = np.ascontiguousarray(vk_g1, dtype=np.uint64).reshape(3, 9)
        self.vk_g2 = np.ascontiguousarray(vk_g2, dtype=np.uint64).reshape(3, 17)
        if isinstance(ic, Bases):
            self.ic, self._own_ic = ic, False
        else:
            pts, inf = ic
            self.ic, self._own_ic = Bases(BN254_G1, pts, inf), True

    @classmethod
    def from_params(cls, params):
        """A verifier on the resident ic query of `params` (groth16.setup): borrowed, not taken, so the parameters keep it and free it."""
        if params.ic is None or params.vk_g2 is None:
            raise ValueError("the parameters hold no ic query or no G2 verifying key (setup with g2=False)")
        return cls(params.vk_g1, params.vk_g2, params.ic)

    @property
    def n_public(self):
        return self.ic.n - 1

    def verify(self, proofs, inputs, rho=None):
        """proofs: a list of (A, B, C) as `prove` / `prove_r1cs` return them ((9,), (17,), (9,) uint64; extra items such as q are ignored), or a
        (k, 35) array.  inputs: (k, n_public, 4) Montgomery Fr, or per proof a list of Python ints — the instance without its leading one.
        rho: (k, 2) uint64 128-bit non-zero batching weights; None draws them from os.urandom (zeros redrawn).  -> (k,) bool"""
        if isinstance(proofs, np.ndarray):
            arr = np.ascontiguousarray(proofs, dtype=np.uint64).reshape(-1, 35)
        else:
            arr = np.stack([np.concatenate([np.asarray(p[0], dtype=np.uint64).reshape(9), np.asarray(p[1], dtype=np.uint64).reshape(17),
                                            np.asarray(p[2], dtype=np.uint64).reshape(9)]) for p in proofs]) if len(proofs) else np.zeros((0, 35), np.uint64)
        k = arr.shape[0]
        if isinstance(inputs, np.ndarray):
            xs = np.ascontiguousarray(inputs, dtype=np.uint64).reshape(k, self.n_public, 4)
        else:
            rows = [list(r) for r in inputs]
            if len(rows) != k or any(len(r) != self.n_public for r in rows):
                raise ValueError(f"inputs: {k} rows of {self.n_public} public inputs expected")
            xs = np.stack([_mont([int(v) for v in r]) for r in rows]) if k and self.n_public else np.zeros((k, self.n_public, 4), np.uint64)
        if rho is None and k >= 2:
            rho = np.zeros((k, 2), dtype=np.uint64)
            for i in range(k):
                while not rho[i].any():
                    rho[i] = np.frombuffer(os.urandom(16), dtype=np.uint64)
        return groth16_verify(self.vk_g1, self.vk_g2, self.ic, arr, xs, rho if k >= 2 else None)

    def free(self):
        if self._own_ic:
            self.ic.free()
