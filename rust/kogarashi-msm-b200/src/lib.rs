//! Drop-in for `groth16::msm::msm_curve_addition` (groth16/src/msm.rs:6), the body of `nova::PedersenCommitment::commit`
//! (nova/src/pedersen.rs:15-20) and the rows built around them (G2 MSM, Fr NTT / H polynomial, the prover's fused query call, Nova's
//! folding vector work) over the C ABI in include/kgr_msm.h.
//!
//! UNTESTED BY A COMPILER: this file has never been compiled (no rustc / cargo in the development image).  What IS checked mechanically:
//! tests/test_rust_shim.py parses the `extern "C"` block below and compares every function — name, argument count, argument types,
//! return type — with the prototypes in include/kgr_msm.h, and examples/abi_demo.c performs each marshalling step of this file in C.
use core::ffi::{c_char, c_long, c_void};
use std::sync::Once;

use zkstd::common::{BNAffine, BNProjective, CurveGroup};

#[allow(non_camel_case_types)]
#[repr(C)]
pub struct kgr_bases_t {
    _private: [u8; 0],
}
#[allow(non_camel_case_types)]
#[repr(C)]
pub struct kgr_r1cs_t {
    _private: [u8; 0],
}
#[allow(non_camel_case_types)]
#[repr(C)]
pub struct kgr_vec_t {
    _private: [u8; 0],
}
/// `kgr_msm_job_t` of the header: one MSM of a batch.
#[allow(non_camel_case_types)]
#[repr(C)]
pub struct kgr_msm_job_t {
    pub bases: *mut kgr_bases_t,
    pub base_off: usize,
    pub scalars: *const u64,
    pub scalar_fmt: i32,
    pub n: usize,
    pub out: *mut u64,
}

extern "C" {
    fn kgr_init(devices: *const i32, n_devices: i32) -> i32;
    fn kgr_shutdown() -> i32;
    fn kgr_last_error() -> *const c_char;
    fn kgr_device_count() -> i32;
    fn kgr_bases_register(curve: i32, xy: *const u64, inf: *const u8, n: usize, out: *mut *mut kgr_bases_t) -> i32;
    fn kgr_bases_free(bases: *mut kgr_bases_t) -> i32;
    fn kgr_bases_len(bases: *const kgr_bases_t) -> usize;
    fn kgr_bases_precompute(bases: *mut kgr_bases_t, window_bits: i32) -> i32;
    fn kgr_msm(bases: *mut kgr_bases_t, base_off: usize, scalars: *const u64, scalar_fmt: i32, n: usize, out: *mut u64) -> i32;
    fn kgr_msm_batch(jobs: *const kgr_msm_job_t, n_jobs: usize) -> i32;
    fn kgr_msm_oneshot(curve: i32, xy: *const u64, inf: *const u8, n_bases: usize, scalars: *const u64, scalar_fmt: i32, n_scalars: usize,
                       out: *mut u64) -> i32;
    fn kgr_msm_device(bases: *mut kgr_bases_t, base_off: usize, d_scalars: *const c_void, scalar_fmt: i32, n: usize, out: *mut u64) -> i32;
    fn kgr_bases_download(bases: *const kgr_bases_t, off: usize, n: usize, xy_out: *mut u64) -> i32;
    fn kgr_pedersen_commit(ck: *mut kgr_bases_t, scalars: *const u64, scalar_fmt: i32, n: usize, out: *mut u64) -> i32;
    fn kgr_to_affine(curve: i32, input: *const u64, out: *mut u64) -> i32;
    fn kgr_proj_add(curve: i32, a: *const u64, b: *const u64, out: *mut u64) -> i32;
    fn kgr_ntt(log_n: u32, op: i32, input: *const u64, n_in: usize, out: *mut u64, n_out: *mut usize) -> i32;
    fn kgr_ntt_device(log_n: u32, op: i32, d_data: *mut c_void) -> i32;
    fn kgr_groth16_h(log_n: u32, a: *const u64, b: *const u64, c: *const u64, m: usize, out: *mut u64, n_out: *mut usize) -> i32;
    fn kgr_r1cs_register(field: i32, m: usize, n_z: usize, row_ptr: *const *const u32, cols: *const *const u32, coeffs: *const *const u64,
                         out: *mut *mut kgr_r1cs_t) -> i32;
    fn kgr_r1cs_free(shape: *mut kgr_r1cs_t) -> i32;
    fn kgr_r1cs_mul(shape: *mut kgr_r1cs_t, which: i32, z: *const u64, out: *mut u64) -> i32;
    fn kgr_nova_cross_term(shape: *mut kgr_r1cs_t, z1: *const u64, z2: *const u64, t_out: *mut u64, ck: *mut kgr_bases_t, commit_out: *mut u64) -> i32;
    fn kgr_r1cs_last_timing(shape: *const kgr_r1cs_t, ms: *mut f32) -> i32;
    fn kgr_vec_fold(field: i32, a: *const u64, b: *const u64, r: *const u64, n: usize, out: *mut u64) -> i32;
    fn kgr_vec_upload(field: i32, host: *const u64, n: usize, out: *mut *mut kgr_vec_t) -> i32;
    fn kgr_vec_download(v: *const kgr_vec_t, off: usize, n: usize, host: *mut u64) -> i32;
    fn kgr_vec_free(v: *mut kgr_vec_t) -> i32;
    fn kgr_vec_len(v: *const kgr_vec_t) -> usize;
    fn kgr_vec_write(v: *mut kgr_vec_t, off: usize, host: *const u64, n: usize) -> i32;
    fn kgr_vec_fold_device(a: *const kgr_vec_t, b: *const kgr_vec_t, r: *const u64, out: *mut kgr_vec_t) -> i32;
    fn kgr_msm_vec(bases: *mut kgr_bases_t, base_off: usize, scalars: *const kgr_vec_t, sc_off: usize, n: usize, out: *mut u64) -> i32;
    fn kgr_pedersen_commit_vec(ck: *mut kgr_bases_t, m: *const kgr_vec_t, sc_off: usize, n: usize, out: *mut u64) -> i32;
    fn kgr_nova_cross_term_device(shape: *mut kgr_r1cs_t, z1: *const kgr_vec_t, z2: *const kgr_vec_t, t: *mut kgr_vec_t, ck: *mut kgr_bases_t,
                                  commit_out: *mut u64) -> i32;
    fn kgr_nova_is_sat(shape: *const kgr_r1cs_t, z: *const kgr_vec_t, e: *const kgr_vec_t, w_off: usize, ck: *mut kgr_bases_t, commit_w: *const u64,
                       commit_e: *const u64, report: *mut u64) -> i32;
    fn kgr_host_alloc(bytes: usize, out: *mut *mut c_void) -> i32;
    fn kgr_host_free(p: *mut c_void) -> i32;
    fn kgr_groth16_msms(log_n: u32, a: *const u64, b: *const u64, c: *const u64, m: usize, h: *mut kgr_bases_t, h_out: *mut u64, q_out: *mut u64,
                        q_len: *mut usize, jobs: *const kgr_msm_job_t, n_jobs: usize) -> i32;
    fn kgr_groth16_prove_r1cs(log_n: u32, cs: *const kgr_r1cs_t, z: *const kgr_vec_t, n_inputs: usize, h: *mut kgr_bases_t, l: *mut kgr_bases_t,
                              a: *mut kgr_bases_t, b_g1: *mut kgr_bases_t, b_g2: *mut kgr_bases_t, out: *mut u64, q_out: *mut u64, q_len: *mut usize,
                              jobs: *const kgr_msm_job_t, n_jobs: usize) -> i32;
    fn kgr_groth16_setup(cs: *const kgr_r1cs_t, n_inputs: usize, toxic: *const u64, log_n_out: *mut u32, h: *mut *mut kgr_bases_t,
                         l: *mut *mut kgr_bases_t, a: *mut *mut kgr_bases_t, b_g1: *mut *mut kgr_bases_t, b_g2: *mut *mut kgr_bases_t,
                         ic: *mut *mut kgr_bases_t, vk_g1: *mut u64, vk_g2: *mut u64) -> i32;
    fn kgr_groth16_setup_last_timing(ms: *mut f32) -> i32;
    fn kgr_pairing(g1: *const u64, g2: *const u64, n: usize, op: i32, out: *mut u64) -> i32;
    fn kgr_groth16_verify(vk_g1: *const u64, vk_g2: *const u64, ic: *mut kgr_bases_t, proofs: *const u64, k: usize, inputs: *const u64,
                          n_public: usize, rho: *const u64, ok: *mut u32) -> i32;
    fn kgr_set_param(name: *const c_char, value: c_long) -> i32;
    fn kgr_last_timing(dev: i32, ms: *mut f32, shape: *mut u32) -> i32;
    fn kgr_event_record(dev: i32, idx: i32) -> i32;
    fn kgr_event_elapsed_ms(dev: i32, idx_a: i32, idx_b: i32, ms: *mut f32) -> i32;
    fn kgr_launch_count(dev: i32, count: *mut u64) -> i32;
    fn kgr_test_field_op(field: i32, op: i32, a: *const u64, b: *const u64, n: usize, out: *mut u64) -> i32;
    fn kgr_test_point_op(curve: i32, op: i32, a_xy: *const u64, a_inf: *const u8, b_xy: *const u64, b_inf: *const u8, n: usize, out: *mut u64) -> i32;
    fn kgr_fixed_base_mul(curve: i32, k: *const u64, n: usize, out_xy: *mut u64) -> i32;
    fn kgr_bases_generate(curve: i32, seed: u64, n: usize, out: *mut *mut kgr_bases_t, k_out: *mut u64) -> i32;
    fn kgr_bases_generate_at(curve: i32, seed: u64, first: u64, n: usize, out: *mut *mut kgr_bases_t, k_out: *mut u64) -> i32;
    fn kgr_microbench(results: *mut f64) -> i32;
}

const SCALARS_MONTGOMERY: i32 = 0;
static INIT: Once = Once::new();

fn check(rc: i32) {
    if rc != 0 {
        let msg = unsafe { std::ffi::CStr::from_ptr(kgr_last_error()) }.to_string_lossy().into_owned();
        panic!("kgr_msm error {rc}: {msg}"); // the reference signature is infallible (it unwraps internally)
    }
}

fn ensure_init() {
    INIT.call_once(|| check(unsafe { kgr_init(core::ptr::null(), 0) }));
}

/// Select the GPUs explicitly (large MSMs are sharded evenly over them); otherwise the first call uses the current device.
pub fn init(devices: &[i32]) {
    INIT.call_once(|| {});
    check(unsafe { kgr_init(devices.as_ptr(), devices.len() as i32) });
}

/// Curves served by the GPU engine — the dispatch trait SURVEY.md H2 asks for: `msm_curve_addition` is ONE generic function in the
/// reference and the prover calls it with `G1Affine` six times and with `G2Affine` twice (groth16/src/prover.rs:51-65).
///
/// `LIMBS` = u64 limbs per coordinate: 4, or 8 for G2 whose coordinates are `Fq2 = c0 || c1` (bn254/src/fqn.rs).  `Fq2`'s array is
/// `pub(crate)` (zkstd/src/macros/extension_field.rs:17), so the G2 impl needs the one-line accessor `pub fn inner(&self) -> &[Fq; 2]`
/// added next to `Fq2::new_unchecked` (bn254/src/fqn.rs:245) — or `parity_scale_codec::Encode::encode(&x)`, which yields the same 64 bytes.
pub trait GpuCurve: BNAffine {
    const CURVE: i32;
    const LIMBS: usize;
    /// x || y as Montgomery limbs, appended to `dst` (2 * LIMBS words)
    fn write_coords(&self, dst: &mut Vec<u64>);
    fn scalar_limbs(s: &Self::Scalar) -> [u64; 4];
    /// (X, Y, Z) from 3 * LIMBS Montgomery limbs
    fn extended_from_limbs(w: &[u64]) -> Self::Extended;
}

fn l4(w: &[u64]) -> [u64; 4] {
    [w[0], w[1], w[2], w[3]]
}

impl GpuCurve for bn_254::G1Affine {
    const CURVE: i32 = 0;
    const LIMBS: usize = 4;
    fn write_coords(&self, dst: &mut Vec<u64>) {
        dst.extend_from_slice(self.get_x().inner()); // bn254/src/fq.rs:102
        dst.extend_from_slice(self.get_y().inner());
    }
    fn scalar_limbs(s: &bn_254::Fr) -> [u64; 4] {
        s.0 // bn254/src/fr.rs:71 (pub field, Montgomery form)
    }
    fn extended_from_limbs(w: &[u64]) -> bn_254::G1Projective {
        use bn_254::Fq;
        bn_254::G1Projective::new_unchecked(Fq::new_unchecked(l4(&w[0..4])), Fq::new_unchecked(l4(&w[4..8])), Fq::new_unchecked(l4(&w[8..12])))
    }
}

impl GpuCurve for grumpkin::Affine {
    const CURVE: i32 = 1;
    const LIMBS: usize = 4;
    fn write_coords(&self, dst: &mut Vec<u64>) {
        dst.extend_from_slice(self.get_x().inner()); // bn254/src/fr.rs:118
        dst.extend_from_slice(self.get_y().inner());
    }
    fn scalar_limbs(s: &bn_254::Fq) -> [u64; 4] {
        *s.inner()
    }
    fn extended_from_limbs(w: &[u64]) -> grumpkin::Projective {
        use bn_254::Fr;
        grumpkin::Projective::new_unchecked(Fr::new_unchecked(l4(&w[0..4])), Fr::new_unchecked(l4(&w[4..8])), Fr::new_unchecked(l4(&w[8..12])))
    }
}

impl GpuCurve for bn_254::G2Affine {
    const CURVE: i32 = 2;
    const LIMBS: usize = 8;
    fn write_coords(&self, dst: &mut Vec<u64>) {
        for c in [self.get_x(), self.get_y()] {
            let [c0, c1] = *c.inner(); // the accessor described above
            dst.extend_from_slice(c0.inner());
            dst.extend_from_slice(c1.inner());
        }
    }
    fn scalar_limbs(s: &bn_254::Fr) -> [u64; 4] {
        s.0
    }
    fn extended_from_limbs(w: &[u64]) -> bn_254::G2Projective {
        use bn_254::{Fq, Fq2};
        let fq2 = |v: &[u64]| Fq2::new_unchecked([Fq::new_unchecked(l4(&v[0..4])), Fq::new_unchecked(l4(&v[4..8]))]); // fqn.rs:245
        bn_254::G2Projective::new_unchecked(fq2(&w[0..8]), fq2(&w[8..16]), fq2(&w[16..24]))
    }
}

/// Page-locked staging memory that is reused from call to call (`kgr_host_alloc`): a fresh `Vec` per call is pageable, which costs the
/// library one extra staging copy (7.7 ms instead of 5.0 ms for a 2^20-point oneshot call, profiles/r01_e2e_pieces.md).
pub struct PinnedArena {
    ptr: *mut u64,
    cap_words: usize,
}

impl PinnedArena {
    pub const fn new() -> Self {
        Self { ptr: core::ptr::null_mut(), cap_words: 0 }
    }
    /// A slice of at least `words` u64 (grow-only).
    pub fn words(&mut self, words: usize) -> &mut [u64] {
        if words > self.cap_words {
            ensure_init();
            if !self.ptr.is_null() {
                unsafe { kgr_host_free(self.ptr as *mut c_void) };
            }
            let want = words + words / 4 + 64;
            let mut p: *mut c_void = core::ptr::null_mut();
            check(unsafe { kgr_host_alloc(want * 8, &mut p) });
            self.ptr = p as *mut u64;
            self.cap_words = want;
        }
        unsafe { core::slice::from_raw_parts_mut(self.ptr, words) }
    }
}

impl Drop for PinnedArena {
    fn drop(&mut self) {
        if !self.ptr.is_null() {
            unsafe { kgr_host_free(self.ptr as *mut c_void) };
        }
    }
}

thread_local! {
    // one arena per calling thread for points and one for scalars: the reference's callers issue their MSMs sequentially from one thread
    static POINTS: core::cell::RefCell<PinnedArena> = core::cell::RefCell::new(PinnedArena::new());
    static SCALARS: core::cell::RefCell<PinnedArena> = core::cell::RefCell::new(PinnedArena::new());
}

fn pack_points<C: GpuCurve>(bases: &[C]) -> (Vec<u64>, Vec<u8>) {
    // G1Affine is not repr(C) (bn254/src/g1.rs:17-22): copy (x, y, is_identity) into flat buffers
    let mut xy = Vec::with_capacity(2 * C::LIMBS * bases.len());
    let mut inf = Vec::with_capacity(bases.len());
    for b in bases {
        b.write_coords(&mut xy);
        inf.push(b.is_identity() as u8);
    }
    (xy, inf)
}

fn pack_scalars_into<C: GpuCurve>(coeffs: &[C::Scalar], dst: &mut [u64]) {
    for (s, d) in coeffs.iter().zip(dst.chunks_exact_mut(4)) {
        d.copy_from_slice(&C::scalar_limbs(s));
    }
}

/// Same signature and semantics as groth16/src/msm.rs:6 (pairs = zip(coeffs, bases), identity bases allowed, any projective
/// representative of the sum) for every curve the prover and Nova use, G2 included.
pub fn msm_curve_addition<C: GpuCurve>(bases: &[C], coeffs: &[C::Scalar]) -> C::Extended {
    ensure_init();
    let n = bases.len().min(coeffs.len());
    let mut out = [0u64; 24];
    POINTS.with(|pa| {
        SCALARS.with(|sa| {
            let (mut pa, mut sa) = (pa.borrow_mut(), sa.borrow_mut());
            let words = 2 * C::LIMBS;
            let xy = pa.words(words * n + (n + 7) / 8);
            let (xy, flags) = xy.split_at_mut(words * n);
            let flags = unsafe { core::slice::from_raw_parts_mut(flags.as_mut_ptr() as *mut u8, n) };
            let mut tmp = Vec::with_capacity(words);
            for (i, b) in bases[..n].iter().enumerate() {
                tmp.clear();
                b.write_coords(&mut tmp);
                xy[words * i..words * (i + 1)].copy_from_slice(&tmp);
                flags[i] = b.is_identity() as u8;
            }
            let sc = sa.words(4 * n);
            pack_scalars_into::<C>(&coeffs[..n], sc);
            check(unsafe { kgr_msm_oneshot(C::CURVE, xy.as_ptr(), flags.as_ptr(), n, sc.as_ptr(), SCALARS_MONTGOMERY, n, out.as_mut_ptr()) });
        })
    });
    C::extended_from_limbs(&out[..3 * C::LIMBS])
}

/// A base vector kept on the GPU(s): a CRS query (groth16/src/params.rs:7-29) or a Pedersen key (nova/src/pedersen.rs:6-8).
pub struct RegisteredBases<C: GpuCurve> {
    handle: *mut kgr_bases_t,
    len: usize,
    _curve: core::marker::PhantomData<C>,
}

impl<C: GpuCurve> RegisteredBases<C> {
    pub fn new(bases: &[C]) -> Self {
        ensure_init();
        let (xy, inf) = pack_points(bases);
        let mut handle = core::ptr::null_mut();
        check(unsafe { kgr_bases_register(C::CURVE, xy.as_ptr(), inf.as_ptr(), bases.len(), &mut handle) });
        Self { handle, len: bases.len(), _curve: core::marker::PhantomData }
    }

    pub fn len(&self) -> usize {
        unsafe { kgr_bases_len(self.handle) }
    }

    /// Window table 2^(c w) * P_i built once (W x the memory): every later MSM on this vector runs window-collapsed.
    pub fn precompute(&mut self) {
        check(unsafe { kgr_bases_precompute(self.handle, 0) });
    }

    /// sum_i coeffs[i] * bases[offset + i]   (e.g. `msm(&params.a[l..], aux)`, groth16/src/prover.rs:59)
    pub fn msm(&self, offset: usize, coeffs: &[C::Scalar]) -> C::Extended {
        let n = coeffs.len().min(self.len.saturating_sub(offset));
        let mut out = [0u64; 24];
        SCALARS.with(|sa| {
            let mut sa = sa.borrow_mut();
            let sc = sa.words(4 * n);
            pack_scalars_into::<C>(&coeffs[..n], sc);
            check(unsafe { kgr_msm(self.handle, offset, sc.as_ptr(), SCALARS_MONTGOMERY, n, out.as_mut_ptr()) });
        });
        C::extended_from_limbs(&out[..3 * C::LIMBS])
    }

    /// PedersenCommitment::commit (nova/src/pedersen.rs:15-20)
    pub fn commit(&self, m: &[C::Scalar]) -> C {
        self.msm(0, m).to_affine()
    }

    /// commit of elements [off, off + n) of a vector that lives on the GPU (the witness part of a resident z)
    pub fn commit_resident(&self, m: &DeviceVec, off: usize, n: usize) -> C {
        let mut out = [0u64; 24];
        check(unsafe { kgr_msm_vec(self.handle, 0, m.handle, off, n.min(self.len), out.as_mut_ptr()) });
        C::extended_from_limbs(&out[..3 * C::LIMBS]).to_affine()
    }
}

impl<C: GpuCurve> Drop for RegisteredBases<C> {
    fn drop(&mut self) {
        unsafe { kgr_bases_free(self.handle) };
    }
}

/// `Prover` (groth16/src/prover.rs:14-16) with `params.{h, l, a, b_g1, b_g2}` registered on the GPU once.
pub struct GpuProver {
    pub h: RegisteredBases<bn_254::G1Affine>,
    pub l: RegisteredBases<bn_254::G1Affine>,
    pub a: RegisteredBases<bn_254::G1Affine>,
    pub b_g1: RegisteredBases<bn_254::G1Affine>,
    pub b_g2: RegisteredBases<bn_254::G2Affine>,
}

/// The five query results of prover.rs:51-65 (the `inputs` / `aux` pairs of a, b_g1, b_g2 already added: they are one MSM over x ++ w each).
pub struct ProverQueries {
    pub q: bn_254::G1Projective,
    pub l: bn_254::G1Projective,
    pub a_answer: bn_254::G1Projective,
    pub b1_answer: bn_254::G1Projective,
    pub b2_answer: bn_254::G2Projective,
}

impl GpuProver {
    pub fn new(h: &[bn_254::G1Affine], l: &[bn_254::G1Affine], a: &[bn_254::G1Affine], b_g1: &[bn_254::G1Affine], b_g2: &[bn_254::G2Affine]) -> Self {
        Self { h: RegisteredBases::new(h), l: RegisteredBases::new(l), a: RegisteredBases::new(a), b_g1: RegisteredBases::new(b_g1), b_g2: RegisteredBases::new(b_g2) }
    }

    /// prover.rs:36-65 in one `kgr_groth16_msms` call: H on the device (seven NTTs) feeding `msm(params.h, q)` without leaving it, the other
    /// queries overlapped on separate lanes.  `a, b, c` = `cs.evaluate()`, `x` = `cs.x()`, `w` = `cs.w()` (Montgomery `Fr`), `log_n` = k.
    pub fn queries(&self, log_n: u32, a: &[bn_254::Fr], b: &[bn_254::Fr], c: &[bn_254::Fr], x: &[bn_254::Fr], w: &[bn_254::Fr]) -> ProverQueries {
        let flat = |v: &[bn_254::Fr]| v.iter().flat_map(|s| s.0).collect::<Vec<u64>>();
        let (fa, fb, fc, fw) = (flat(a), flat(b), flat(c), flat(w));
        let mut z = flat(x);
        z.extend_from_slice(&fw);
        let nz = x.len() + w.len();
        let (mut oh, mut ol, mut oa, mut ob1, mut ob2) = ([0u64; 12], [0u64; 12], [0u64; 12], [0u64; 12], [0u64; 24]);
        let job = |bases: *mut kgr_bases_t, len: usize, sc: &[u64], n: usize, out: *mut u64| kgr_msm_job_t {
            bases, base_off: 0, scalars: sc.as_ptr(), scalar_fmt: SCALARS_MONTGOMERY, n: n.min(len), out,
        };
        // the G2 query is the longest job: first, so that the G1 queries overlap with it
        let jobs = [job(self.b_g2.handle, self.b_g2.len, &z, nz, ob2.as_mut_ptr()), job(self.a.handle, self.a.len, &z, nz, oa.as_mut_ptr()),
                    job(self.b_g1.handle, self.b_g1.len, &z, nz, ob1.as_mut_ptr()), job(self.l.handle, self.l.len, &fw, w.len(), ol.as_mut_ptr())];
        check(unsafe {
            kgr_groth16_msms(log_n, fa.as_ptr(), fb.as_ptr(), fc.as_ptr(), a.len(), self.h.handle, oh.as_mut_ptr(), core::ptr::null_mut(),
                             core::ptr::null_mut(), jobs.as_ptr(), jobs.len())
        });
        use bn_254::{G1Affine, G2Affine};
        ProverQueries { q: G1Affine::extended_from_limbs(&oh), l: G1Affine::extended_from_limbs(&ol), a_answer: G1Affine::extended_from_limbs(&oa),
                        b1_answer: G1Affine::extended_from_limbs(&ob1), b2_answer: G2Affine::extended_from_limbs(&ob2) }
    }

    /// prover.rs:32-65 in one `kgr_groth16_prove_r1cs` call, straight after synthesis: `cs.evaluate()` on the device from the registered shape
    /// (`R1csShapeGpu` over Fr, columns `Wire::Instance(i) -> i`, `Wire::Witness(i) -> n_inputs + i`), H, and every query with its scalars read
    /// from the resident `z = cs.x() ++ cs.w()` (`DeviceVec` over Fr; `n_inputs = cs.x().len()`, the constant one first).  The blinding sums of
    /// :75-92 stay with the caller, as after `queries`.
    pub fn prove_r1cs(&self, log_n: u32, cs: &R1csShapeGpu, z: &DeviceVec, n_inputs: usize) -> ProverQueries {
        let mut out = [0u64; 72];
        check(unsafe {
            kgr_groth16_prove_r1cs(log_n, cs.handle, z.handle, n_inputs, self.h.handle, self.l.handle, self.a.handle, self.b_g1.handle, self.b_g2.handle,
                                   out.as_mut_ptr(), core::ptr::null_mut(), core::ptr::null_mut(), core::ptr::null(), 0)
        });
        use bn_254::{G1Affine, G2Affine};
        ProverQueries { q: G1Affine::extended_from_limbs(&out[0..12]), l: G1Affine::extended_from_limbs(&out[12..24]),
                        a_answer: G1Affine::extended_from_limbs(&out[24..36]), b1_answer: G1Affine::extended_from_limbs(&out[36..48]),
                        b2_answer: G2Affine::extended_from_limbs(&out[48..72]) }
    }
}

/// `Parameters` of `ZkSnark::setup` (groth16/src/zksnark.rs:17-127) generated on the GPU by `kgr_groth16_setup` (uncompiled, like the rest of this
/// file): the queries stay resident, the verifying key comes back as limbs (`vk_g1`: alpha, beta, delta as x[4] y[4] is_infinity; `vk_g2`: beta,
/// gamma, delta as x[8] y[8] is_infinity).  The h query has m - 1 entries as the reference's: proofs are guaranteed valid for m = 2^log_n only.
pub struct GpuParams {
    pub log_n: u32,
    pub prover: GpuProver,
    pub ic: RegisteredBases<bn_254::G1Affine>,
    pub vk_g1: [u64; 27],
    pub vk_g2: [u64; 51],
}

impl GpuParams {
    /// `cs`: the circuit's shape over Fr (columns `Wire::Instance(i) -> i`, `Wire::Witness(i) -> n_inputs + i`); `toxic`: alpha, beta, gamma, delta,
    /// tau (the five `Fr::random` draws of zksnark.rs:24-28).  The b_g2 query is always built here (the prover needs it).
    pub fn setup(cs: &R1csShapeGpu, n_inputs: usize, toxic: [bn_254::Fr; 5]) -> Self {
        let tox: Vec<u64> = toxic.iter().flat_map(|t| t.0).collect();
        let mut log_n = 0u32;
        let mut hs = [core::ptr::null_mut(); 6];
        let (mut vk_g1, mut vk_g2) = ([0u64; 27], [0u64; 51]);
        let [h, l, a, b_g1, b_g2, ic] = &mut hs;
        check(unsafe { kgr_groth16_setup(cs.handle, n_inputs, tox.as_ptr(), &mut log_n, h, l, a, b_g1, b_g2, ic, vk_g1.as_mut_ptr(), vk_g2.as_mut_ptr()) });
        fn adopt<C: GpuCurve>(handle: *mut kgr_bases_t) -> RegisteredBases<C> {
            RegisteredBases { handle, len: unsafe { kgr_bases_len(handle) }, _curve: core::marker::PhantomData }
        }
        let prover = GpuProver { h: adopt(hs[0]), l: adopt(hs[1]), a: adopt(hs[2]), b_g1: adopt(hs[3]), b_g2: adopt(hs[4]) };
        Self { log_n, prover, ic: adopt(hs[5]), vk_g1, vk_g2 }
    }

    /// Device time (ms) of the phases of the last setup (`kgr_groth16_setup_last_timing`).
    pub fn last_timing() -> [f32; 10] {
        let mut ms = [0f32; 10];
        check(unsafe { kgr_groth16_setup_last_timing(ms.as_mut_ptr()) });
        ms
    }
}

/// Several independent MSMs on registered G1 vectors in one call (`kgr_msm_batch`): results in job order.
pub fn msm_batch(jobs: &[(&RegisteredBases<bn_254::G1Affine>, usize, &[bn_254::Fr])]) -> Vec<bn_254::G1Projective> {
    let scalars: Vec<Vec<u64>> = jobs.iter().map(|(_, _, s)| s.iter().flat_map(|x| x.0).collect()).collect();
    let mut outs = vec![[0u64; 12]; jobs.len()];
    let raw: Vec<kgr_msm_job_t> = jobs.iter().zip(scalars.iter()).zip(outs.iter_mut()).map(|(((b, off, s), sc), o)| kgr_msm_job_t {
        bases: b.handle, base_off: *off, scalars: sc.as_ptr(), scalar_fmt: SCALARS_MONTGOMERY, n: s.len().min(b.len.saturating_sub(*off)), out: o.as_mut_ptr(),
    }).collect();
    check(unsafe { kgr_msm_batch(raw.as_ptr(), raw.len()) });
    outs.iter().map(|o| <bn_254::G1Affine as GpuCurve>::extended_from_limbs(o)).collect()
}

/// `Fft::<Fr>::{dft, idft, coset_dft, coset_idft}` (groth16/src/fft.rs:92-127): op 0..3, zero padding and trailing-zero stripping as there.
pub fn ntt(log_n: u32, op: i32, values: &[bn_254::Fr]) -> Vec<bn_254::Fr> {
    ensure_init();
    let flat: Vec<u64> = values.iter().flat_map(|s| s.0).collect();
    let mut out = vec![0u64; 4 << log_n];
    let mut n_out = 0usize;
    check(unsafe { kgr_ntt(log_n, op, flat.as_ptr(), values.len(), out.as_mut_ptr(), &mut n_out) });
    out[..4 * n_out].chunks_exact(4).map(|w| bn_254::Fr(l4(w))).collect()
}

/// prover.rs:36-47: the coefficients of H from the R1CS evaluations.
pub fn groth16_h(log_n: u32, a: &[bn_254::Fr], b: &[bn_254::Fr], c: &[bn_254::Fr]) -> Vec<bn_254::Fr> {
    ensure_init();
    let flat = |v: &[bn_254::Fr]| v.iter().flat_map(|s| s.0).collect::<Vec<u64>>();
    let (fa, fb, fc) = (flat(a), flat(b), flat(c));
    let mut out = vec![0u64; 4 << log_n];
    let mut n_out = 0usize;
    check(unsafe { kgr_groth16_h(log_n, fa.as_ptr(), fb.as_ptr(), fc.as_ptr(), a.len(), out.as_mut_ptr(), &mut n_out) });
    out[..4 * n_out].chunks_exact(4).map(|w| bn_254::Fr(l4(w))).collect()
}

/// A vector of field elements resident on the GPU (`kgr_vec_t`): nova's z = (u, x, w), E and T between folding steps
/// (nova/src/relaxed_r1cs/witness.rs:20-21).  `field`: 0 = Fq (GrumpkinDriver), 1 = Fr (Bn254Driver); limbs are Montgomery.
pub struct DeviceVec {
    handle: *mut kgr_vec_t,
}

impl DeviceVec {
    pub fn upload(field: i32, limbs: &[u64]) -> Self {
        ensure_init();
        let mut handle = core::ptr::null_mut();
        check(unsafe { kgr_vec_upload(field, limbs.as_ptr(), limbs.len() / 4, &mut handle) });
        Self { handle }
    }
    pub fn zeros(field: i32, n: usize) -> Self {
        ensure_init();
        let mut handle = core::ptr::null_mut();
        check(unsafe { kgr_vec_upload(field, core::ptr::null(), n, &mut handle) });
        Self { handle }
    }
    pub fn len(&self) -> usize {
        unsafe { kgr_vec_len(self.handle) }
    }
    pub fn download(&self) -> Vec<u64> {
        let mut out = vec![0u64; 4 * self.len()];
        check(unsafe { kgr_vec_download(self.handle, 0, self.len(), out.as_mut_ptr()) });
        out
    }
    pub fn write(&mut self, off: usize, limbs: &[u64]) {
        check(unsafe { kgr_vec_write(self.handle, off, limbs.as_ptr(), limbs.len() / 4) });
    }
    /// self <- self + other * r   (RelaxedR1csWitness::fold, witness.rs:67-68)
    pub fn fold(&mut self, other: &DeviceVec, r: [u64; 4]) {
        check(unsafe { kgr_vec_fold_device(self.handle, other.handle, r.as_ptr(), self.handle) });
    }
}

impl Drop for DeviceVec {
    fn drop(&mut self) {
        unsafe { kgr_vec_free(self.handle) };
    }
}

/// `R1csShape` (nova/src/relaxed_r1cs.rs) resident on the GPU: A, B, C in CSR over flat columns of z = (u, x, w).
pub struct R1csShapeGpu {
    handle: *mut kgr_r1cs_t,
    pub m: usize,
    pub n_z: usize,
}

impl R1csShapeGpu {
    /// matrices[k] = (row_ptr (m + 1), cols (nnz), coeffs (nnz x 4 Montgomery limbs)) for k = A, B, C
    pub fn new(field: i32, m: usize, n_z: usize, matrices: [(&[u32], &[u32], &[u64]); 3]) -> Self {
        ensure_init();
        let rp = [matrices[0].0.as_ptr(), matrices[1].0.as_ptr(), matrices[2].0.as_ptr()];
        let cl = [matrices[0].1.as_ptr(), matrices[1].1.as_ptr(), matrices[2].1.as_ptr()];
        let cf = [matrices[0].2.as_ptr(), matrices[1].2.as_ptr(), matrices[2].2.as_ptr()];
        let mut handle = core::ptr::null_mut();
        check(unsafe { kgr_r1cs_register(field, m, n_z, rp.as_ptr(), cl.as_ptr(), cf.as_ptr(), &mut handle) });
        Self { handle, m, n_z }
    }
    /// compute_cross_term + ck.commit(&t) (nova/src/prover.rs:33-35) with everything resident: T is left in `t`, the commitment comes back
    pub fn cross_term_commit<C: GpuCurve>(&self, z1: &DeviceVec, z2: &DeviceVec, t: &mut DeviceVec, ck: &RegisteredBases<C>) -> [u64; 9] {
        let mut commit = [0u64; 9];
        check(unsafe { kgr_nova_cross_term_device(self.handle, z1.handle, z2.handle, t.handle, ck.handle, commit.as_mut_ptr()) });
        commit
    }
    /// host-buffer variant (kgr_nova_cross_term): T copied back, optional commitment
    pub fn cross_term_host(&self, z1: &[u64], z2: &[u64]) -> Vec<u64> {
        let mut t = vec![0u64; 4 * self.m];
        check(unsafe { kgr_nova_cross_term(self.handle, z1.as_ptr(), z2.as_ptr(), t.as_mut_ptr(), core::ptr::null_mut(), core::ptr::null_mut()) });
        t
    }
    /// `R1csShape::is_sat` (nova/src/relaxed_r1cs.rs:117-146) on the resident z = (1, x, w): (A z) o (B z) = C z row by row and, with a key,
    /// commit(z[w_off ..]) == commit_w.  `report` as `kgr_nova_is_sat`: [0] sat, [1] violating rows, [2] first of them (m if none), [3] commit(W)
    /// 1 equal / 0 different / 2 not checked, [4] 2, [5] z[0] == 1.
    pub fn is_sat<C: GpuCurve>(&self, z: &DeviceVec, w_off: usize, ck: Option<(&RegisteredBases<C>, &[u64; 9])>) -> [u64; 6] {
        let mut report = [0u64; 6];
        let (key, cw) = ck.map_or((core::ptr::null_mut(), core::ptr::null()), |(b, c)| (b.handle, c.as_ptr()));
        check(unsafe { kgr_nova_is_sat(self.handle, z.handle, core::ptr::null(), w_off, key, cw, core::ptr::null(), report.as_mut_ptr()) });
        report
    }
    /// The relaxed relation (relaxed_r1cs.rs:80-114), u = z[0], with E resident; each expected commitment is optional (`None` skips that check).
    pub fn is_sat_relaxed<C: GpuCurve>(&self, z: &DeviceVec, e: &DeviceVec, w_off: usize, ck: Option<&RegisteredBases<C>>, commit_w: Option<&[u64; 9]>,
                                       commit_e: Option<&[u64; 9]>) -> [u64; 6] {
        let mut report = [0u64; 6];
        let key = ck.map_or(core::ptr::null_mut(), |b| b.handle);
        let cw = commit_w.map_or(core::ptr::null(), |c| c.as_ptr());
        let ce = commit_e.map_or(core::ptr::null(), |c| c.as_ptr());
        check(unsafe { kgr_nova_is_sat(self.handle, z.handle, e.handle, w_off, key, cw, ce, report.as_mut_ptr()) });
        report
    }
    /// SparseMatrix::prod (zkstd/src/matrix.rs:36-48): which = 0 A, 1 B, 2 C
    pub fn prod(&self, which: i32, z: &[u64]) -> Vec<u64> {
        let mut out = vec![0u64; 4 * self.m];
        check(unsafe { kgr_r1cs_mul(self.handle, which, z.as_ptr(), out.as_mut_ptr()) });
        out
    }
}

impl Drop for R1csShapeGpu {
    fn drop(&mut self) {
        unsafe { kgr_r1cs_free(self.handle) };
    }
}

/// out[i] = a[i] + b[i] * r with host buffers (kgr_vec_fold); `DeviceVec::fold` is the resident form.
pub fn vec_fold(field: i32, a: &[u64], b: &[u64], r: [u64; 4]) -> Vec<u64> {
    ensure_init();
    let n = a.len().min(b.len()) / 4;
    let mut out = vec![0u64; 4 * n];
    check(unsafe { kgr_vec_fold(field, a.as_ptr(), b.as_ptr(), r.as_ptr(), n, out.as_mut_ptr()) });
    out
}

/// Bindings that exist for tests, benchmarks and tools; listed so that the extern block above is the complete ABI.
#[allow(dead_code)]
mod unused {
    use super::*;
    pub(crate) unsafe fn touch() {
        let _ = (kgr_shutdown as usize, kgr_device_count as usize, kgr_msm_device as usize, kgr_bases_download as usize, kgr_pedersen_commit as usize,
                 kgr_to_affine as usize, kgr_proj_add as usize, kgr_ntt_device as usize, kgr_r1cs_last_timing as usize, kgr_pedersen_commit_vec as usize,
                 kgr_set_param as usize, kgr_last_timing as usize, kgr_event_record as usize, kgr_event_elapsed_ms as usize, kgr_launch_count as usize,
                 kgr_test_field_op as usize, kgr_test_point_op as usize, kgr_fixed_base_mul as usize, kgr_bases_generate as usize,
                 kgr_bases_generate_at as usize, kgr_microbench as usize);
    }
}

/// `groth16/src/verifier.rs` on the GPU (`kgr_groth16_verify`, uncompiled like the rest of this file): the verifying key as the limbs `GpuParams`
/// holds and the ic query borrowed from it.  `proofs`: per proof A[9] B[17] C[9] (x, y, is_infinity; Montgomery limbs); `inputs`: per proof the
/// public inputs without the leading one.  For two or more proofs one batched pairing check runs with the caller's 128-bit weights `rho`
/// (non-zero, unpredictable to the prover); if it fails, every proof is checked on its own.
pub struct GpuVerifier<'a> {
    pub vk_g1: [u64; 27],
    pub vk_g2: [u64; 51],
    pub ic: &'a RegisteredBases<bn_254::G1Affine>,
}

impl<'a> GpuVerifier<'a> {
    pub fn from_params(params: &'a GpuParams) -> Self {
        Self { vk_g1: params.vk_g1, vk_g2: params.vk_g2, ic: &params.ic }
    }

    pub fn verify(&self, proofs: &[[u64; 35]], inputs: &[Vec<bn_254::Fr>], rho: &[[u64; 2]]) -> Vec<bool> {
        let k = proofs.len();
        let n_public = self.ic.len - 1;
        assert!(inputs.len() == k && inputs.iter().all(|x| x.len() == n_public));
        let flat_p: Vec<u64> = proofs.iter().flat_map(|p| p.iter().copied()).collect();
        let flat_x: Vec<u64> = inputs.iter().flat_map(|x| x.iter().flat_map(|s| s.0)).collect();
        let flat_r: Vec<u64> = rho.iter().flat_map(|r| r.iter().copied()).collect();
        let mut ok = vec![0u32; k];
        check(unsafe {
            kgr_groth16_verify(self.vk_g1.as_ptr(), self.vk_g2.as_ptr(), self.ic.handle, flat_p.as_ptr(), k, flat_x.as_ptr(), n_public,
                               if k >= 2 { flat_r.as_ptr() } else { core::ptr::null() }, ok.as_mut_ptr())
        });
        ok.into_iter().map(|v| v != 0).collect()
    }
}
