//! bpg -- safe Rust surface over libbpg for the five hot entry points of the reference
//! (SURVEY.md section 8b / INTEGRATION.md section 3):
//!
//!   BulletproofGens::new(cap, 1) / PedersenGens::default()   -> Device::gens_ensure          prover.rs:53,92  verifier.rs:89
//!   PedersenGens::commit(v, r)                                -> Device::pedersen_commit      gadget.rs:31  commitments.rs:27,39  cs_buffer.rs:39
//!   Prover::prove(&bp_gens)                                   -> Device::r1cs_prove           prover.rs:93
//!   Verifier::verify(&proof, &pc_gens, &bp_gens)              -> Device::r1cs_verify          verifier.rs:90
//!   mimc_hash(&Vec<u8>)                                       -> Device::mimc_hash            mimc.rs:61 (callers prover.rs:171,197,325 verifier.rs:451)
//!
//! Scalars and points cross the boundary as the 32-byte encodings dalek already uses (`Scalar::as_bytes`,
//! `CompressedRistretto::as_bytes`), so this crate needs no curve25519-dalek types.  One `Device` per thread (a bpg_ctx is
//! not thread-safe); `Device::global()` is the process-wide one the patched fork uses from its (single-threaded) call sites.
#[macro_use]
extern crate lazy_static;
extern crate rand;

pub mod ffi;

use std::ptr;
use std::sync::Mutex;

#[derive(Debug, Clone, PartialEq)]
pub enum BpgError {
    Cuda(String),
    InvalidGeneratorsLength,
    Decompress,
    Argument,
    Format,
    NoMemory,
    Comm(String),
}

pub struct Device { ctx: *mut ffi::BpgCtx, mimc_ready: bool }
unsafe impl Send for Device {}

lazy_static! {
    static ref GLOBAL: Mutex<Device> = Mutex::new(Device::new(0).expect("no CUDA device: libbpg has no CPU fallback"));
}

/// The constraint system of one proof in the flat form bpg_circuit_create takes: constraint r is
/// sum_k coeff[k] * var[k] = 0 over k in row_ptr[r]..row_ptr[r+1]; var = kind << 29 | index,
/// kind 0 = a_L, 1 = a_R, 2 = a_O, 3 = V, 4 = One (r1cs::Variable as recorded by ConstraintSystem::constrain).
pub struct FlatConstraints { pub row_ptr: Vec<u32>, pub term_var: Vec<u32>, pub term_coeff: Vec<u8> }

/// One statement of Device::r1cs_prove_batch: the arguments of one Device::r1cs_prove call.
pub struct ProveJob<'a> {
    pub label: &'a [u8],
    pub cs: &'a FlatConstraints,
    pub a_l: &'a [u8],
    pub a_r: &'a [u8],
    pub a_o: &'a [u8],
    pub v: &'a [u8],
    pub v_blinding: &'a [u8],
}

/// One statement of Device::r1cs_verify_each: the arguments of one Device::r1cs_verify call.
pub struct VerifyJob<'a> {
    pub label: &'a [u8],
    pub cs: &'a FlatConstraints,
    pub n: usize,
    pub commitments: &'a [u8],
    pub proof: &'a [u8],
}

pub const VAR_L: u32 = 0;
pub const VAR_R: u32 = 1;
pub const VAR_O: u32 = 2;
pub const VAR_V: u32 = 3;
pub const VAR_ONE: u32 = 4;

impl FlatConstraints {
    pub fn new() -> Self { FlatConstraints { row_ptr: vec![0], term_var: Vec::new(), term_coeff: Vec::new() } }
    /// one LinearCombination: (kind, index, coefficient bytes) terms
    pub fn push_row<'a, I: IntoIterator<Item = (u32, usize, &'a [u8; 32])>>(&mut self, terms: I) {
        for (kind, index, coeff) in terms {
            self.term_var.push((kind << 29) | index as u32);
            self.term_coeff.extend_from_slice(coeff);
        }
        self.row_ptr.push(self.term_var.len() as u32);
    }
    pub fn rows(&self) -> usize { self.row_ptr.len() - 1 }
}

impl Device {
    pub fn new(device: i32) -> Result<Device, BpgError> {
        let mut ctx = ptr::null_mut();
        let rc = unsafe { ffi::bpg_ctx_create(device, &mut ctx) };
        if rc != ffi::BPG_OK { return Err(Device::error(ptr::null_mut(), rc)); }
        Ok(Device { ctx: ctx, mimc_ready: false })
    }
    pub fn global() -> std::sync::MutexGuard<'static, Device> { GLOBAL.lock().unwrap() }

    fn error(ctx: *mut ffi::BpgCtx, rc: i32) -> BpgError {
        let msg = unsafe {
            let p = ffi::bpg_last_error(ctx);
            if p.is_null() { String::new() } else { std::ffi::CStr::from_ptr(p).to_string_lossy().into_owned() }
        };
        match rc {
            ffi::BPG_E_CUDA => BpgError::Cuda(msg),
            ffi::BPG_E_SIZE => BpgError::InvalidGeneratorsLength,
            ffi::BPG_E_DECOMPRESS => BpgError::Decompress,
            ffi::BPG_E_FORMAT => BpgError::Format,
            ffi::BPG_E_NOMEM => BpgError::NoMemory,
            ffi::BPG_E_COMM => BpgError::Comm(msg),
            _ => BpgError::Argument,
        }
    }
    fn check(&self, rc: i32) -> Result<(), BpgError> { if rc == ffi::BPG_OK { Ok(()) } else { Err(Device::error(self.ctx, rc)) } }

    /// BulletproofGens::new(capacity, 1) + PedersenGens::default(): generators resident in HBM (idempotent)
    pub fn gens_ensure(&mut self, capacity: usize) -> Result<(), BpgError> {
        let rc = unsafe { ffi::bpg_gens_ensure(self.ctx, capacity) };
        self.check(rc)
    }
    /// compressed G[i0..i0+n), H[i0..i0+n) for the host-side accessors of BulletproofGens
    pub fn gens_export(&mut self, i0: usize, n: usize) -> Result<(Vec<u8>, Vec<u8>), BpgError> {
        let (mut g, mut h) = (vec![0u8; 32 * n], vec![0u8; 32 * n]);
        let rc = unsafe { ffi::bpg_gens_export(self.ctx, i0, n, g.as_mut_ptr(), h.as_mut_ptr()) };
        self.check(rc).map(|_| (g, h))
    }
    /// PedersenGens::commit for n openings at once: values / blindings are n x 32 bytes (Scalar::as_bytes)
    pub fn pedersen_commit(&mut self, values: &[u8], blindings: &[u8]) -> Result<Vec<u8>, BpgError> {
        assert!(values.len() == blindings.len() && values.len() % 32 == 0);
        let n = values.len() / 32;
        let mut out = vec![0u8; 32 * n];
        let rc = unsafe { ffi::bpg_pedersen_commit(self.ctx, values.as_ptr(), blindings.as_ptr(), n, out.as_mut_ptr()) };
        self.check(rc).map(|_| out)
    }
    /// RistrettoPoint::vartime_multiscalar_mul / optional_multiscalar_mul (None if a point fails to decode)
    pub fn msm(&mut self, scalars: &[u8], points: &[u8]) -> Result<Option<[u8; 32]>, BpgError> {
        assert!(scalars.len() == points.len() && scalars.len() % 32 == 0);
        let mut out = [0u8; 32];
        let rc = unsafe { ffi::bpg_msm(self.ctx, scalars.as_ptr(), points.as_ptr(), scalars.len() / 32, out.as_mut_ptr()) };
        if rc == ffi::BPG_E_DECOMPRESS { return Ok(None); }
        self.check(rc).map(|_| Some(out))
    }
    /// Prover::prove: label = the bytes given to Transcript::new, a_l/a_r/a_o = n x 32 bytes, v/v_blinding = m x 32 bytes.
    /// Returns (R1CSProof::to_bytes(), m compressed commitments).  The 32 bytes the reference's TranscriptRngBuilder::finalize
    /// draws from thread_rng are drawn here with the same generator.
    pub fn r1cs_prove(&mut self, label: &[u8], cs: &FlatConstraints, a_l: &[u8], a_r: &[u8], a_o: &[u8], v: &[u8], v_blinding: &[u8],
                      flags: u32) -> Result<(Vec<u8>, Vec<u8>), BpgError> {
        use rand::RngCore;
        let (n, m) = (a_l.len() / 32, v.len() / 32);
        assert!(a_r.len() == a_l.len() && a_o.len() == a_l.len() && v_blinding.len() == v.len());
        let mut ext = [0u8; 32];
        rand::thread_rng().fill_bytes(&mut ext);
        let mut circuit = ptr::null_mut();
        let rc = unsafe { ffi::bpg_circuit_create(self.ctx, n, m, cs.rows(), cs.row_ptr.as_ptr(), cs.term_var.as_ptr(), cs.term_coeff.as_ptr(), &mut circuit) };
        self.check(rc)?;
        let cap = 1 + 32 * (14 + 64 + 2);
        let (mut proof, mut vout) = (vec![0u8; cap], vec![0u8; 32 * std::cmp::max(m, 1)]);
        let len = unsafe {
            ffi::bpg_r1cs_prove(self.ctx, circuit, label.as_ptr(), label.len(), a_l.as_ptr(), a_r.as_ptr(), a_o.as_ptr(), v.as_ptr(),
                                v_blinding.as_ptr(), ext.as_ptr(), flags, vout.as_mut_ptr(), proof.as_mut_ptr(), cap)
        };
        unsafe { ffi::bpg_circuit_destroy(circuit) };
        if len < 0 { return Err(Device::error(self.ctx, len as i32)); }
        proof.truncate(len as usize);
        vout.truncate(32 * m);
        Ok((proof, vout))
    }
    /// Prover::prove for many statements in one call (bpg_r1cs_prove_batch): entry i is what r1cs_prove returns for jobs[i]
    /// with the same thread_rng bytes.  Small circuits (padded size <= 4096) are proved in lockstep, larger ones one by one.
    pub fn r1cs_prove_batch(&mut self, jobs: &[ProveJob], flags: u32) -> Result<Vec<(Vec<u8>, Vec<u8>)>, BpgError> {
        use rand::RngCore;
        let k = jobs.len();
        let mut ext = vec![0u8; 32 * k];
        rand::thread_rng().fill_bytes(&mut ext);
        for j in jobs {
            assert!(j.a_r.len() == j.a_l.len() && j.a_o.len() == j.a_l.len() && j.v_blinding.len() == j.v.len());
        }
        // every circuit in one call (one device allocation shared by the k handles)
        let ns: Vec<usize> = jobs.iter().map(|j| j.a_l.len() / 32).collect();
        let ms: Vec<usize> = jobs.iter().map(|j| j.v.len() / 32).collect();
        let qs: Vec<usize> = jobs.iter().map(|j| j.cs.rows()).collect();
        let row_ptrs: Vec<*const u32> = jobs.iter().map(|j| j.cs.row_ptr.as_ptr()).collect();
        let term_vars: Vec<*const u32> = jobs.iter().map(|j| j.cs.term_var.as_ptr()).collect();
        let term_coeffs: Vec<*const u8> = jobs.iter().map(|j| j.cs.term_coeff.as_ptr()).collect();
        let mut circuits: Vec<*mut ffi::BpgCircuit> = vec![ptr::null_mut(); k];
        let rc = unsafe {
            ffi::bpg_circuit_create_batch(self.ctx, k, ns.as_ptr(), ms.as_ptr(), qs.as_ptr(), row_ptrs.as_ptr(), term_vars.as_ptr(), term_coeffs.as_ptr(),
                                          circuits.as_mut_ptr())
        };
        self.check(rc)?;
        let cap = 1 + 32 * (14 + 64 + 2);
        let mut proofs: Vec<Vec<u8>> = (0..k).map(|_| vec![0u8; cap]).collect();
        let mut vouts: Vec<Vec<u8>> = jobs.iter().map(|j| vec![0u8; std::cmp::max(j.v.len(), 32)]).collect();
        let labels: Vec<*const u8> = jobs.iter().map(|j| j.label.as_ptr()).collect();
        let label_lens: Vec<usize> = jobs.iter().map(|j| j.label.len()).collect();
        let a_l: Vec<*const u8> = jobs.iter().map(|j| j.a_l.as_ptr()).collect();
        let a_r: Vec<*const u8> = jobs.iter().map(|j| j.a_r.as_ptr()).collect();
        let a_o: Vec<*const u8> = jobs.iter().map(|j| j.a_o.as_ptr()).collect();
        let v: Vec<*const u8> = jobs.iter().map(|j| j.v.as_ptr()).collect();
        let v_blinding: Vec<*const u8> = jobs.iter().map(|j| j.v_blinding.as_ptr()).collect();
        let vout_ptrs: Vec<*mut u8> = vouts.iter_mut().map(|x| x.as_mut_ptr()).collect();
        let proof_ptrs: Vec<*mut u8> = proofs.iter_mut().map(|x| x.as_mut_ptr()).collect();
        let caps = vec![cap; k];
        let mut lens = vec![0usize; k];
        let rc = unsafe {
            ffi::bpg_r1cs_prove_batch(self.ctx, k, circuits.as_ptr(), labels.as_ptr(), label_lens.as_ptr(), a_l.as_ptr(), a_r.as_ptr(), a_o.as_ptr(),
                                      v.as_ptr(), v_blinding.as_ptr(), ext.as_ptr(), flags, vout_ptrs.as_ptr(), proof_ptrs.as_ptr(), caps.as_ptr(),
                                      lens.as_mut_ptr())
        };
        for c in &circuits { unsafe { ffi::bpg_circuit_destroy(*c) } }
        self.check(rc)?;
        let mut out = Vec::with_capacity(k);
        for (i, (mut proof, mut vout)) in proofs.into_iter().zip(vouts.into_iter()).enumerate() {
            proof.truncate(lens[i]);
            vout.truncate(jobs[i].v.len());
            out.push((proof, vout));
        }
        Ok(out)
    }
    /// Verifier::verify: Ok(true) for Ok(()), Ok(false) for Err(VerificationError | FormatError)
    pub fn r1cs_verify(&mut self, label: &[u8], cs: &FlatConstraints, n: usize, commitments: &[u8], proof: &[u8], flags: u32) -> Result<bool, BpgError> {
        use rand::RngCore;
        let m = commitments.len() / 32;
        let mut ext = [0u8; 32];
        rand::thread_rng().fill_bytes(&mut ext);
        let mut circuit = ptr::null_mut();
        let rc = unsafe { ffi::bpg_circuit_create(self.ctx, n, m, cs.rows(), cs.row_ptr.as_ptr(), cs.term_var.as_ptr(), cs.term_coeff.as_ptr(), &mut circuit) };
        self.check(rc)?;
        let mut accept = 0i32;
        let rc = unsafe {
            ffi::bpg_r1cs_verify(self.ctx, circuit, label.as_ptr(), label.len(), commitments.as_ptr(), proof.as_ptr(), proof.len(), ext.as_ptr(), flags, &mut accept)
        };
        unsafe { ffi::bpg_circuit_destroy(circuit) };
        self.check(rc).map(|_| accept == 1)
    }
    /// Verifier::verify for many statements in one call (bpg_r1cs_verify_each): entry i is exactly what r1cs_verify returns for
    /// jobs[i]; every proof is checked against its own equation, small ones (padded size <= 4096) in lockstep.
    pub fn r1cs_verify_each(&mut self, jobs: &[VerifyJob], flags: u32) -> Result<Vec<bool>, BpgError> {
        use rand::RngCore;
        let k = jobs.len();
        let mut ext = vec![0u8; 32 * k];
        rand::thread_rng().fill_bytes(&mut ext);
        let ns: Vec<usize> = jobs.iter().map(|j| j.n).collect();
        let ms: Vec<usize> = jobs.iter().map(|j| j.commitments.len() / 32).collect();
        let qs: Vec<usize> = jobs.iter().map(|j| j.cs.rows()).collect();
        let row_ptrs: Vec<*const u32> = jobs.iter().map(|j| j.cs.row_ptr.as_ptr()).collect();
        let term_vars: Vec<*const u32> = jobs.iter().map(|j| j.cs.term_var.as_ptr()).collect();
        let term_coeffs: Vec<*const u8> = jobs.iter().map(|j| j.cs.term_coeff.as_ptr()).collect();
        let mut circuits: Vec<*mut ffi::BpgCircuit> = vec![ptr::null_mut(); k];
        let rc = unsafe {
            ffi::bpg_circuit_create_batch(self.ctx, k, ns.as_ptr(), ms.as_ptr(), qs.as_ptr(), row_ptrs.as_ptr(), term_vars.as_ptr(), term_coeffs.as_ptr(),
                                          circuits.as_mut_ptr())
        };
        self.check(rc)?;
        let labels: Vec<*const u8> = jobs.iter().map(|j| j.label.as_ptr()).collect();
        let label_lens: Vec<usize> = jobs.iter().map(|j| j.label.len()).collect();
        let vs: Vec<*const u8> = jobs.iter().map(|j| j.commitments.as_ptr()).collect();
        let proofs: Vec<*const u8> = jobs.iter().map(|j| j.proof.as_ptr()).collect();
        let proof_lens: Vec<usize> = jobs.iter().map(|j| j.proof.len()).collect();
        let mut accept = vec![0i32; k];
        let rc = unsafe {
            ffi::bpg_r1cs_verify_each(self.ctx, k, circuits.as_ptr(), labels.as_ptr(), label_lens.as_ptr(), vs.as_ptr(), proofs.as_ptr(),
                                      proof_lens.as_ptr(), ext.as_ptr(), flags, accept.as_mut_ptr())
        };
        for c in &circuits { unsafe { ffi::bpg_circuit_destroy(*c) } }
        self.check(rc).map(|_| accept.iter().map(|&a| a == 1).collect())
    }
    /// install ROUND_CONSTANTS_769 (mimc_consts.rs:2-489) once: 486 x 32 bytes
    pub fn mimc_set_constants(&mut self, consts: &[u8]) -> Result<(), BpgError> {
        assert!(consts.len() == 486 * 32);
        let rc = unsafe { ffi::bpg_mimc_set_constants(self.ctx, consts.as_ptr()) };
        self.mimc_ready = rc == ffi::BPG_OK;
        self.check(rc)
    }
    /// mimc_hash for a batch of preimages (mimc.rs:61-75): returns n x 32 bytes (Scalar bytes)
    pub fn mimc_hash(&mut self, preimages: &[&[u8]]) -> Result<Vec<u8>, BpgError> {
        assert!(self.mimc_ready, "call mimc_set_constants first");
        let mut data = Vec::new();
        let mut offs = vec![0u64];
        for p in preimages { data.extend_from_slice(p); offs.push(data.len() as u64); }
        let mut out = vec![0u8; 32 * preimages.len()];
        let rc = unsafe { ffi::bpg_mimc_hash_batch(self.ctx, data.as_ptr(), offs.as_ptr(), preimages.len(), out.as_mut_ptr()) };
        self.check(rc).map(|_| out)
    }
    /// unpadded sponge (Merkle nodes, merkle_tree_gadget.rs:7-12) with the in-circuit witness trace of every absorbed block:
    /// 972 x (a_L, a_R, a_O) x 32 bytes per block in gadget order (mimc_hash_gadget.rs:133-144)
    pub fn mimc_sponge_trace(&mut self, blocks: &[u8], block_off: &[u32]) -> Result<(Vec<u8>, Vec<u8>), BpgError> {
        assert!(self.mimc_ready, "call mimc_set_constants first");
        let n = block_off.len() - 1;
        let nblocks = block_off[n] as usize;
        let (mut out, mut trace) = (vec![0u8; 32 * n], vec![0u8; nblocks * 972 * 96]);
        let rc = unsafe { ffi::bpg_mimc_sponge_batch(self.ctx, blocks.as_ptr(), block_off.as_ptr(), n, out.as_mut_ptr(), trace.as_mut_ptr()) };
        self.check(rc).map(|_| (out, trace))
    }
}

impl Drop for Device {
    fn drop(&mut self) { unsafe { ffi::bpg_ctx_destroy(self.ctx) } }
}
