//! ffi.rs -- the C ABI of libbpg (include/bpg.h) as a Rust `extern "C"` block, one declaration per header prototype, in header order.
//!
//! This file is what the patched `bulletproofs` fork (Cargo.toml:17-20 of the reference) and this crate's `mimc_hash`
//! (src/mimc_hash/mimc.rs:61) bind against.  tests/test_abi_and_host.py::test_rust_ffi_matches_header checks name, order and
//! arity of every declaration against include/bpg.h (no Rust toolchain exists in the build image, so the check is textual).
#![allow(non_snake_case, non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_void};

#[repr(C)] pub struct BpgCtx { _private: [u8; 0] }
#[repr(C)] pub struct BpgCircuit { _private: [u8; 0] }
#[repr(C)] pub struct BpgTranscript { _private: [u8; 0] }
pub type BpgAllgatherFn = extern "C" fn(user: *mut c_void, bytes_per_rank: usize) -> i32;

pub const BPG_OK: i32 = 0;
pub const BPG_E_CUDA: i32 = -1;
pub const BPG_E_SIZE: i32 = -2;
pub const BPG_E_DECOMPRESS: i32 = -3;
pub const BPG_E_ARG: i32 = -4;
pub const BPG_E_FORMAT: i32 = -5;
pub const BPG_E_NOMEM: i32 = -6;
pub const BPG_E_COMM: i32 = -7;
pub const BPG_FLAG_LEGACY_FRAMING: u32 = 1;
pub const BPG_FLAG_FAST_BLINDING: u32 = 2;
pub const BPG_FLAG_WITNESS_ON_DEVICE: u32 = 4;
pub const BPG_FLAG_NO_LATE_FOLD: u32 = 8;
pub const BPG_FLAG_FORCE_LATE_FOLD: u32 = 16;

#[link(name = "bpg")]
extern "C" {
    pub fn bpg_ctx_create(device: i32, out: *mut *mut BpgCtx) -> i32;
    pub fn bpg_ctx_destroy(ctx: *mut BpgCtx);
    pub fn bpg_last_error(ctx: *mut BpgCtx) -> *const c_char;
    pub fn bpg_strerror(code: i32) -> *const c_char;
    pub fn bpg_launch_count(ctx: *mut BpgCtx) -> u64;
    pub fn bpg_sync(ctx: *mut BpgCtx) -> i32;
    pub fn bpg_set_blocking_sync(on: i32);
    pub fn bpg_set_sizing_mode(mode: i32);
    pub fn bpg_gens_ensure(ctx: *mut BpgCtx, capacity: usize) -> i32;
    pub fn bpg_gens_capacity(ctx: *mut BpgCtx) -> usize;
    pub fn bpg_gens_export(ctx: *mut BpgCtx, i0: usize, n: usize, G32: *mut u8, H32: *mut u8) -> i32;
    pub fn bpg_pedersen_gens(ctx: *mut BpgCtx, B32: *mut u8, Bblinding32: *mut u8) -> i32;
    pub fn bpg_pedersen_commit(ctx: *mut BpgCtx, v: *const u8, r: *const u8, n: usize, out32: *mut u8) -> i32;
    pub fn bpg_msm(ctx: *mut BpgCtx, scalars: *const u8, points32: *const u8, n: usize, out32: *mut u8) -> i32;
    pub fn bpg_msm_gens(ctx: *mut BpgCtx, sG: *const u8, sH: *const u8, n: usize, offset: usize, extra_scalars: *const u8, extra_points32: *const u8, k: usize, out32: *mut u8) -> i32;
    pub fn bpg_msm_gens_dev(ctx: *mut BpgCtx, d_sG: *const c_void, d_sH: *const c_void, n: usize, offset: usize, out32: *mut u8) -> i32;
    pub fn bpg_msm_gens_partial_dev(ctx: *mut BpgCtx, d_sG: *const c_void, d_sH: *const c_void, n: usize, offset: usize, out128: *mut u8) -> i32;
    pub fn bpg_points_sum_compress(ctx: *mut BpgCtx, ext128: *const u8, n: usize, out32: *mut u8) -> i32;
    pub fn bpg_ctx_set_shard(ctx: *mut BpgCtx, rank: i32, world: i32, d_send: *mut c_void, d_recv: *mut c_void, send_cap: usize, allgather: Option<BpgAllgatherFn>, user: *mut c_void) -> i32;
    pub fn bpg_comm_unique_id(out128: *mut u8) -> i32;
    pub fn bpg_comm_init(ctx: *mut BpgCtx, rank: i32, world: i32, id128: *const u8) -> i32;
    pub fn bpg_comm_destroy(ctx: *mut BpgCtx) -> i32;
    pub fn bpg_msm_gens_sharded_dev(ctx: *mut BpgCtx, d_sG: *const c_void, d_sH: *const c_void, n_local: usize, offset: usize, out32: *mut u8) -> i32;
    pub fn bpg_msm_gens_partial_to_dev(ctx: *mut BpgCtx, d_sG: *const c_void, d_sH: *const c_void, n: usize, offset: usize, d_out128: *mut c_void) -> i32;
    pub fn bpg_points_sum_compress_dev(ctx: *mut BpgCtx, d_ext128: *const c_void, n: usize, out32: *mut u8) -> i32;
    pub fn bpg_fold_points(ctx: *mut BpgCtx, sl: *const u8, sr: *const u8, PL32: *const u8, PR32: *const u8, n: usize, out32: *mut u8) -> i32;
    pub fn bpg_mimc_set_constants(ctx: *mut BpgCtx, consts486x32: *const u8) -> i32;
    pub fn bpg_mimc_hash_batch(ctx: *mut BpgCtx, data: *const u8, offsets: *const u64, n: usize, out32: *mut u8) -> i32;
    pub fn bpg_mimc_sponge_batch(ctx: *mut BpgCtx, blocks: *const u8, block_off: *const u32, n: usize, out32: *mut u8, trace: *mut u8) -> i32;
    pub fn bpg_circuit_create(ctx: *mut BpgCtx, n_multipliers: usize, m_commitments: usize, q_constraints: usize, row_ptr: *const u32, term_var: *const u32, term_coeff: *const u8, out: *mut *mut BpgCircuit) -> i32;
    pub fn bpg_circuit_destroy(c: *mut BpgCircuit);
    pub fn bpg_witness_eval(ctx: *mut BpgCtx, n: usize, m: usize, lc_ptr: *const u32, term_var: *const u32, term_coeff: *const u8, v: *const u8, aL: *mut u8, aR: *mut u8, aO: *mut u8) -> i32;
    pub fn bpg_r1cs_prove(ctx: *mut BpgCtx, c: *mut BpgCircuit, label: *const u8, label_len: usize, aL: *const u8, aR: *const u8, aO: *const u8, v: *const u8, v_blinding: *const u8, ext_rng32: *const u8, flags: u32, V_out: *mut u8, proof: *mut u8, proof_cap: usize) -> i64;
    pub fn bpg_r1cs_prove_prefetch(ctx: *mut BpgCtx, c: *mut BpgCircuit, label: *const u8, label_len: usize, v: *const u8, v_blinding: *const u8, ext_rng32: *const u8, flags: u32) -> i32;
    pub fn bpg_r1cs_prove_batch(ctx: *mut BpgCtx, count: usize, circuits: *const *mut BpgCircuit, labels: *const *const u8, label_lens: *const usize, aL: *const *const u8, aR: *const *const u8, aO: *const *const u8, v: *const *const u8, v_blinding: *const *const u8, ext_rng32: *const u8, flags: u32, V_out: *const *mut u8, proofs: *const *mut u8, proof_caps: *const usize, proof_lens: *mut usize) -> i32;
    pub fn bpg_r1cs_verify(ctx: *mut BpgCtx, c: *mut BpgCircuit, label: *const u8, label_len: usize, V32: *const u8, proof: *const u8, proof_len: usize, ext_rng32: *const u8, flags: u32, accept: *mut i32) -> i32;
    pub fn bpg_r1cs_verify_batch(ctx: *mut BpgCtx, count: usize, circuits: *const *mut BpgCircuit, labels: *const *const u8, label_lens: *const usize, V32: *const *const u8, proofs: *const *const u8, proof_lens: *const usize, ext_rng32: *const u8, flags: u32, accept: *mut i32) -> i32;
    pub fn bpg_transcript_new(label: *const u8, len: usize) -> *mut BpgTranscript;
    pub fn bpg_transcript_free(t: *mut BpgTranscript);
    pub fn bpg_transcript_append(t: *mut BpgTranscript, label: *const u8, ll: usize, msg: *const u8, ml: usize);
    pub fn bpg_transcript_challenge(t: *mut BpgTranscript, label: *const u8, ll: usize, out: *mut u8, n: usize);
    pub fn bpg_host_rng_lanes() -> i32;
    pub fn bpg_host_rng_draw64(label: *const u8, label_len: usize, ext32: *const u8, warm: usize, count: usize, use_service: i32, out: *mut u8) -> i32;
    pub fn bpg_dev_alloc(ctx: *mut BpgCtx, bytes: usize, d_ptr: *mut *mut c_void) -> i32;
    pub fn bpg_dev_free(ctx: *mut BpgCtx, d_ptr: *mut c_void) -> i32;
    pub fn bpg_dev_upload(ctx: *mut BpgCtx, d_dst: *mut c_void, h_src: *const c_void, bytes: usize) -> i32;
    pub fn bpg_dev_download(ctx: *mut BpgCtx, h_dst: *mut c_void, d_src: *const c_void, bytes: usize) -> i32;
    pub fn bpg_host_alloc(ctx: *mut BpgCtx, bytes: usize, h_ptr: *mut *mut c_void) -> i32;
    pub fn bpg_host_free(ctx: *mut BpgCtx, h_ptr: *mut c_void) -> i32;
    pub fn bpg_event_record(ctx: *mut BpgCtx, slot: i32) -> i32;
    pub fn bpg_event_elapsed_ms(ctx: *mut BpgCtx, slot_a: i32, slot_b: i32, ms: *mut f32) -> i32;
    pub fn bpg_prof_enable(ctx: *mut BpgCtx, on: i32) -> i32;
    pub fn bpg_prof_read(ctx: *mut BpgCtx, launches: *mut u64, ms_total: *mut f64, pairs_total: *mut u64) -> i32;
    pub fn bpg_prof_read_launches(ctx: *mut BpgCtx, ms: *mut f32, pairs: *mut u32, cap: usize) -> i64;
    pub fn bpg_bench_imad(ctx: *mut BpgCtx, iters: i32, ms: *mut f32, mac32: *mut f64) -> i32;
    pub fn bpg_bench_latency(ctx: *mut BpgCtx, iters: i32, cycles_per_op: *mut f64) -> i32;
}
