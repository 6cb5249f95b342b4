// kernels_batch.cuh -- ragged (many-proof) versions of the prover's and the verifier's vector kernels and a many-output
// small MSM, for bpg_r1cs_prove_batch (prover_batch.inl) and bpg_r1cs_verify_batch (verify_batch.inl).
//
// The K proofs of a batch keep their vectors at ragged offsets off_p = sum_{k<p} N_k of shared buffers.  A kernel either
// walks 128-element blocks of those vectors -- blkp[block] = proof, the element index is (block - blk0_p) * 128 + thread --
// or looks its proof up by binary search over a prefix held in the descriptors, and hands the per-element body of
// kernels_vec.cuh / kernels_msm.cuh (the one its per-proof kernel calls) base pointers offset to that proof, so every scalar
// and every point equals what bpg_r1cs_prove computes.
#pragma once
#include "kernels_msm.cuh"
#include "kernels_vec.cuh"

// small scalars of proof p: small[PB_SLOTS p + k], k as in bpg_r1cs_prove's d_small:
//   [0..2] blindings  [3] y  [4] z  [5] yinv  [6..9] x, x^2, x^3, u  [10] w  [11..12] u_j, u_j^-1  [13..14] cL w, cR w
#define PB_SLOTS 16u
struct pb_desc {
    uint32_t n, N, lgN, m;
    uint32_t off;      // vectors: element 0 of this proof in every N-padded region
    uint32_t blk0;     // first 128-element block of this proof (blocks per proof: ceil(N / 128))
    uint32_t woff;     // w (3n + m + 1 columns) of this proof
    uint32_t poff;     // flatten partial slots of this proof
    uint32_t roff;     // raw transcript-RNG draws of this proof (2n x 64 bytes)
    uint32_t vc0, sp0; // prefix counts of virtual columns / split columns of the earlier proofs
    uint32_t nv, nsplit;
    uint32_t pt, nz, ny; // power tables of this proof: z at pt, y at pt + nz, y^-1 at pt + nz + ny (PB_POW_LO + hi entries each)
    uint32_t st, slot;   // bpg_r1cs_verify_batch only: s table (ny entries) at st of the table array, delta | wV | wc at slot
    const uint32_t *vcol_ptr, *vcol_dst, *row, *split;
    const sc *coeff;
};

// largest p < K with key(D[p]) <= x (the keys are non-decreasing)
template <class Key>
__device__ __forceinline__ uint32_t pb_find(const pb_desc *__restrict__ D, uint32_t K, uint32_t x, Key key) {
    uint32_t lo = 0, hi = K;
    while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (key(D[mid]) <= x) lo = mid; else hi = mid; }
    return lo;
}

// s_L, s_R of every proof from its raw draws
__global__ void __launch_bounds__(128) k_pb_reduce_wide(const pb_desc *__restrict__ D, const uint32_t *__restrict__ blkp, const uint32_t *__restrict__ raw,
                                                        sc *__restrict__ sL, sc *__restrict__ sR) {
    const pb_desc &P = D[blkp[blockIdx.x]];
    uint32_t i = (blockIdx.x - P.blk0) * 128u + threadIdx.x;
    if (i >= P.n) return;
#pragma unroll 1
    for (int side = 0; side < 2; side++) {
        sc r;
        reduce_wide_draw(r, raw + 16ull * (P.roff + side * P.n + i));
        st_sc(side ? &sR[P.off + i] : &sL[P.off + i], r);
    }
}

// Power tables sized per proof: lo[t] = base^t (t < 64) followed by hi[j] = base^(64 j), read as pow_lookup<PB_POW_LG>(r, tab,
// tab + PB_POW_LO, e) -- the same field elements as bpg_r1cs_prove's 1024-entry split, in a few KB per proof (table entries:
// 64 + (max exponent >> 6) + 2)
#define PB_POW_LG 6
#define PB_POW_LO (1u << PB_POW_LG)
__host__ __device__ __forceinline__ uint32_t pb_pow_entries(uint32_t max_exp) { return PB_POW_LO + (max_exp >> PB_POW_LG) + 2u; }
// z, y, y^-1 tables of every proof, one thread per entry of the concatenated tables (total entries: the last proof's pt + 3 tables)
__global__ void __launch_bounds__(128) k_pb_pow_tables(const pb_desc *__restrict__ D, uint32_t K, uint32_t total, const sc *__restrict__ small,
                                                       sc *__restrict__ pt) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    uint32_t p = pb_find(D, K, g, [](const pb_desc &d) { return d.pt; });
    uint32_t e = g - D[p].pt, nz = D[p].nz, ny = D[p].ny, slot;
    if (e < nz) slot = 4u;                          // z
    else if (e < nz + ny) { slot = 3u; e -= nz; }   // y
    else { slot = 5u; e -= nz + ny; }               // y^-1
    sc b, r;
    ld_sc(b, &small[PB_SLOTS * p + slot]);
    sc_pow_u32(r, b, e < PB_POW_LO ? e : (e - PB_POW_LO) << PB_POW_LG);
    st_sc(&pt[g], r);
}

// k_flatten_vcols over the concatenated virtual columns of all circuits
__global__ void __launch_bounds__(128) k_pb_flatten_vcols(const pb_desc *__restrict__ D, uint32_t K, uint32_t nv_total, const sc *__restrict__ pt, sc *__restrict__ w,
                                                          sc *__restrict__ partial) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nv_total) return;
    const pb_desc &P = D[pb_find(D, K, g, [](const pb_desc &d) { return d.vc0; })];
    const uint32_t c = g - P.vc0;
    const sc *zt = pt + P.pt;
    sc acc;
    flatten_vcol<PB_POW_LG>(acc, c, P.vcol_ptr, P.row, P.coeff, zt, zt + PB_POW_LO);
    uint32_t d = P.vcol_dst[c];
    if (d & 0x80000000u) st_sc(&partial[P.poff + (d & 0x7FFFFFFFu)], acc); else st_sc(&w[P.woff + d], acc);
}
// k_flatten_split: one block per split column of any circuit
__global__ void __launch_bounds__(128) k_pb_flatten_split(const pb_desc *__restrict__ D, uint32_t K, const sc *__restrict__ partial, sc *__restrict__ w) {
    __shared__ sc smem[128];
    const pb_desc &P = D[pb_find(D, K, blockIdx.x, [](const pb_desc &d) { return d.sp0; })];
    const uint32_t *sp = P.split + 3 * (blockIdx.x - P.sp0); // (col, first, count)
    sc acc;
    block_sum_rows<1>(&acc, partial + P.poff, sp[1], sp[2], smem);
    if (threadIdx.x == 0) st_sc(&w[P.woff + sp[0]], acc);
}

// k_poly_phase1, one 128-element block of one proof per block; tparts[block][6]
__global__ void __launch_bounds__(128) k_pb_poly_phase1(const pb_desc *__restrict__ D, const uint32_t *__restrict__ blkp, const sc *__restrict__ aL,
                                                        const sc *__restrict__ aR, const sc *__restrict__ aO, const sc *__restrict__ sL, const sc *__restrict__ sR,
                                                        const sc *__restrict__ w, const sc *__restrict__ pt, sc *__restrict__ l1o,
                                                        sc *__restrict__ r0o, sc *__restrict__ r1o, sc *__restrict__ r3o, sc *__restrict__ tparts) {
    __shared__ sc smem[6 * 128];
    const pb_desc &P = D[blkp[blockIdx.x]];
    const uint32_t i = (blockIdx.x - P.blk0) * 128u + threadIdx.x;
    sc t[6];
#pragma unroll
    for (int k = 0; k < 6; k++) sc_zero(t[k]);
    if (i < P.n) {
        const sc *yt = pt + P.pt + P.nz, *yit = yt + P.ny;
        const uint32_t o = P.off;
        poly_phase1_elem<PB_POW_LG>(i, P.n, aL + o, aR + o, aO + o, sL + o, sR + o, w + P.woff, yt, yt + PB_POW_LO, yit, yit + PB_POW_LO, l1o + o,
                                    r0o + o, r1o + o, r3o + o, t);
    }
    block_sum_scalars<6>(t, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < 6; k++) st_sc(&tparts[(size_t)blockIdx.x * 6 + k], t[k]);
    }
}
// one block per proof: t_1..t_6 (sum of the proof's block partials) and wV[0..m) -> out[ooff_p ..] (6 + m scalars per proof)
__global__ void __launch_bounds__(128) k_pb_phase1_out(const pb_desc *__restrict__ D, const sc *__restrict__ tparts, const sc *__restrict__ w,
                                                       const uint32_t *__restrict__ ooff, sc *__restrict__ out) {
    __shared__ sc smem[6 * 128];
    const pb_desc &P = D[blockIdx.x];
    sc acc[6];
    block_sum_rows<6>(acc, tparts, P.blk0, (P.N + 127u) / 128u, smem);
    sc *o = out + ooff[blockIdx.x];
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < 6; k++) st_sc(&o[k], acc[k]);
    }
    for (uint32_t k = threadIdx.x; k < P.m; k += 128) { sc x; ld_sc(x, &w[P.woff + 3 * P.n + k]); st_sc(&o[6 + k], x); }
}

// k_poly_phase2 over every proof's N elements (xs = small[PB_SLOTS p + 6 ..])
__global__ void __launch_bounds__(128) k_pb_poly_phase2(const pb_desc *__restrict__ D, const uint32_t *__restrict__ blkp, const sc *__restrict__ small,
                                                        const sc *__restrict__ l1, const sc *__restrict__ aO, const sc *__restrict__ sL, const sc *__restrict__ r0,
                                                        const sc *__restrict__ r1, const sc *__restrict__ r3, const sc *__restrict__ pt,
                                                        sc *__restrict__ a, sc *__restrict__ b, sc *__restrict__ EG, sc *__restrict__ EH) {
    const uint32_t p = blkp[blockIdx.x];
    const pb_desc &P = D[p];
    const uint32_t i = (blockIdx.x - P.blk0) * 128u + threadIdx.x;
    if (i >= P.N) return;
    const sc *yt = pt + P.pt + P.nz, *yit = yt + P.ny;
    const uint32_t o = P.off;
    poly_phase2_elem<PB_POW_LG>(i, P.n, small + PB_SLOTS * p + 6, l1 + o, aO + o, sL + o, r0 + o, r1 + o, r3 + o, yt, yt + PB_POW_LO, yit,
                                yit + PB_POW_LO, a + o, b + o, EG + o, EH + o);
}

// ---- inner-product round j: proof p takes part while j < lgN_p (h = N_p >> (j + 1), nj = 2 h)
// k_ipp_cross per block: cparts[block] = (<a_lo, b_hi>, <a_hi, b_lo>) over the block's share of [0, h)
__global__ void __launch_bounds__(128) k_pb_ipp_cross(const pb_desc *__restrict__ D, const uint32_t *__restrict__ blkp, uint32_t j, const sc *__restrict__ a,
                                                      const sc *__restrict__ b, sc *__restrict__ cparts) {
    __shared__ sc smem[2 * 128];
    const pb_desc &P = D[blkp[blockIdx.x]];
    if (j >= P.lgN) return; // whole block: k_pb_ipp_cw reads no partial of an inactive proof
    const uint32_t i = (blockIdx.x - P.blk0) * 128u + threadIdx.x, h = P.N >> (j + 1);
    sc t[2];
    sc_zero(t[0]); sc_zero(t[1]);
    if (i < h) ipp_cross_elem(i, h, a + P.off, b + P.off, t);
    block_sum_scalars<2>(t, smem);
    if (threadIdx.x == 0) { st_sc(&cparts[2 * (size_t)blockIdx.x], t[0]); st_sc(&cparts[2 * (size_t)blockIdx.x + 1], t[1]); }
}
// k_sum_partials<2> + k_ipp_cw, one block per proof: small[13] = cL w, small[14] = cR w
__global__ void __launch_bounds__(128) k_pb_ipp_cw(const pb_desc *__restrict__ D, uint32_t j, const sc *__restrict__ cparts, sc *__restrict__ small) {
    __shared__ sc smem[2 * 128];
    const pb_desc &P = D[blockIdx.x];
    if (j >= P.lgN) return;
    sc acc[2];
    block_sum_rows<2>(acc, cparts, P.blk0, ((P.N >> (j + 1)) + 127u) / 128u, smem);
    if (threadIdx.x == 0) {
        sc *sm = small + PB_SLOTS * blockIdx.x;
        sc w, r;
        ld_sc(w, &sm[10]);
        sc_mul(r, acc[0], w); st_sc(&sm[13], r);
        sc_mul(r, acc[1], w); st_sc(&sm[14], r);
    }
}
// k_ipp_expand over the N original generators of every active proof
__global__ void __launch_bounds__(128) k_pb_ipp_expand(const pb_desc *__restrict__ D, const uint32_t *__restrict__ blkp, uint32_t j, const sc *__restrict__ a,
                                                       const sc *__restrict__ b, const sc *__restrict__ EG, const sc *__restrict__ EH, sc *__restrict__ sG,
                                                       sc *__restrict__ sH) {
    const pb_desc &P = D[blkp[blockIdx.x]];
    const uint32_t i = (blockIdx.x - P.blk0) * 128u + threadIdx.x;
    if (j >= P.lgN || i >= P.N) return;
    const uint32_t o = P.off;
    ipp_expand_elem(i, P.N >> j, a + o, b + o, EG + o, EH + o, sG + o, sH + o);
}
// k_ipp_fold of every active proof; uu[2 p], uu[2 p + 1] = u_j, u_j^-1 of proof p
__global__ void __launch_bounds__(128) k_pb_ipp_fold(const pb_desc *__restrict__ D, const uint32_t *__restrict__ blkp, uint32_t j, const sc *__restrict__ uu,
                                                     sc *__restrict__ a, sc *__restrict__ b, sc *__restrict__ EG, sc *__restrict__ EH) {
    const uint32_t p = blkp[blockIdx.x];
    const pb_desc &P = D[p];
    const uint32_t i = (blockIdx.x - P.blk0) * 128u + threadIdx.x;
    if (j >= P.lgN || i >= P.N) return;
    const uint32_t nj = P.N >> j, h = nj >> 1, o = P.off;
    sc u, ui;
    ld_sc(u, &uu[2 * p]); ld_sc(ui, &uu[2 * p + 1]);
    ipp_fold_factors(i, nj, h, u, ui, EG + o, EH + o);
    if (i < h) ipp_fold_ab(i, h, u, ui, a + o, b + o);
}
// final (a, b) of every proof -> out[2 p], out[2 p + 1]
__global__ void __launch_bounds__(128) k_pb_final_ab(const pb_desc *__restrict__ D, uint32_t K, const sc *__restrict__ a, const sc *__restrict__ b,
                                                     sc *__restrict__ out) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= K) return;
    sc x;
    ld_sc(x, &a[D[p].off]); st_sc(&out[2 * p], x);
    ld_sc(x, &b[D[p].off]); st_sc(&out[2 * p + 1], x);
}

// ---- bpg_r1cs_verify_batch (verify_batch.inl): the verifier's scalar preparation of the K proofs of a pass.  The descriptors
// are pb_desc with off = g | h of the proof (g at off, h at off + N, relative to the pass's gh base) and the small scalars use
// the prover's stride with the verifier's meaning:
//   small[PB_SLOTS p + k]:  [0] x  [1] a  [2] b  [3] y  [4] z  [5] y^-1  [6] u  [7] allinv      usq[VB_LGMAX p + j] = u_j^2
// (k_pb_pow_tables also builds the y table there, which the verifier does not read.)
#define VB_LGMAX 12u // lg N of BPG_BATCH_MAX_N
// s tables of every proof, one thread per entry; the proofs' tables are at D[p].st (non-decreasing), st0 .. st0 + total
__global__ void __launch_bounds__(128) k_pb_s_tables(const pb_desc *__restrict__ D, uint32_t K, uint32_t st0, uint32_t total, const sc *__restrict__ small,
                                                     const sc *__restrict__ usq, sc *__restrict__ pt) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    g += st0;
    const uint32_t p = pb_find(D, K, g, [](const pb_desc &d) { return d.st; });
    sc acc;
    s_table_entry<PB_POW_LG>(acc, g - D[p].st, usq + VB_LGMAX * p, &small[PB_SLOTS * p + 7], D[p].lgN);
    st_sc(&pt[g], acc);
}
// k_verify_scalars, one 128-element block of one proof per block: g | h of the proof, dparts[block] = the block's share of delta
__global__ void __launch_bounds__(128) k_pb_verify_scalars(const pb_desc *__restrict__ D, const uint32_t *__restrict__ blkp, const sc *__restrict__ small,
                                                           const sc *__restrict__ w, const sc *__restrict__ pt, sc *__restrict__ gh, sc *__restrict__ dparts) {
    __shared__ sc smem[128];
    const uint32_t p = blkp[blockIdx.x];
    const pb_desc &P = D[p];
    const uint32_t i = (blockIdx.x - P.blk0) * 128u + threadIdx.x;
    sc d;
    sc_zero(d);
    if (i < P.N) {
        const sc *sm = small + PB_SLOTS * p, *yit = pt + P.pt + P.nz + P.ny, *stab = pt + P.st;
        sc x, ia, ib, u;
        ld_sc(x, &sm[0]); ld_sc(ia, &sm[1]); ld_sc(ib, &sm[2]); ld_sc(u, &sm[6]);
        sc *g = gh + P.off;
        verify_scalars_elem<PB_POW_LG>(i, P.n, P.N, x, ia, ib, u, w + P.woff, yit, yit + PB_POW_LO, stab, stab + PB_POW_LO, g, g + P.N, d);
    }
    block_sum_scalars<1>(&d, smem);
    if (threadIdx.x == 0) st_sc(&dparts[blockIdx.x], d);
}
// one block per proof: delta (sum of the proof's block partials), wV[0..m), wc -> slots[slot_p ..] (m + 2 scalars per proof)
__global__ void __launch_bounds__(128) k_pb_verify_out(const pb_desc *__restrict__ D, const sc *__restrict__ dparts, const sc *__restrict__ w,
                                                       sc *__restrict__ slots) {
    __shared__ sc smem[128];
    const pb_desc &P = D[blockIdx.x];
    sc acc;
    block_sum_rows<1>(&acc, dparts, P.blk0, (P.N + 127u) / 128u, smem);
    sc *o = slots + P.slot;
    if (threadIdx.x == 0) st_sc(&o[0], acc);
    for (uint32_t k = threadIdx.x; k <= P.m; k += 128) { sc x; ld_sc(x, &w[P.woff + 3 * P.n + k]); st_sc(&o[1 + k], x); }
}
// Combined check of a set of proofs (verify_finish): acc[i] = sum_t rho_t g_t[i], acc[Nmax + i] = sum_t rho_t h_t[i] over the
// terms with i < N_t (h_t = g_t + N_t).  The terms are sorted by N_t, largest first.  One thread per output scalar.
struct vb_term {
    sc rho;
    const sc *g;
    uint32_t N, pad;
};
__global__ void __launch_bounds__(128) k_pb_axpy_gh(const vb_term *__restrict__ T, uint32_t nt, uint32_t Nmax, sc *__restrict__ acc) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * Nmax) return;
    const uint32_t side = t >= Nmax ? 1u : 0u, i = t - side * Nmax;
    sc a;
    sc_zero(a);
#pragma unroll 1
    for (uint32_t k = 0; k < nt; k++) {
        const uint32_t N = T[k].N;
        if (i >= N) break;
        sc x, r, p;
        ld_sc(x, &T[k].g[side * N + i]); ld_sc(r, &T[k].rho);
        sc_mul(p, r, x);
        sc_add_r(a, a, p);
    }
    st_sc(&acc[t], a);
}

// ---- per-proof check of a pass (verify_check_pass, verify_batch.inl): every proof against its own verification equation.
// The own-point terms of the pass are concatenated, proof p owning terms [toff[p], toff[p+1]) (at least 11 each), t2p[t] =
// proof of term t.  Variable-base part, one thread per term: decode (a failure clears ok[p] of that proof only), windowed
// scalar multiplication, then one block sum per proof the block touches -> part[block + p].  Consecutive blocks share at most
// one proof, so block + p is unique per (block, proof) pair and part holds blocks + K points.
__global__ void __launch_bounds__(64) k_pb_varbase(const sc *__restrict__ es, const uint8_t *__restrict__ ep, const uint32_t *__restrict__ t2p, uint32_t k,
                                                   uint32_t *__restrict__ ok, ge *__restrict__ part) {
    __shared__ ge smem[64];
    const uint32_t t0 = blockIdx.x * 64u, t = t0 + threadIdx.x;
    const uint32_t q0 = t2p[t0], q1 = t2p[min(t0 + 63u, k - 1u)];
    uint32_t q = 0xFFFFFFFFu;
    ge acc;
    ge_identity(acc);
    if (t < k) {
        q = t2p[t];
        uint8_t b[32];
        for (int i = 0; i < 32; i++) b[i] = ep[32ull * t + i];
        ge p;
        if (ristretto_decode(p, b)) {
            sc s;
            ld_sc(s, &es[t]);
            sc_reduce(s, s);
            ge_scalarmul_w4(acc, s, p);
        } else atomicAnd(&ok[q], 0u);
    }
#pragma unroll 1
    for (uint32_t r = q0; r <= q1; r++) {
        ge x;
        if (q == r) x = acc; else ge_identity(x);
        block_sum_points(x, smem);
        if (threadIdx.x == 0) st_ge(&part[blockIdx.x + r], x);
    }
}
// one block per proof: its variable-base partials + its fixed-base output, verdict[p] = decoded && identity (all-zero encoding),
// the test verify_finish applies to one proof
__global__ void __launch_bounds__(64) k_pb_check_out(const uint32_t *__restrict__ toff, const ge *__restrict__ fixed, const ge *__restrict__ part,
                                                     const uint32_t *__restrict__ ok, int *__restrict__ verdict) {
    __shared__ ge smem[64];
    const uint32_t p = blockIdx.x, b0 = toff[p] / 64u, b1 = (toff[p + 1] - 1u) / 64u;
    ge acc;
    ge_identity(acc);
#pragma unroll 1
    for (uint32_t b = b0 + threadIdx.x; b <= b1; b += 64u) {
        ge x;
        ld_ge(x, &part[b + p]);
        ge_add(acc, acc, x);
    }
    block_sum_points(acc, smem);
    if (threadIdx.x == 0) {
        ge f;
        ld_ge(f, &fixed[p]);
        ge_add(acc, acc, f);
        uint8_t e[32], nz = 0;
        ristretto_encode(e, acc);
        for (int i = 0; i < 32; i++) nz |= e[i];
        verdict[p] = (ok[p] && nz == 0) ? 1 : 0;
    }
}

// ---- many-output small MSM (msm_run_many): k_msm_digits<*, SPLIT = 1> with the segments in a device table (any number of
// them, ascending `start`) and one bucket group per output, so the group count is not bounded by msm_params
template <int SCATTER>
__global__ void __launch_bounds__(256) k_many_digits(const msm_seg *__restrict__ segs, uint32_t nseg, uint32_t total, uint32_t ptotal,
                                                     uint32_t *__restrict__ counts_or_cursor, uint32_t *__restrict__ sorted) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = t < total; // no early return: the warp-aggregated counter update needs all 32 lanes
    int d[16];
#pragma unroll
    for (int w = 0; w < 16; w++) d[w] = 0;
    uint32_t grp = 0, pidx = 0;
    if (valid) {
        uint32_t lo = 0, hi = nseg; // segment of term t: the last one with start <= t
        while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (segs[mid].start <= t) lo = mid; else hi = mid; }
        const msm_seg S = segs[lo];
        uint32_t j = t - S.start;
        msm_seg_digits(S, j, d, pidx);
        grp = S.group;
        if (S.alt) grp ^= ((j + S.j0) >> (S.alt - 1)) & 1u;
    }
    const uint32_t base = grp * 2u * BPG_MAT_NB;
#pragma unroll
    for (int w = 0; w < 16; w++) emit_split_digit<SCATTER>(counts_or_cursor, sorted, base, d[w], (uint32_t)w * ptotal + pidx);
}
