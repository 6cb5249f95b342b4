// kernels_vec.cuh -- scalar-field (mod l) kernels: batched MiMC (K8) and the O(n) vector phases of the R1CS
// prover / verifier and of the inner-product argument (K9).
#pragma once
#include "kernels_core.cuh"

// ---------------------------------------------------------------- MiMC (src/mimc_hash/mimc.rs:7-40)
#define MIMC_ROUNDS 486
__constant__ sc c_mimc[MIMC_ROUNDS];

// One thread per independent sponge.  state += block; 486 x state = (state + c_i)^3  (zero key).
// trace (nullable): per absorbed block 972 multipliers x (a_L, a_R, a_O): (t,t,t^2) then (t^2,t,t^3)
// (mimc_hash_gadget.rs:133-144), block-major in absorption order of the whole batch.
__global__ void __launch_bounds__(128) k_mimc_sponge(const sc *__restrict__ blocks, const uint32_t *__restrict__ block_off, uint32_t n,
                                                      sc *__restrict__ out, sc *__restrict__ trace) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sc st;
    sc_set_u32(st, 0);
    uint32_t b0 = block_off[i], b1 = block_off[i + 1];
#pragma unroll 1
    for (uint32_t b = b0; b < b1; b++) {
        sc x;
        ld_sc(x, &blocks[b]);
        x.v[7] &= 0x7FFFFFFFu; // Scalar::from_bits
        sc_reduce(x, x);
        sc_add_r(st, st, x);
        sc *tr = trace ? trace + (size_t)b * (MIMC_ROUNDS * 6) : nullptr;
#pragma unroll 1
        for (int r = 0; r < MIMC_ROUNDS; r++) {
            sc t, t2, t3;
            sc_add_r(t, st, c_mimc[r]);
            sc_mul(t2, t, t);
            sc_mul(t3, t2, t);
            if (tr) {
                sc *o = tr + 6 * r;
                st_sc(o, t); st_sc(o + 1, t); st_sc(o + 2, t2);
                st_sc(o + 3, t2); st_sc(o + 4, t); st_sc(o + 5, t3);
            }
            st = t3;
        }
    }
    st_sc(&out[i], st);
}

// ---------------------------------------------------------------- helpers
__device__ __forceinline__ void sc_zero(sc &r) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = 0;
}
// base^e from the two-level tables lo[e & (2^LO - 1)] * hi[e >> LO]  (lo[t] = base^t, hi[j] = base^(2^LO j)).
// bpg_r1cs_prove uses LO = 10; the batch prover LO = 6 (tables sized per proof, kernels_batch.cuh).
template <int LO>
__device__ __forceinline__ void pow_lookup(sc &r, const sc *__restrict__ lo, const sc *__restrict__ hi, uint32_t e) {
    sc a, b;
    ld_sc(a, &lo[e & ((1u << LO) - 1u)]);
    if (e >> LO) { ld_sc(b, &hi[e >> LO]); sc_mul(r, a, b); } else r = a;
}
// block-wide sum of NS scalars per thread (blockDim.x == 128); result valid in thread 0
template <int NS>
__device__ __forceinline__ void block_sum_scalars(sc *vals, sc *smem /* [NS][128] */) {
    int t = threadIdx.x;
#pragma unroll
    for (int k = 0; k < NS; k++) st_sc(&smem[k * 128 + t], vals[k]);
    __syncthreads();
    for (int s = 64; s > 0; s >>= 1) {
        if (t < s) {
#pragma unroll
            for (int k = 0; k < NS; k++) {
                sc a, b;
                ld_sc(a, &smem[k * 128 + t]); ld_sc(b, &smem[k * 128 + t + s]);
                sc_add_r(a, a, b);
                st_sc(&smem[k * 128 + t], a);
            }
        }
        __syncthreads();
    }
    if (t == 0) {
#pragma unroll
        for (int k = 0; k < NS; k++) ld_sc(vals[k], &smem[k * 128]);
    }
}

// zero NS accumulators, add the rows first + threadIdx.x, first + threadIdx.x + 128, ... < first + cnt of rows (row-major
// [][NS]) into them and sum them over the block (blockDim.x == 128); result valid in thread 0
template <int NS>
__device__ __forceinline__ void block_sum_rows(sc *acc, const sc *__restrict__ rows, uint32_t first, uint32_t cnt, sc *smem /* [NS][128] */) {
#pragma unroll
    for (int k = 0; k < NS; k++) sc_zero(acc[k]);
    for (uint32_t p = threadIdx.x; p < cnt; p += 128) {
#pragma unroll
        for (int k = 0; k < NS; k++) { sc x; ld_sc(x, &rows[(size_t)(first + p) * NS + k]); sc_add_r(acc[k], acc[k], x); }
    }
    block_sum_scalars<NS>(acc, smem);
}

__global__ void __launch_bounds__(256) k_sc_reduce_inplace(sc *v, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sc x; ld_sc(x, &v[i]); sc_reduce(x, x); st_sc(&v[i], x);
}
// Scalar::from_bytes_mod_order_wide of one raw 64-byte TranscriptRng draw
__device__ __forceinline__ void reduce_wide_draw(sc &r, const uint32_t *__restrict__ raw) {
    const uint4 *src = (const uint4 *)raw;
    u32 R[16];
#pragma unroll
    for (int k = 0; k < 4; k++) { uint4 q = src[k]; R[4 * k] = q.x; R[4 * k + 1] = q.y; R[4 * k + 2] = q.z; R[4 * k + 3] = q.w; }
    sc_reduce512(r, R);
}
// element i < n of the raw draws goes to outL[i], n <= i < 2n to outR[i - n]
__global__ void __launch_bounds__(128) k_sc_reduce_wide(const uint32_t *__restrict__ raw, uint32_t n, sc *__restrict__ outL, sc *__restrict__ outR) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * n) return;
    sc r;
    reduce_wide_draw(r, raw + 16ull * i);
    st_sc(i < n ? &outL[i] : &outR[i - n], r);
}
// lo[t] = base^t (t < 1024), hi[j] = base^(1024 j) (j < nhi)
__global__ void __launch_bounds__(128) k_pow_tables(const sc *__restrict__ base, sc *__restrict__ lo, sc *__restrict__ hi, uint32_t nhi) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 1024 + nhi) return;
    sc b; ld_sc(b, base);
    sc r;
    if (t < 1024) { sc_pow_u32(r, b, t); st_sc(&lo[t], r); }
    else { sc_pow_u32(r, b, (t - 1024u) << 10); st_sc(&hi[t - 1024], r); }
}
// sums `nparts` rows of NS scalars (row-major [nparts][NS]) into out[NS]; one block
template <int NS>
__global__ void __launch_bounds__(128) k_sum_partials(const sc *__restrict__ parts, uint32_t nparts, sc *__restrict__ out) {
    __shared__ sc smem[NS * 128];
    sc acc[NS];
    block_sum_rows<NS>(acc, parts, 0, nparts, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < NS; k++) st_sc(&out[k], acc[k]);
    }
}

// ---------------------------------------------------------------- flattened constraints (a4 / a8)
// Entries are sorted by (virtual) column.  A virtual column is a run of <= 32 entries of one variable; it either
// writes w[dst] directly or, for variables split over several virtual columns, a partial slot (dst | 1<<31).
// value = sum_k z^(row_k+1) * coeff_k   (coefficients of V / One columns are stored negated).
template <int LO>
__device__ __forceinline__ void flatten_vcol(sc &acc, uint32_t c, const uint32_t *__restrict__ vcol_ptr, const uint32_t *__restrict__ e_row,
                                             const sc *__restrict__ e_coeff, const sc *__restrict__ zlo, const sc *__restrict__ zhi) {
    sc_zero(acc);
    uint32_t k0 = vcol_ptr[c], k1 = vcol_ptr[c + 1];
#pragma unroll 1
    for (uint32_t k = k0; k < k1; k++) {
        sc zp, cf, p;
        pow_lookup<LO>(zp, zlo, zhi, e_row[k] + 1u);
        ld_sc(cf, &e_coeff[k]);
        sc_mul(p, zp, cf);
        sc_add_r(acc, acc, p);
    }
}
__global__ void __launch_bounds__(128) k_flatten_vcols(const uint32_t *__restrict__ vcol_ptr, const uint32_t *__restrict__ vcol_dst, uint32_t nv,
                                                        const uint32_t *__restrict__ e_row, const sc *__restrict__ e_coeff,
                                                        const sc *__restrict__ zlo, const sc *__restrict__ zhi, sc *__restrict__ w, sc *__restrict__ partial) {
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nv) return;
    sc acc;
    flatten_vcol<10>(acc, c, vcol_ptr, e_row, e_coeff, zlo, zhi);
    uint32_t d = vcol_dst[c];
    if (d & 0x80000000u) st_sc(&partial[d & 0x7FFFFFFFu], acc); else st_sc(&w[d], acc);
}
// one block per split variable: w[col] = sum of its partial slots
__global__ void __launch_bounds__(128) k_flatten_split(const uint32_t *__restrict__ split /* (col, first, count) x ns */, uint32_t ns,
                                                        const sc *__restrict__ partial, sc *__restrict__ w) {
    __shared__ sc smem[128];
    uint32_t s = blockIdx.x;
    if (s >= ns) return;
    uint32_t col = split[3 * s], first = split[3 * s + 1], cnt = split[3 * s + 2];
    sc acc;
    block_sum_rows<1>(&acc, partial, first, cnt, smem);
    if (threadIdx.x == 0) st_sc(&w[col], acc);
}

// ---------------------------------------------------------------- prover polynomial phase (SURVEY App. A.5)
// l1 = aL + y^-i wR ; l2 = aO ; l3 = sL ; r0 = wO - y^i ; r1 = y^i aR + wL ; r3 = y^i sR
// t1=<l1,r0> t2=<l1,r1>+<l2,r0> t3=<l2,r1>+<l3,r0> t4=<l1,r3>+<l3,r1> t5=<l2,r3> t6=<l3,r3>
// stores l1,r0,r1,r3 and per-block partial sums of t1..t6.
template <int LO>
__device__ __forceinline__ void poly_phase1_elem(uint32_t i, uint32_t n, const sc *__restrict__ aL, const sc *__restrict__ aR, const sc *__restrict__ aO,
                                                 const sc *__restrict__ sL, const sc *__restrict__ sR, const sc *__restrict__ w /* wL|wR|wO */,
                                                 const sc *__restrict__ ylo, const sc *__restrict__ yhi, const sc *__restrict__ yilo,
                                                 const sc *__restrict__ yihi, sc *__restrict__ l1o, sc *__restrict__ r0o, sc *__restrict__ r1o,
                                                 sc *__restrict__ r3o, sc *t /* [6] */) {
    sc yi, yinv, a_l, a_r, a_o, s_l, s_r, wl, wr, wo, l1, r0, r1, r3, p;
    pow_lookup<LO>(yi, ylo, yhi, i);
    pow_lookup<LO>(yinv, yilo, yihi, i);
    ld_sc(a_l, &aL[i]); ld_sc(a_r, &aR[i]); ld_sc(a_o, &aO[i]); ld_sc(s_l, &sL[i]); ld_sc(s_r, &sR[i]);
    ld_sc(wl, &w[i]); ld_sc(wr, &w[n + i]); ld_sc(wo, &w[2 * (size_t)n + i]);
    sc_mul(p, yinv, wr); sc_add_r(l1, a_l, p);
    sc_sub_r(r0, wo, yi);
    sc_mul(p, yi, a_r); sc_add_r(r1, p, wl);
    sc_mul(r3, yi, s_r);
    st_sc(&l1o[i], l1); st_sc(&r0o[i], r0); st_sc(&r1o[i], r1); st_sc(&r3o[i], r3);
    sc_mul(p, l1, r0); sc_add_r(t[0], t[0], p);
    sc_mul(p, l1, r1); sc_add_r(t[1], t[1], p); sc_mul(p, a_o, r0); sc_add_r(t[1], t[1], p);
    sc_mul(p, a_o, r1); sc_add_r(t[2], t[2], p); sc_mul(p, s_l, r0); sc_add_r(t[2], t[2], p);
    sc_mul(p, l1, r3); sc_add_r(t[3], t[3], p); sc_mul(p, s_l, r1); sc_add_r(t[3], t[3], p);
    sc_mul(p, a_o, r3); sc_add_r(t[4], t[4], p);
    sc_mul(p, s_l, r3); sc_add_r(t[5], t[5], p);
}
__global__ void __launch_bounds__(128) k_poly_phase1(uint32_t n, const sc *__restrict__ aL, const sc *__restrict__ aR, const sc *__restrict__ aO,
                                                      const sc *__restrict__ sL, const sc *__restrict__ sR, const sc *__restrict__ w /* wL|wR|wO */,
                                                      const sc *__restrict__ ylo, const sc *__restrict__ yhi, const sc *__restrict__ yilo,
                                                      const sc *__restrict__ yihi, sc *__restrict__ l1o, sc *__restrict__ r0o, sc *__restrict__ r1o,
                                                      sc *__restrict__ r3o, sc *__restrict__ tparts /* [grid][6] */) {
    __shared__ sc smem[6 * 128];
    sc t[6];
#pragma unroll
    for (int k = 0; k < 6; k++) sc_zero(t[k]);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        poly_phase1_elem<10>(i, n, aL, aR, aO, sL, sR, w, ylo, yhi, yilo, yihi, l1o, r0o, r1o, r3o, t);
    block_sum_scalars<6>(t, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < 6; k++) st_sc(&tparts[(size_t)blockIdx.x * 6 + k], t[k]);
    }
}
// l = x l1 + x^2 l2 + x^3 l3 ; r = r0 + x r1 + x^3 r3 ; padding: l = 0, r = -y^i.
// Also initialises the per-generator IPP factors EG = G_factors, EH = H_factors (1 or u, times y^-i for H).
// xs = [x, x^2, x^3, u]
template <int LO>
__device__ __forceinline__ void poly_phase2_elem(uint32_t i, uint32_t n, const sc *__restrict__ xs, const sc *__restrict__ l1, const sc *__restrict__ aO,
                                                 const sc *__restrict__ sL, const sc *__restrict__ r0, const sc *__restrict__ r1, const sc *__restrict__ r3,
                                                 const sc *__restrict__ ylo, const sc *__restrict__ yhi, const sc *__restrict__ yilo,
                                                 const sc *__restrict__ yihi, sc *__restrict__ a, sc *__restrict__ b, sc *__restrict__ EG, sc *__restrict__ EH) {
    sc x, x2, x3, u, yinv;
    ld_sc(x, &xs[0]); ld_sc(x2, &xs[1]); ld_sc(x3, &xs[2]); ld_sc(u, &xs[3]);
    pow_lookup<LO>(yinv, yilo, yihi, i);
    sc one; sc_set_u32(one, 1);
    if (i < n) {
        sc v, p, acc;
        ld_sc(v, &l1[i]); sc_mul(acc, x, v);
        ld_sc(v, &aO[i]); sc_mul(p, x2, v); sc_add_r(acc, acc, p);
        ld_sc(v, &sL[i]); sc_mul(p, x3, v); sc_add_r(acc, acc, p);
        st_sc(&a[i], acc);
        ld_sc(acc, &r0[i]);
        ld_sc(v, &r1[i]); sc_mul(p, x, v); sc_add_r(acc, acc, p);
        ld_sc(v, &r3[i]); sc_mul(p, x3, v); sc_add_r(acc, acc, p);
        st_sc(&b[i], acc);
        st_sc(&EG[i], one);
        st_sc(&EH[i], yinv);
    } else {
        sc z, yi, ny, eh;
        sc_zero(z);
        pow_lookup<LO>(yi, ylo, yhi, i);
        sc_neg_r(ny, yi);
        st_sc(&a[i], z);
        st_sc(&b[i], ny);
        st_sc(&EG[i], u);
        sc_mul(eh, yinv, u);
        st_sc(&EH[i], eh);
    }
}
__global__ void __launch_bounds__(128) k_poly_phase2(uint32_t n, uint32_t N, const sc *__restrict__ xs, const sc *__restrict__ l1, const sc *__restrict__ aO,
                                                      const sc *__restrict__ sL, const sc *__restrict__ r0, const sc *__restrict__ r1, const sc *__restrict__ r3,
                                                      const sc *__restrict__ ylo, const sc *__restrict__ yhi, const sc *__restrict__ yilo,
                                                      const sc *__restrict__ yihi, sc *__restrict__ a, sc *__restrict__ b, sc *__restrict__ EG, sc *__restrict__ EH) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    poly_phase2_elem<10>(i, n, xs, l1, aO, sL, r0, r1, r3, ylo, yhi, yilo, yihi, a, b, EG, EH);
}

// ---------------------------------------------------------------- inner-product argument rounds (a6 / a7)
// current vectors a,b have length nj = 2h.  cparts[block] = (<a_lo,b_hi>, <a_hi,b_lo>)
__device__ __forceinline__ void ipp_cross_elem(uint32_t i, uint32_t h, const sc *__restrict__ a, const sc *__restrict__ b, sc *t /* [2] */) {
    sc al, ah, bl, bh, p;
    ld_sc(al, &a[i]); ld_sc(ah, &a[h + i]); ld_sc(bl, &b[i]); ld_sc(bh, &b[h + i]);
    sc_mul(p, al, bh); sc_add_r(t[0], t[0], p);
    sc_mul(p, ah, bl); sc_add_r(t[1], t[1], p);
}
__global__ void __launch_bounds__(128) k_ipp_cross(uint32_t h, const sc *__restrict__ a, const sc *__restrict__ b, sc *__restrict__ cparts) {
    __shared__ sc smem[2 * 128];
    sc t[2];
    sc_zero(t[0]); sc_zero(t[1]);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < h; i += gridDim.x * blockDim.x) ipp_cross_elem(i, h, a, b, t);
    block_sum_scalars<2>(t, smem);
    if (threadIdx.x == 0) { st_sc(&cparts[2 * (size_t)blockIdx.x], t[0]); st_sc(&cparts[2 * (size_t)blockIdx.x + 1], t[1]); }
}
// out[0] = cL * w, out[1] = cR * w   (scalars of the Q = w*B terms of L and R)
__global__ void k_ipp_cw(const sc *__restrict__ c2, const sc *__restrict__ w, sc *__restrict__ out) {
    if (threadIdx.x >= 2 || blockIdx.x) return;
    sc c, ww, r;
    ld_sc(c, &c2[threadIdx.x]); ld_sc(ww, w);
    sc_mul(r, c, ww);
    st_sc(&out[threadIdx.x], r);
}
// Scalars of the round's two MSMs over the ORIGINAL generators (no folded generators are materialised):
// with r = i mod nj:  r >= h:  G_i -> L with a[r-h]*EG[i],  H_i -> R with b[r-h]*EH[i]
//                     r <  h:  G_i -> R with a[h+r]*EG[i],  H_i -> L with b[h+r]*EH[i]
// [i0, i1): the part of [0, N) this call has to produce (a rank of a sharded proof only needs the scalars of its own point range)
__device__ __forceinline__ void ipp_expand_elem(uint32_t i, uint32_t nj, const sc *__restrict__ a, const sc *__restrict__ b, const sc *__restrict__ EG,
                                                const sc *__restrict__ EH, sc *__restrict__ sG, sc *__restrict__ sH) {
    uint32_t h = nj >> 1, r = i & (nj - 1);
    uint32_t src = r >= h ? r - h : r + h;
    sc av, bv, eg, eh, p;
    ld_sc(av, &a[src]); ld_sc(bv, &b[src]); ld_sc(eg, &EG[i]); ld_sc(eh, &EH[i]);
    sc_mul(p, av, eg); st_sc(&sG[i], p);
    sc_mul(p, bv, eh); st_sc(&sH[i], p);
}
__global__ void __launch_bounds__(128) k_ipp_expand(uint32_t N, uint32_t nj, const sc *__restrict__ a, const sc *__restrict__ b, const sc *__restrict__ EG,
                                                     const sc *__restrict__ EH, sc *__restrict__ sG, sc *__restrict__ sH, uint32_t i0, uint32_t i1) {
    uint32_t i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= i1 || i >= N) return;
    ipp_expand_elem(i, nj, a, b, EG, EH, sG, sH);
}
// a' = a_lo u + a_hi u^-1 ; b' = b_lo u^-1 + b_hi u ; EG[i] *= (right half ? u : u^-1) ; EH[i] *= (right half ? u^-1 : u)
// uu = [u, u^-1].  The per-generator factors are only updated on [i0, i1) (see k_ipp_expand); a, b always in full.
__device__ __forceinline__ void ipp_fold_factors(uint32_t i, uint32_t nj, uint32_t h, const sc &u, const sc &ui, sc *__restrict__ EG, sc *__restrict__ EH) {
    sc e, p;
    bool right = (i & (nj - 1)) >= h;
    ld_sc(e, &EG[i]); sc_mul(p, e, right ? u : ui); st_sc(&EG[i], p);
    ld_sc(e, &EH[i]); sc_mul(p, e, right ? ui : u); st_sc(&EH[i], p);
}
// (i < h)
__device__ __forceinline__ void ipp_fold_ab(uint32_t i, uint32_t h, const sc &u, const sc &ui, sc *__restrict__ a, sc *__restrict__ b) {
    sc lo, hi, p, q;
    ld_sc(lo, &a[i]); ld_sc(hi, &a[h + i]);
    sc_mul(p, lo, u); sc_mul(q, hi, ui); sc_add_r(p, p, q); st_sc(&a[i], p);
    ld_sc(lo, &b[i]); ld_sc(hi, &b[h + i]);
    sc_mul(p, lo, ui); sc_mul(q, hi, u); sc_add_r(p, p, q); st_sc(&b[i], p);
}
__global__ void __launch_bounds__(128) k_ipp_fold(uint32_t N, uint32_t nj, const sc *__restrict__ uu, sc *__restrict__ a, sc *__restrict__ b, sc *__restrict__ EG,
                                                   sc *__restrict__ EH, uint32_t i0, uint32_t i1) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    uint32_t h = nj >> 1;
    sc u, ui;
    ld_sc(u, &uu[0]); ld_sc(ui, &uu[1]);
    if (i >= i0 && i < i1) ipp_fold_factors(i, nj, h, u, ui, EG, EH);
    if (i < h) ipp_fold_ab(i, h, u, ui, a, b);
}

// ---------------------------------------------------------------- verifier scalars (a8)
// stab_lo[t] = allinv * prod_{bit k of t set} usq[lg-1-k]  (t < 1024, bits k < min(lg,10))
// stab_hi[j] = prod_{bit k of j set} usq[lg-1-(k+10)]
__global__ void __launch_bounds__(128) k_s_tables(const sc *__restrict__ usq, const sc *__restrict__ allinv, uint32_t lg, sc *__restrict__ lo,
                                                   sc *__restrict__ hi, uint32_t nhi) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 1024 + nhi) return;
    sc acc;
    uint32_t idx, shift;
    if (t < 1024) { ld_sc(acc, allinv); idx = t; shift = 0; } else { sc_set_u32(acc, 1); idx = t - 1024; shift = 10; }
#pragma unroll 1
    for (uint32_t k = 0; k < 22; k++) {
        if (!((idx >> k) & 1u)) continue;
        uint32_t bit = k + shift;
        if (bit >= lg) continue;
        sc f; ld_sc(f, &usq[lg - 1 - bit]);
        sc_mul(acc, acc, f);
    }
    if (t < 1024) st_sc(&lo[t], acc); else st_sc(&hi[t - 1024], acc);
}
// g_i = uf (x y^-i wR_i - a s_i) ; h_i = uf (y^-i (x wL_i + wO_i - b s_{N-1-i}) - 1) ; delta partials <y^-i wR_i, wL_i>
// vs = [x, a, b, u]
__global__ void __launch_bounds__(128) k_verify_scalars(uint32_t n, uint32_t N, const sc *__restrict__ vs, const sc *__restrict__ w,
                                                         const sc *__restrict__ yilo, const sc *__restrict__ yihi, const sc *__restrict__ slo,
                                                         const sc *__restrict__ shi, sc *__restrict__ g, sc *__restrict__ hh, sc *__restrict__ dparts) {
    __shared__ sc smem[128];
    sc d; sc_zero(d);
    sc x, ia, ib, u, one;
    ld_sc(x, &vs[0]); ld_sc(ia, &vs[1]); ld_sc(ib, &vs[2]); ld_sc(u, &vs[3]);
    sc_set_u32(one, 1);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        sc yinv, s_i, s_r, p, q, gv, hv;
        pow_lookup<10>(yinv, yilo, yihi, i);
        pow_lookup<10>(s_i, slo, shi, i);
        pow_lookup<10>(s_r, slo, shi, N - 1 - i);
        sc_mul(p, ia, s_i);
        sc_mul(q, ib, s_r);
        if (i < n) {
            sc wl, wr, wo, ywr, t;
            ld_sc(wl, &w[i]); ld_sc(wr, &w[n + i]); ld_sc(wo, &w[2 * (size_t)n + i]);
            sc_mul(ywr, yinv, wr);
            sc_mul(t, ywr, wl); sc_add_r(d, d, t);
            sc_mul(t, x, ywr); sc_sub_r(gv, t, p);
            sc_mul(t, x, wl); sc_add_r(t, t, wo); sc_sub_r(t, t, q); sc_mul(hv, yinv, t); sc_sub_r(hv, hv, one);
        } else {
            sc z, t; sc_zero(z);
            sc_sub_r(gv, z, p);
            sc_sub_r(t, z, q); sc_mul(hv, yinv, t); sc_sub_r(hv, hv, one);
            sc_mul(gv, gv, u); sc_mul(hv, hv, u);
        }
        st_sc(&g[i], gv); st_sc(&hh[i], hv);
    }
    block_sum_scalars<1>(&d, smem);
    if (threadIdx.x == 0) st_sc(&dparts[blockIdx.x], d);
}

// ---------------------------------------------------------------- witness evaluation (SURVEY 8 f-3)
// ConstraintSystem::multiply(left, right) of the reference evaluates both linear combinations over the assignment so far
// (cs_buffer.rs:94-97 -> Prover::multiply, replayed by prover.rs:102-117): a_L[i] = <left_i>, a_R[i] = <right_i>, a_O[i] = a_L a_R.
// One thread per multiplier of the current dependency level (order[k0 .. k1)): every variable an LC references is either a
// committed value, One, or a multiplier of an earlier level.  var = kind << 29 | index (kind 0 a_L, 1 a_R, 2 a_O, 3 V, 4 One).
__device__ __forceinline__ void lc_eval(sc &acc, uint32_t t0, uint32_t t1, const uint32_t *__restrict__ term_var, const sc *__restrict__ term_coeff,
                                        const sc *aL, const sc *aR, const sc *aO, const sc *__restrict__ v) {
    sc_zero(acc);
#pragma unroll 1
    for (uint32_t t = t0; t < t1; t++) {
        uint32_t var = term_var[t], kind = var >> 29, idx = var & 0x1FFFFFFFu;
        sc cf, val, p;
        ld_sc(cf, &term_coeff[t]);
        if (kind == 4) { sc_add_r(acc, acc, cf); continue; }
        ld_sc(val, kind == 0 ? &aL[idx] : kind == 1 ? &aR[idx] : kind == 2 ? &aO[idx] : &v[idx]);
        sc_mul(p, cf, val);
        sc_add_r(acc, acc, p);
    }
}
__global__ void __launch_bounds__(128) k_witness_level(const uint32_t *__restrict__ order, uint32_t k0, uint32_t k1, const uint32_t *__restrict__ lc_ptr,
                                                        const uint32_t *__restrict__ term_var, const sc *__restrict__ term_coeff, sc *aL, sc *aR, sc *aO,
                                                        const sc *__restrict__ v) {
    uint32_t k = k0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= k1) return;
    uint32_t i = order[k];
    sc l, r, o;
    lc_eval(l, lc_ptr[2 * i], lc_ptr[2 * i + 1], term_var, term_coeff, aL, aR, aO, v);
    lc_eval(r, lc_ptr[2 * i + 1], lc_ptr[2 * i + 2], term_var, term_coeff, aL, aR, aO, v);
    sc_mul(o, l, r);
    st_sc(&aL[i], l); st_sc(&aR[i], r); st_sc(&aO[i], o);
}
// A run of consecutive NARROW levels (a MiMC chain is 972 levels of one multiplier each) in ONE launch: a single block walks the
// levels [l0, l1) with a barrier between them instead of one launch per level (~0.7 us against ~3 us per level).
__global__ void __launch_bounds__(256) k_witness_levels_block(const uint32_t *__restrict__ order, const uint32_t *__restrict__ lptr, uint32_t l0, uint32_t l1,
                                                               const uint32_t *__restrict__ lc_ptr, const uint32_t *__restrict__ term_var,
                                                               const sc *__restrict__ term_coeff, sc *aL, sc *aR, sc *aO, const sc *__restrict__ v) {
    for (uint32_t l = l0; l < l1; l++) {
        const uint32_t k1 = lptr[l + 1];
        for (uint32_t k = lptr[l] + threadIdx.x; k < k1; k += blockDim.x) {
            uint32_t i = order[k];
            sc a, b, o;
            lc_eval(a, lc_ptr[2 * i], lc_ptr[2 * i + 1], term_var, term_coeff, aL, aR, aO, v);
            lc_eval(b, lc_ptr[2 * i + 1], lc_ptr[2 * i + 2], term_var, term_coeff, aL, aR, aO, v);
            sc_mul(o, a, b);
            st_sc(&aL[i], a); st_sc(&aR[i], b); st_sc(&aO[i], o);
        }
        __syncthreads(); // the next level reads what this one wrote (same block: the barrier orders the global accesses)
    }
}
// a_O = a_L a_R for the multipliers the caller assigned directly (allocate_multiplier / allocate)
__global__ void __launch_bounds__(128) k_witness_assigned(const uint32_t *__restrict__ order, uint32_t k1, const sc *__restrict__ aL, const sc *__restrict__ aR,
                                                           sc *__restrict__ aO) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= k1) return;
    uint32_t i = order[k];
    sc l, r, o;
    ld_sc(l, &aL[i]); ld_sc(r, &aR[i]);
    sc_mul(o, l, r);
    st_sc(&aO[i], o);
}

// ---------------------------------------------------------------- BPG_FLAG_FAST_BLINDING: s_L, s_R on the device
// out[i] = wide_reduce(Keccak-f[1600](seed || i || pad)[0..64)) : a transcript-seeded counter-mode expansion replacing the
// 2n sequential Merlin TranscriptRng draws of the byte-exact mode (valid proofs, different bytes).
__device__ __forceinline__ uint64_t rotl64(uint64_t x, int n) { return (x << n) | (x >> (64 - n)); }
__device__ void keccak_f1600_dev(uint64_t *a) {
    const uint64_t RC[24] = {0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808AULL, 0x8000000080008000ULL, 0x000000000000808BULL,
                             0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL, 0x000000000000008AULL, 0x0000000000000088ULL,
                             0x0000000080008009ULL, 0x000000008000000AULL, 0x000000008000808BULL, 0x800000000000008BULL, 0x8000000000008089ULL,
                             0x8000000000008003ULL, 0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800AULL, 0x800000008000000AULL,
                             0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL};
    const int RHO[25] = {0, 1, 62, 28, 27, 36, 44, 6, 55, 20, 3, 10, 43, 25, 39, 41, 45, 15, 21, 8, 18, 2, 61, 56, 14};
#pragma unroll 1
    for (int rnd = 0; rnd < 24; rnd++) {
        uint64_t c[5], b[25];
#pragma unroll
        for (int x = 0; x < 5; x++) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
#pragma unroll
        for (int x = 0; x < 5; x++) {
            uint64_t d = c[(x + 4) % 5] ^ rotl64(c[(x + 1) % 5], 1);
#pragma unroll
            for (int y = 0; y < 25; y += 5) a[y + x] ^= d;
        }
#pragma unroll
        for (int x = 0; x < 5; x++)
#pragma unroll
            for (int y = 0; y < 5; y++) {
                int src = x + 5 * y, dst = y + 5 * ((2 * x + 3 * y) % 5);
                b[dst] = RHO[src] ? rotl64(a[src], RHO[src]) : a[src];
            }
#pragma unroll
        for (int y = 0; y < 25; y += 5)
#pragma unroll
            for (int x = 0; x < 5; x++) a[y + x] = b[y + x] ^ (~b[y + (x + 1) % 5] & b[y + (x + 2) % 5]);
        a[0] ^= RC[rnd];
    }
}
__global__ void __launch_bounds__(128) k_expand_blinding(const uint64_t *__restrict__ seed4, uint32_t n, sc *__restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t st[25];
#pragma unroll
    for (int k = 0; k < 25; k++) st[k] = 0;
    st[0] = seed4[0]; st[1] = seed4[1]; st[2] = seed4[2]; st[3] = seed4[3];
    st[4] = i; st[5] = 0x1F; st[16] = 0x8000000000000000ULL;
    keccak_f1600_dev(st);
    u32 R[16];
#pragma unroll
    for (int k = 0; k < 8; k++) { R[2 * k] = (u32)st[k]; R[2 * k + 1] = (u32)(st[k] >> 32); }
    sc r;
    sc_reduce512(r, R);
    st_sc(&out[i], r);
}

// batch verification: Gacc[i] += rho * g[i], Hacc[i] += rho * h[i]  (scalars of proof i folded into the combined check)
__global__ void __launch_bounds__(128) k_axpy_gh(sc rho, const sc *__restrict__ g, const sc *__restrict__ h, uint32_t n, sc *__restrict__ Gacc,
                                                  sc *__restrict__ Hacc) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sc a, x, p;
    ld_sc(x, &g[i]); ld_sc(a, &Gacc[i]); sc_mul(p, rho, x); sc_add_r(a, a, p); st_sc(&Gacc[i], a);
    ld_sc(x, &h[i]); ld_sc(a, &Hacc[i]); sc_mul(p, rho, x); sc_add_r(a, a, p); st_sc(&Hacc[i], a);
}
