// kernels_msm.cuh -- fixed-base signed-digit Pippenger over the resident window tables (K2/K4/K6).
//
// Replaces RistrettoPoint::multiscalar_mul / vartime_multiscalar_mul of curve25519-dalek 1.x as called by
// the bulletproofs fork inside Prover::prove, InnerProductProof::create and Verifier::verify
// (reference call sites src/bin/prover.rs:93, src/bin/verifier.rs:90).
//
// Every term (scalar k, resident point P) is recoded into 16 signed 16-bit digits d_w.  Because the table holds
// 2^(16w) P for every window, the pair (term, w) contributes d_w * tab[w][P] and ALL windows share one bucket
// set per output group: bucket |d| accumulates sign(d) * tab[w][P].  The result is sum_b b * bucket[b]; there
// are no doublings and no per-window combine.
//   1. k_msm_digits<COUNT>   histogram of bucket populations            (atomics on a 128 KB..400 KB array, L2)
//   2. k_msm_scan            exclusive scan -> bucket offsets
//   3. k_msm_digits<SCATTER> counting-sort scatter of (table index | sign) into bucket order
//   4. k_msm_accumulate      each thread sums one fixed-size chunk of the sorted pairs (uniform work whatever the
//                            scalar distribution); runs that cover a whole bucket are written directly, runs cut
//                            by a chunk boundary go to per-chunk partial slots
//   5. k_msm_finish          per bucket: identity if empty, sum of partial slots if split over few chunks,
//                            else queued for 6
//   6. k_msm_heavy           block-wide tree reduction for buckets split over many chunks (e.g. the bit-valued
//                            a_L/a_R of range proofs put half of all terms in bucket 1)
//   7. k_msm_rowcol / k_msm_wfinal / k_msm_combine   sum_b b * bucket[b] via row and column sums (depth ~40)
#pragma once
#include "kernels_core.cuh"

struct msm_params {
    msm_seg seg[BPG_MAX_SEGS];
    int nseg;
    uint32_t total;
    uint32_t ptotal;
    uint32_t varbase; // 1: variable points (no window tables): entry = point index, window w of group g sums into group 16 g + w
};

// signed 16-bit digits: d in [-32768, 32767], sum d_w 2^(16w) = k  (k < 2^253 so the top digit never carries out)
__device__ __forceinline__ void sc_digits16(int *d, const sc &k) {
    int carry = 0;
#pragma unroll
    for (int w = 0; w < 16; w++) {
        int raw = (int)((k.v[w >> 1] >> (16 * (w & 1))) & 0xFFFF) + carry;
        carry = raw >= 32768;
        d[w] = raw - (carry << 16);
    }
}

// SPLIT = 0: bucket = group * BPG_NBP + |d|                               (2^15 buckets per group, one pair per digit)
// SPLIT = 1: d = dl + 256 dh, buckets (2 group + 0) * 129 + |dl| and (2 group + 1) * 129 + |dh|   (small MSMs: 2 x 129 buckets
//            per group and two pairs per digit, reduced by k_mat_reduce -- see the late-fold section below)
// One counter update per lane, aggregated when every active lane of the warp hits the SAME counter (binary-valued witnesses
// of range proofs: a_L in {0,1}, a_R in {0,-1} put whole warps into one bucket per window, and 2^19 same-address atomics
// serialise; MSM-bits at 2^22 terms: 3.8 -> ms).  All 32 lanes must call it.  Returns the old counter value + the lane's
// rank among the active lanes (its slot when scattering).
__device__ __forceinline__ uint32_t warp_counter_add(uint32_t *__restrict__ arr, uint32_t bkt, bool active) {
    const unsigned full = 0xFFFFFFFFu;
    unsigned mask = __ballot_sync(full, active);
    if (!mask) return 0;
    int leader = __ffs(mask) - 1;
    uint32_t lb = __shfl_sync(full, bkt, leader);
    if (__all_sync(full, !active || bkt == lb)) {
        uint32_t lane = threadIdx.x & 31u, base = 0;
        if ((int)lane == leader) base = atomicAdd(&arr[lb], (uint32_t)__popc(mask));
        base = __shfl_sync(full, base, leader);
        return base + (uint32_t)__popc(mask & ((1u << lane) - 1u));
    }
    return active ? atomicAdd(&arr[bkt], 1u) : 0u;
}
// SPLIT = 1 pairs of one digit dw = dl + 256 dh: buckets base + |dl| and base + 129 + |dh|, entry ent with the digit's sign
template <int SCATTER>
__device__ __forceinline__ void emit_split_digit(uint32_t *__restrict__ counts_or_cursor, uint32_t *__restrict__ sorted, uint32_t base, int dw, uint32_t ent) {
    int dl = ((dw + 128) & 255) - 128; // [-128, 127]
    int dh = (dw - dl) >> 8;           // exact ; [-128, 128]
#pragma unroll
    for (int part = 0; part < 2; part++) {
        int dd = part ? dh : dl;
        uint32_t mag = dd < 0 ? (uint32_t)(-dd) : (uint32_t)dd;
        uint32_t pos = warp_counter_add(counts_or_cursor, base + part * 129u + mag, dd != 0);
        if (SCATTER && dd != 0) sorted[pos] = ent | (dd < 0 ? 0x80000000u : 0u);
    }
}
template <int SCATTER, int SPLIT>
__global__ void __launch_bounds__(256) k_msm_digits(msm_params P, uint32_t *__restrict__ counts_or_cursor, uint32_t *__restrict__ sorted) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = t < P.total; // no early return: the warp-aggregated counter update needs all 32 lanes
    int d[16];
#pragma unroll
    for (int w = 0; w < 16; w++) d[w] = 0;
    uint32_t grp = 0, pidx = 0;
    if (valid) {
        int si = 0;
#pragma unroll
        for (int k = 1; k < BPG_MAX_SEGS; k++)
            if (k < P.nseg && t >= P.seg[k].start) si = k;
        const msm_seg &S = P.seg[si];
        uint32_t j = t - S.start;
        sc k;
        ld_sc(k, &S.scalars[j]);
        if (S.reduce) sc_reduce(k, k);
        sc_digits16(d, k);
        grp = S.group;
        if (S.alt) grp ^= ((j + S.j0) >> (S.alt - 1)) & 1u;
        pidx = S.p0 + j;
    }
    const uint32_t gstride = SPLIT ? 2u * 129u : BPG_NBP;
    if (P.varbase) grp *= 16u;
    uint32_t base = grp * gstride;
#pragma unroll
    for (int w = 0; w < 16; w++) {
        int dw = d[w];
        uint32_t ent = P.varbase ? pidx : (uint32_t)w * P.ptotal + pidx;
        if (P.varbase) base = (grp + (uint32_t)w) * gstride;
        if (SPLIT) {
            emit_split_digit<SCATTER>(counts_or_cursor, sorted, base, dw, ent);
        } else {
            uint32_t mag = dw < 0 ? (uint32_t)(-dw) : (uint32_t)dw;
            uint32_t pos = warp_counter_add(counts_or_cursor, base + mag, dw != 0);
            if (SCATTER && dw != 0) sorted[pos] = ent | (dw < 0 ? 0x80000000u : 0u);
        }
    }
}

// ---- large MSMs (>= 2^19 terms, fixed-base, up to 4 output groups): the two passes above are bound by global atomics (16 per term and pass:
// 0.61 + 1.02 ms of a 7.3 ms MSM at 2^22 terms).  Privatised versions (histogram: always; scatter: up to 2^20 terms, see msm_run): one 1024-thread block per SM keeps the 33 024
// counters of the group in shared memory (132 KB).
//   histogram: shared-memory atomics, then one global atomic per non-empty counter and block;
//   scatter:   the block counts its own tile again, reserves a contiguous range per bucket with ONE global atomic
//              (cursor[b] += local count), and hands out positions inside the range with shared-memory atomics.
// Both kernels walk the terms with the same grid-stride pattern, so a block meets the same terms in both phases.
// The order of the pairs inside a bucket differs from the plain kernels'; the bucket sums (group elements) do not.
// segment / group of term t without touching its scalar (the privatised kernels below skip the terms of other groups first)
__device__ __forceinline__ const msm_seg &msm_term_seg(const msm_params &P, uint32_t t, uint32_t &j, uint32_t &grp) {
    int si = 0;
#pragma unroll
    for (int k = 1; k < BPG_MAX_SEGS; k++)
        if (k < P.nseg && t >= P.seg[k].start) si = k;
    const msm_seg &S = P.seg[si];
    j = t - S.start;
    grp = S.group;
    if (S.alt) grp ^= ((j + S.j0) >> (S.alt - 1)) & 1u;
    return S;
}
__device__ __forceinline__ void msm_seg_digits(const msm_seg &S, uint32_t j, int *d, uint32_t &pidx) {
    sc k;
    ld_sc(k, &S.scalars[j]);
    if (S.reduce) sc_reduce(k, k);
    sc_digits16(d, k);
    pidx = S.p0 + j;
}
// grid (blocks, groups): blockIdx.y = the output group whose 33 024 counters this block keeps in shared memory; terms of other
// groups are skipped before their scalar is read (IPP rounds: L / R alternate by halves, so a block reads half of the scalars)
__global__ void __launch_bounds__(1024, 1) k_msm_hist_smem(msm_params P, uint32_t *__restrict__ counts) {
    extern __shared__ uint32_t scnt[];
    const uint32_t g = blockIdx.y;
    for (uint32_t i = threadIdx.x; i < BPG_NBP; i += blockDim.x) scnt[i] = 0;
    __syncthreads();
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < P.total; t += gridDim.x * blockDim.x) {
        uint32_t j, grp;
        const msm_seg &S = msm_term_seg(P, t, j, grp);
        if (grp != g) continue;
        int d[16];
        uint32_t pidx;
        msm_seg_digits(S, j, d, pidx);
#pragma unroll
        for (int w = 0; w < 16; w++) {
            int dw = d[w];
            if (dw == 0) continue;
            atomicAdd(&scnt[dw < 0 ? (uint32_t)(-dw) : (uint32_t)dw], 1u);
        }
    }
    __syncthreads();
    uint32_t *cg = counts + (size_t)g * BPG_NBP;
    for (uint32_t i = threadIdx.x; i < BPG_NBP; i += blockDim.x) {
        uint32_t c = scnt[i];
        if (c) atomicAdd(&cg[i], c);
    }
}
// (g0: first group of this launch -- msm_run_local launches the groups of a multi-group MSM one after the other when each of
// them is within the privatised scatter's reach, so that only ONE group's open ranges compete for L2 at a time)
__global__ void __launch_bounds__(1024, 1) k_msm_scatter_smem(msm_params P, uint32_t *__restrict__ cursor, uint32_t *__restrict__ sorted, uint32_t g0) {
    extern __shared__ uint32_t scnt[];
    const uint32_t g = g0 + blockIdx.y;
    for (uint32_t i = threadIdx.x; i < BPG_NBP; i += blockDim.x) scnt[i] = 0;
    __syncthreads();
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < P.total; t += gridDim.x * blockDim.x) {
        uint32_t j, grp;
        const msm_seg &S = msm_term_seg(P, t, j, grp);
        if (grp != g) continue;
        int d[16];
        uint32_t pidx;
        msm_seg_digits(S, j, d, pidx);
#pragma unroll
        for (int w = 0; w < 16; w++) {
            int dw = d[w];
            if (dw == 0) continue;
            atomicAdd(&scnt[dw < 0 ? (uint32_t)(-dw) : (uint32_t)dw], 1u);
        }
    }
    __syncthreads();
    uint32_t *cg = cursor + (size_t)g * BPG_NBP;
    for (uint32_t i = threadIdx.x; i < BPG_NBP; i += blockDim.x) { // reserve [base, base + count) of bucket i for this block
        uint32_t c = scnt[i];
        scnt[i] = c ? atomicAdd(&cg[i], c) : 0u;
    }
    __syncthreads();
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < P.total; t += gridDim.x * blockDim.x) {
        uint32_t j, grp;
        const msm_seg &S = msm_term_seg(P, t, j, grp);
        if (grp != g) continue;
        int d[16];
        uint32_t pidx;
        msm_seg_digits(S, j, d, pidx);
#pragma unroll
        for (int w = 0; w < 16; w++) {
            int dw = d[w];
            if (dw == 0) continue;
            uint32_t pos = atomicAdd(&scnt[dw < 0 ? (uint32_t)(-dw) : (uint32_t)dw], 1u);
            sorted[pos] = ((uint32_t)w * P.ptotal + pidx) | (dw < 0 ? 0x80000000u : 0u);
        }
    }
}

// (Tried and dropped, profiles/r02_sort_variants.jsonl: a two-pass bin sort for MSMs beyond the reach of k_msm_scatter_smem --
// partition the pairs into bins of 32 buckets with shared-memory counters per tile, then distribute every 8 192-record slice
// with one global atomic per (slice, bucket).  0.46 + 0.42 ms against 0.70 ms for the plain cursor-ordered scatter at 2^21 terms.)
// Exclusive scan of counts[0..n) into offsets[0..n] and cursor[0..n).  Tiles of 1024 counters, one 256-thread block
// each (small blocks so the scan can run in the register space left over by another context's accumulate grid).
// A block publishes its tile total, then sums the totals of all earlier tiles (<= 128 values, one coalesced read);
// tiles are claimed through a ticket so a block only ever waits for blocks that have already started.
// state[0] = ticket, state[1 + i] = total of tile i | 0x80000000 once published (zeroed by the host before launch).
__global__ void __launch_bounds__(256) k_msm_scan(const uint32_t *__restrict__ counts, uint32_t n, uint32_t *__restrict__ offsets, uint32_t *__restrict__ cursor,
                                                   volatile uint32_t *state) {
    __shared__ uint32_t wsum[8];
    __shared__ uint32_t s_tile, s_prefix;
    uint32_t t = threadIdx.x, lane = t & 31, wid = t >> 5;
    if (t == 0) s_tile = atomicAdd((uint32_t *)&state[0], 1u);
    __syncthreads();
    uint32_t tile = s_tile;
    uint32_t i0 = tile * 1024u + 4u * t;
    uint32_t v[4];
#pragma unroll
    for (int k = 0; k < 4; k++) v[k] = (i0 + k < n) ? counts[i0 + k] : 0u;
    uint32_t local = v[0] + v[1] + v[2] + v[3];
    uint32_t x = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o); if (lane >= o) x += y; }
    if (lane == 31) wsum[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = lane < 8 ? wsum[lane] : 0u;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { uint32_t y = __shfl_up_sync(0xFFFFFFFFu, w, o); if (lane >= o) w += y; }
        if (lane < 8) wsum[lane] = w;
        if (lane == 7) { __threadfence(); state[1 + tile] = w | 0x80000000u; } // publish this tile's total
    }
    __syncthreads();
    // look back: sum of all earlier tiles' totals (each thread polls at most one predecessor)
    uint32_t part = 0;
    for (uint32_t p = t; p < tile; p += 256) {
        uint32_t a;
        do { a = state[1 + p]; } while (!(a & 0x80000000u));
        part += a & 0x7FFFFFFFu;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xFFFFFFFFu, part, o);
    __shared__ uint32_t psum[8];
    if (lane == 0) psum[wid] = part;
    __syncthreads();
    if (t == 0) { uint32_t pp = 0; for (int k = 0; k < 8; k++) pp += psum[k]; s_prefix = pp; }
    __syncthreads();
    uint32_t excl = s_prefix + (wid ? wsum[wid - 1] : 0u) + x - local;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (i0 + k < n) { offsets[i0 + k] = excl; cursor[i0 + k] = excl; }
        excl += v[k];
    }
    if (i0 <= n - 1 && n - 1 < i0 + 4) offsets[n] = excl; // the thread owning the last counter writes the grand total
}

__device__ __forceinline__ void block_tree_sum_ilp(ge &acc, ge *smem, int nthreads) { // result in thread 0
    int t = threadIdx.x;
    st_ge(&smem[t], acc);
    __syncthreads();
    for (int s = nthreads >> 1; s > 0; s >>= 1) {
        if (t < s) {
            ge b;
            ld_ge(b, &smem[t + s]);
            ge_add_ilp(acc, acc, b);
            st_ge(&smem[t], acc);
        }
        __syncthreads();
    }
}
// value -> table entry (negated if the sign bit is set)
__device__ __forceinline__ void msm_load_entry(ge_an &a, const ge_an *__restrict__ tab, uint32_t v) {
    ld_an(a, &tab[v & 0x7FFFFFFFu]);
    if (v & 0x80000000u) {
        fe t = a.ypx; a.ypx = a.ymx; a.ymx = t;
        fe_neg(a.t2d, a.t2d);
    }
}

// partial slot layout: partial[2*chunk + 0] = run touching the chunk start, [2*chunk + 1] = run touching the chunk end only
// (Tried and dropped, profiles/r02_accumulate_variants.jsonl: prefetch.global.L1 / .L2 of the next pair's entry one iteration
// ahead -- 12.9 -> 9.6 G additions/s; entries padded to one aligned 128-byte line -- DRAM traffic down, time unchanged;
// 5 / 6 resident blocks per SM (96 / 80 registers) -- neutral / slower; requesting the next entry between the two multiplication
// stages keeps it live through stage 2: 134 registers, and ptxas sinks the loads to the end of the body anyway.)
#ifndef BPG_ACC_MINBLOCKS
#define BPG_ACC_MINBLOCKS 1
#endif
__global__ void __launch_bounds__(128, BPG_ACC_MINBLOCKS) k_msm_accumulate(const uint32_t *__restrict__ sorted, const uint32_t *__restrict__ offsets, uint32_t nbuckets,
                                                         const ge_an *__restrict__ tab, ge *__restrict__ buckets, ge *__restrict__ partial, uint32_t CH) {
    uint32_t M = offsets[nbuckets];
    uint32_t chunk = blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t start64 = (uint64_t)chunk * CH;
    if (start64 >= M) return;
    uint32_t start = (uint32_t)start64, end = min(M, start + CH);
    // bucket containing `start`: largest b with offsets[b] <= start
    uint32_t lo = 0, hi = nbuckets;
    while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (offsets[mid] <= start) lo = mid; else hi = mid; }
    uint32_t b = lo;
    uint32_t bend = offsets[b + 1];
    while (bend <= start) { b++; bend = offsets[b + 1]; } // skip empty buckets that share the offset
    uint32_t bstart = offsets[b];
    uint32_t run_start = start;
    ge acc;
    ge_identity(acc);
    // Flat loop: every lane performs exactly one mixed addition per iteration, in lockstep.  A bucket boundary only
    // triggers a short divergent prologue (store the finished run, step to the next non-empty bucket); the nested
    // run/flush loops this replaces left half of the lanes idle (ncu: 16.6 active threads per instruction).
    uint32_t v = sorted[start];
#pragma unroll 1
    for (uint32_t pos = start; pos < end; pos++) {
        if (pos == bend) {
            bool complete = (run_start == bstart);
            if (complete) st_ge(&buckets[b], acc);
            else st_ge(&partial[2ull * chunk + (run_start == start ? 0 : 1)], acc);
            do { b++; bstart = bend; bend = offsets[b + 1]; } while (bend <= pos);
            run_start = pos;
            ge_identity(acc);
        }
        uint32_t vn = (pos + 1 < end) ? sorted[pos + 1] : 0u;
        ge_an a;
        msm_load_entry(a, tab, v);
        ge_add_an(acc, acc, a);
        v = vn;
    }
    // last run of the chunk: complete only if it started at its bucket's first pair and ends at its last
    bool complete = (run_start == bstart) && (end == bend);
    if (complete) st_ge(&buckets[b], acc);
    else st_ge(&partial[2ull * chunk + (run_start == start ? 0 : 1)], acc);
}

__global__ void __launch_bounds__(64) k_msm_finish(const uint32_t *__restrict__ offsets, uint32_t nbuckets, ge *__restrict__ buckets,
                                                     const ge *__restrict__ partial, uint32_t *__restrict__ heavy_list, uint32_t *__restrict__ heavy_count,
                                                     uint32_t CH) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbuckets) return;
    uint32_t s = offsets[b], e = offsets[b + 1];
    if (s == e) { ge id; ge_identity(id); st_ge(&buckets[b], id); return; }
    uint32_t c0 = s / CH, c1 = (e - 1) / CH;
    if (c0 == c1) return; // written by the accumulate kernel
    if (c1 - c0 + 1 > BPG_HEAVY_SPAN) { heavy_list[atomicAdd(heavy_count, 1u)] = b; return; }
    ge acc;
    ld_ge(acc, &partial[2ull * c0 + ((s % CH) == 0 ? 0 : 1)]);
#pragma unroll 1
    for (uint32_t c = c0 + 1; c <= c1; c++) {
        ge q;
        ld_ge(q, &partial[2ull * c]);
        ge_add_ilp(acc, acc, q);
    }
    st_ge(&buckets[b], acc);
}
// Heavy buckets (spanning more than BPG_HEAVY_SPAN chunks): grid (heavy bucket, segment).  Block (h, y) sums segment y of
// BPG_HEAVY_SEGS equal parts of the bucket's partial slots (threads stride, then a tree in shared memory) into
// heavy_part[h][y]; k_msm_heavy_final adds the segments.  A range-proof witness puts half of ALL pairs into one bucket
// (2^15 partial slots at 2^22 terms): one 64-thread block per bucket took 1 ms for it.
#define BPG_HEAVY_SEGS 32u
__global__ void __launch_bounds__(64) k_msm_heavy(const uint32_t *__restrict__ offsets, const ge *__restrict__ partial, const uint32_t *__restrict__ heavy_list,
                                                   const uint32_t *__restrict__ heavy_count, uint32_t CH, ge *__restrict__ heavy_part) {
    __shared__ ge smem[64];
    uint32_t nh = *heavy_count, y = blockIdx.y;
    for (uint32_t h = blockIdx.x; h < nh; h += gridDim.x) {
        uint32_t b = heavy_list[h];
        uint32_t s = offsets[b], e = offsets[b + 1];
        uint32_t c0 = s / CH, c1 = (e - 1) / CH;
        uint32_t nc = c1 - c0 + 1, per = (nc + BPG_HEAVY_SEGS - 1) / BPG_HEAVY_SEGS;
        uint32_t lo = c0 + y * per, hi = min(c1 + 1, lo + per);
        ge acc;
        ge_identity(acc);
        for (uint32_t c = lo + threadIdx.x; c < hi; c += blockDim.x) {
            ge q;
            uint32_t slot = (c == c0 && (s % CH) != 0) ? 1u : 0u;
            ld_ge(q, &partial[2ull * c + slot]);
            ge_add_ilp(acc, acc, q);
        }
        block_tree_sum_ilp(acc, smem, 64);
        if (threadIdx.x == 0) st_ge(&heavy_part[(size_t)h * BPG_HEAVY_SEGS + y], acc);
        __syncthreads();
    }
}
__global__ void __launch_bounds__(32) k_msm_heavy_final(ge *__restrict__ buckets, const uint32_t *__restrict__ heavy_list, const uint32_t *__restrict__ heavy_count,
                                                         const ge *__restrict__ heavy_part) {
    __shared__ ge smem[32];
    uint32_t nh = *heavy_count, lane = threadIdx.x;
    for (uint32_t h = blockIdx.x; h < nh; h += gridDim.x) {
        ge acc, o;
        ld_ge(acc, &heavy_part[(size_t)h * BPG_HEAVY_SEGS + lane]);
        st_ge(&smem[lane], acc);
        __syncwarp();
        for (int s2 = 16; s2 > 0; s2 >>= 1) {
            if (lane < (uint32_t)s2) { ld_ge(o, &smem[lane + s2]); ge_add_ilp(acc, acc, o); st_ge(&smem[lane], acc); }
            __syncwarp();
        }
        if (lane == 0) st_ge(&buckets[heavy_list[h]], acc);
        __syncwarp();
    }
}

// ---- weighted bucket sum  S = sum_b b * bucket[b]  over b = 256 q + r  (q < 129, r < 256):
//      S = sum_r r * C_r + 256 * sum_q q * R_q   with row sums R_q = sum_r bucket[256 q + r] and column sums C_r.
// Depth ~40 point operations instead of one serial pass over 32 768 buckets; every level is a block-wide tree
// whose additions interleave their independent field multiplications (ge_add_ilp) because these kernels run at
// one or two warps per scheduler.
#define BPG_NROWS 129u
#define BPG_NCOLS 256u
// grid (129 + 256, groups), 64 threads: rc[g][0..129) = row sums, rc[g][129..385) = column sums
// (64-thread blocks, like every tail kernel: <= 8 K registers per block, so they fit next to resident accumulate blocks)
__global__ void __launch_bounds__(64) k_msm_rowcol(const ge *__restrict__ buckets, ge *__restrict__ rc) {
    __shared__ ge smem[64];
    uint32_t g = blockIdx.y, idx = blockIdx.x, t = threadIdx.x;
    const ge *B = buckets + (size_t)g * BPG_NBP;
    ge acc, o;
    if (idx < BPG_NROWS) {
        ld_ge(acc, &B[256u * idx + t]);
#pragma unroll 1
        for (uint32_t k = 1; k < 4; k++) { ld_ge(o, &B[256u * idx + 64u * k + t]); ge_add_ilp(acc, acc, o); }
    } else {
        uint32_t r = idx - BPG_NROWS;
        ld_ge(acc, &B[256u * t + r]);
        ld_ge(o, &B[256u * (t + 64u) + r]);
        ge_add_ilp(acc, acc, o);
        if (t == 0) { ld_ge(o, &B[256u * 128u + r]); ge_add_ilp(acc, acc, o); }
    }
    block_tree_sum_ilp(acc, smem, 64);
    if (t == 0) st_ge(&rc[(size_t)g * (BPG_NROWS + BPG_NCOLS) + idx], acc);
}
// Work-lean variant of k_msm_rowcol for the throughput regime (many provers share the GPU, so issue slots matter more than
// the depth of one reduction): every lane first sums 8 (rows) or ~16 (columns) buckets serially and only the last 5 / 3
// levels are a tree with idle lanes: ~2 800 warp-level additions per group instead of ~5 000.
// grid (129 + 64, groups), 32 threads.  Blocks [0,129): row q = blockIdx.x, lane l sums columns l, l+32, ...;
// blocks [129,193): columns 4 c .. 4 c + 3, lane = (part = lane >> 2, col = lane & 3) sums rows part, part + 8, ...
__global__ void __launch_bounds__(32) k_msm_rowcol_lean(const ge *__restrict__ buckets, ge *__restrict__ rc) {
    __shared__ ge smem[32];
    uint32_t g = blockIdx.y, idx = blockIdx.x, lane = threadIdx.x;
    const ge *B = buckets + (size_t)g * BPG_NBP;
    ge acc, o;
    if (idx < BPG_NROWS) {
        ld_ge(acc, &B[256u * idx + lane]);
#pragma unroll 1
        for (uint32_t k = 1; k < 8; k++) { ld_ge(o, &B[256u * idx + 32u * k + lane]); ge_add_ilp(acc, acc, o); }
        st_ge(&smem[lane], acc);
        __syncwarp();
        for (int s2 = 16; s2 > 0; s2 >>= 1) {
            if (lane < (uint32_t)s2) { ld_ge(o, &smem[lane + s2]); ge_add_ilp(acc, acc, o); st_ge(&smem[lane], acc); }
            __syncwarp();
        }
        if (lane == 0) st_ge(&rc[(size_t)g * (BPG_NROWS + BPG_NCOLS) + idx], acc);
    } else {
        uint32_t part = lane >> 2, col = 4u * (idx - BPG_NROWS) + (lane & 3u);
        ld_ge(acc, &B[256u * part + col]);
#pragma unroll 1
        for (uint32_t q = part + 8; q < BPG_NROWS; q += 8) { ld_ge(o, &B[256u * q + col]); ge_add_ilp(acc, acc, o); }
        st_ge(&smem[lane], acc);
        __syncwarp();
        for (int s2 = 16; s2 >= 4; s2 >>= 1) { // lanes 4 p + c: add the lane 4 (p + s2/4) + c
            if (lane < (uint32_t)s2) { ld_ge(o, &smem[lane + s2]); ge_add_ilp(acc, acc, o); st_ge(&smem[lane], acc); }
            __syncwarp();
        }
        if (lane < 4) st_ge(&rc[(size_t)g * (BPG_NROWS + BPG_NCOLS) + BPG_NROWS + col], acc);
    }
}
// w * P for a small weight (<= 8 bits), double-and-add from the top bit
__device__ __forceinline__ void ge_small_mul(ge &r, uint32_t w, const ge &p) {
    ge acc;
    ge_identity(acc);
    if (w) {
        int top = 31 - __clz(w);
        acc = p;
#pragma unroll 1
        for (int k = top - 1; k >= 0; k--) {
            ge_dbl_ilp(acc, acc);
            if ((w >> k) & 1u) ge_add_ilp(acc, acc, p);
        }
    }
    r = acc;
}
// grid (8, groups), 64 threads.  Blocks 0..3: columns [64 x, 64 x + 64) -> sum r C_r ; blocks 4..7: rows [64 (x-4), ..) -> 256 sum q R_q
// (rows exist for q < 129; the remaining threads contribute the identity).
// out8[g][x] ; k_msm_combine adds the eight partial results of a group.
__global__ void __launch_bounds__(64, 8) k_msm_wfinal(const ge *__restrict__ rc, ge *__restrict__ out8) {
    __shared__ ge smem[64];
    uint32_t g = blockIdx.y, x = blockIdx.x, t = threadIdx.x;
    const ge *base = rc + (size_t)g * (BPG_NROWS + BPG_NCOLS);
    ge item, acc;
    if (x < 4) {
        uint32_t r = 64u * x + t;
        ld_ge(item, &base[BPG_NROWS + r]);
        ge_small_mul(acc, r, item);
    } else {
        uint32_t q = 64u * (x - 4) + t;
        if (q < BPG_NROWS) { ld_ge(item, &base[q]); ge_small_mul(acc, q, item); } else ge_identity(acc);
    }
    block_tree_sum_ilp(acc, smem, 64);
    if (t == 0) {
        if (x >= 4) {
#pragma unroll 1
            for (int k = 0; k < 8; k++) ge_dbl_ilp(acc, acc);
        }
        st_ge(&out8[8 * (size_t)g + x], acc);
    }
}
// one 32-thread block per group: sum of the 8 partial results
__global__ void __launch_bounds__(32) k_msm_combine(const ge *__restrict__ in8, ge *__restrict__ out) {
    __shared__ ge smem[8];
    uint32_t g = blockIdx.x, t = threadIdx.x;
    ge acc;
    if (t < 8) { ld_ge(acc, &in8[8 * (size_t)g + t]); st_ge(&smem[t], acc); }
    __syncwarp();
    for (int s2 = 4; s2 > 0; s2 >>= 1) {
        if (t < (uint32_t)s2) { ge b; ld_ge(b, &smem[t + s2]); ge_add_ilp(acc, acc, b); st_ge(&smem[t], acc); }
        __syncwarp();
    }
    if (t == 0) st_ge(&out[g], acc);
}

// =====================================================================================================================
// Late fold: materialise the folded generators G^(k), H^(k) of the inner-product argument once, after k rounds.
//
// dalek's InnerProductProof::create (behind src/bin/prover.rs:93) folds the generator vectors in every round.  Here the
// first k rounds are evaluated over the original generators with expanded scalars (k_ipp_expand); every later round would
// still pay a full 2N-term MSM although only n' = N / 2^k folded generators remain.  So at round k the folded generators
//     G^(k)_i = sum_{p = i (mod n')} EG[p] G_p ,   H^(k)_i = sum_{p = i (mod n')} EH[p] H_p        (i < n')
// are computed as ONE multi-output MSM over the resident window tables (2 n' outputs), 16-window tables are built for
// them, and the remaining rounds run the same engine over those 2 n' points -- a few thousand pairs instead of 2N * 16.
//
// Multi-output MSM: an output has only N / n' * 16 pairs, too few for 2^15 buckets.  Each signed 16-bit digit d of a
// (term, window) pair is split again, d = dl + 256 dh with dl in [-128, 127], dh in [-128, 128], and the SAME table entry
// 2^(16w) P goes to bucket |dl| of the output's "low" set and to bucket |dh| of its "high" set (2 x 129 buckets per
// output, no extra tables, no doublings).  Output = sum_b b * low_b + 256 * sum_b b * high_b.
// The sort / accumulate / finish kernels above are reused unchanged (bucket = (2 * output + set) * 129 + |digit|).
#define BPG_MAT_NB 129u
// [p0, p1): this rank's point range (all of [0, N) unless the proof is sharded): thread t < p1 - p0 handles G_{p0 + t}, the next
// p1 - p0 threads handle H_{p0 + ..} -- the same per-vector slices the round MSMs use, so EG / EH are only ever needed there
template <int SCATTER>
__global__ void __launch_bounds__(256) k_mat_digits(uint32_t N, uint32_t nprime, uint32_t cap, uint32_t ptotal, const sc *__restrict__ EG, const sc *__restrict__ EH,
                                                     uint32_t p0, uint32_t p1, uint32_t *__restrict__ counts_or_cursor, uint32_t *__restrict__ sorted) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, span = p1 - p0;
    if (t >= 2 * span) return;
    bool isH = t >= span;
    uint32_t p = p0 + (isH ? t - span : t);
    (void)N;
    sc k;
    ld_sc(k, isH ? &EH[p] : &EG[p]);
    int d[16];
    sc_digits16(d, k);
    uint32_t out = (p & (nprime - 1)) + (isH ? nprime : 0u);
    uint32_t pidx = p + (isH ? cap : 0u);
    uint32_t base = 2u * out * BPG_MAT_NB;
#pragma unroll
    for (int w = 0; w < 16; w++) {
        int dw = d[w];
        if (dw == 0) continue;
        int dl = ((dw + 128) & 255) - 128;   // [-128, 127]
        int dh = (dw - dl) >> 8;             // exact: dw - dl is a multiple of 256 ; [-128, 128]
        uint32_t ent = (uint32_t)w * ptotal + pidx;
#pragma unroll
        for (int part = 0; part < 2; part++) {
            int dd = part ? dh : dl;
            if (dd == 0) continue;
            uint32_t mag = dd < 0 ? (uint32_t)(-dd) : (uint32_t)dd;
            uint32_t bkt = base + part * BPG_MAT_NB + mag;
            if (SCATTER) {
                uint32_t pos = atomicAdd(&counts_or_cursor[bkt], 1u);
                sorted[pos] = ent | (dd < 0 ? 0x80000000u : 0u);
            } else {
                atomicAdd(&counts_or_cursor[bkt], 1u);
            }
        }
    }
}
// The same two passes with ONE BLOCK PER OUTPUT: all pairs of output o (terms p = o, o + n', o + 2n', ... inside this rank's
// point range [p0, p1)) land in the 2 x 129 buckets of that output, so the block counts them in shared memory,
// writes the counts without atomics, and -- after the scan -- places the pairs with shared-memory ranks: no global atomics and
// every block writes one contiguous 32 KB region (k_mat_digits: 2 x 67 M global atomics, 0.31 + 1.44 ms of a 2^20 proof).
template <int PLACE>
__global__ void __launch_bounds__(256) k_mat_block(uint32_t p0, uint32_t p1, uint32_t nprime, uint32_t cap, uint32_t ptotal, const sc *__restrict__ EG,
                                                   const sc *__restrict__ EH, uint32_t *__restrict__ counts, const uint32_t *__restrict__ offsets, uint32_t *__restrict__ sorted) {
    __shared__ uint32_t scnt[2 * BPG_MAT_NB];
    const uint32_t out = blockIdx.x; // [0, n') : G side, [n', 2 n') : H side
    const bool isH = out >= nprime;
    const uint32_t q = isH ? out - nprime : out;
    const uint32_t base = 2u * out * BPG_MAT_NB;
    for (uint32_t i = threadIdx.x; i < 2 * BPG_MAT_NB; i += blockDim.x) scnt[i] = PLACE ? offsets[base + i] : 0u;
    __syncthreads();
    const uint32_t kfirst = p0 > q ? (p0 - q + nprime - 1) / nprime : 0u; // first term of this output inside [p0, p1)
    for (uint32_t p = q + nprime * (kfirst + threadIdx.x); p < p1; p += nprime * blockDim.x) {
        sc k;
        ld_sc(k, isH ? &EH[p] : &EG[p]);
        int d[16];
        sc_digits16(d, k);
        const uint32_t pidx = p + (isH ? cap : 0u);
#pragma unroll
        for (int w = 0; w < 16; w++) {
            int dw = d[w];
            if (dw == 0) continue;
            int dl = ((dw + 128) & 255) - 128;
            int dh = (dw - dl) >> 8;
            uint32_t ent = (uint32_t)w * ptotal + pidx;
#pragma unroll
            for (int part = 0; part < 2; part++) {
                int dd = part ? dh : dl;
                if (dd == 0) continue;
                uint32_t mag = dd < 0 ? (uint32_t)(-dd) : (uint32_t)dd;
                uint32_t pos = atomicAdd(&scnt[part * BPG_MAT_NB + mag], 1u);
                if (PLACE) sorted[pos] = ent | (dd < 0 ? 0x80000000u : 0u);
            }
        }
    }
    if (!PLACE) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < 2 * BPG_MAT_NB; i += blockDim.x) counts[base + i] = scnt[i];
    }
}
// Two lanes per output, lane parity = set (0 low, 1 high): a plain running sum over the set's 128 buckets from the top,
// run = sum_{b' >= b} T_b', acc = sum_b run_b = sum_b b T_b: 2 x 127 + 1 additions, the same on every lane, so the warp
// never diverges (empty buckets hold the identity).  The high lane then doubles 8 times and the low lane adds it.
// (The earlier 32-lane layout per output -- 8-bucket segments, small multiples of the segment sums, a 16-lane tree and an
// 8-doubling tail on one lane -- issued ~2.3 x the lane-operations of this and ran 38 dependent point operations per
// warp; with 2^15 and more outputs per proof every lane has enough outputs to stay busy.)
__global__ void __launch_bounds__(64) k_mat_reduce(const ge *__restrict__ buckets, uint32_t nout, ge *__restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, o = t >> 1, set = t & 1u;
    const bool valid = o < nout; // (nout is even, so both lanes of a pair agree; the shuffle below needs the whole warp)
    ge run, acc, q;
    ge_identity(acc);
    if (valid) {
        const ge *B = buckets + ((size_t)2 * o + set) * BPG_MAT_NB;
        ld_ge(run, &B[BPG_MAT_NB - 1]);
        acc = run;
        ld_ge(q, &B[BPG_MAT_NB - 2]);
#pragma unroll 1
        for (uint32_t b = BPG_MAT_NB - 2; b >= 1; b--) {
            ge qn;
            ld_ge(qn, &B[b - 1]); // one bucket ahead (b - 1 = 0 is the set's unused digit-0 slot): the load overlaps the additions
            ge_add_ilp(run, run, q);
            ge_add_ilp(acc, acc, run);
            q = qn;
        }
        if (set) {
#pragma unroll 1
            for (int k = 0; k < 8; k++) ge_dbl_ilp(acc, acc);
        }
    }
    ge hi;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        hi.X.v[i] = __shfl_down_sync(0xFFFFFFFFu, acc.X.v[i], 1);
        hi.Y.v[i] = __shfl_down_sync(0xFFFFFFFFu, acc.Y.v[i], 1);
        hi.Z.v[i] = __shfl_down_sync(0xFFFFFFFFu, acc.Z.v[i], 1);
        hi.T.v[i] = __shfl_down_sync(0xFFFFFFFFu, acc.T.v[i], 1);
    }
    if (valid && !set) {
        ge_add_ilp(acc, acc, hi);
        st_ge(&out[o], acc);
    }
}
// Latency-lean reduction of the same 2 x 129 bucket layout for the few groups of a SMALL MSM (late IPP rounds: 2 groups,
// nothing else of this proof can run until L_j, R_j are known).  One 128-thread block per (group, set), thread = b - 1:
// b * T_b by a fixed 8-step double-and-add (uniform across the warp), block-wide tree; k_small_combine: low + 2^8 high.
// Depth ~ 16 + 8 + 9 point operations instead of ~ 55 in k_mat_reduce, at ~ 3x its work (irrelevant for 2 groups; the
// late-fold materialisation with its 1024 outputs keeps the work-lean kernel).
__global__ void __launch_bounds__(128) k_small_reduce(const ge *__restrict__ buckets, ge *__restrict__ part) {
    // grid = 2 * groups blocks of 128 threads: block (2 g + set) weights and sums the 128 buckets of one set.  One warp per
    // SM sub-partition: with both sets in one 256-thread block two warps shared each integer pipe and every step took 1.4 x longer.
    __shared__ ge smem[128];
    uint32_t gs = blockIdx.x, t = threadIdx.x, b = t + 1u;
    ge p, acc;
    ld_ge(p, &buckets[(size_t)gs * BPG_MAT_NB + b]);
    ge_identity(acc);
#pragma unroll 1
    for (int k = 7; k >= 0; k--) {
        ge_dbl_ilp(acc, acc);
        if ((b >> k) & 1u) ge_add_ilp(acc, acc, p);
    }
    st_ge(&smem[t], acc);
    __syncthreads();
    for (int s2 = 64; s2 > 0; s2 >>= 1) {
        if (t < (uint32_t)s2) {
            ge o;
            ld_ge(o, &smem[t + s2]);
            ge_add_ilp(acc, acc, o);
            st_ge(&smem[t], acc);
        }
        __syncthreads();
    }
    if (t == 0) st_ge(&part[gs], acc);
}
// out[g] = part[2 g] + 2^8 part[2 g + 1]
__global__ void __launch_bounds__(32) k_small_combine(const ge *__restrict__ part, uint32_t G, ge *__restrict__ out) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    ge lo, hi;
    ld_ge(lo, &part[2 * g]); ld_ge(hi, &part[2 * g + 1]);
#pragma unroll 1
    for (int k = 0; k < 8; k++) ge_dbl_ilp(hi, hi);
    ge_add_ilp(lo, lo, hi);
    st_ge(&out[g], lo);
}
// window chain of the materialised points: ext[w][q] = 2^(16 w) P_q  (one thread per point, 240 doublings)
__global__ void __launch_bounds__(64) k_mat_chain(const ge *__restrict__ pts, uint32_t npts, ge *__restrict__ ext) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= npts) return;
    ge p;
    ld_ge(p, &pts[q]);
#pragma unroll 1
    for (int w = 0; w < BPG_NWIN; w++) {
        st_ge(&ext[(size_t)w * npts + q], p);
        if (w + 1 < BPG_NWIN) {
#pragma unroll 1
            for (int k = 0; k < BPG_WBITS; k++) ge_dbl_ilp(p, p);
        }
    }
}
// affine-Niels table of the materialised points, plus the entries of one resident point (B) copied from the main table to
// index npts.  One thread per POINT: the 16 window multiples of a point share ONE field inversion (Montgomery's trick over
// their Z coordinates: 45 multiplications instead of 15 more inversions of ~265 each; round 1 inverted per entry -- 0.62 ms of
// integer-pipe work per 2^20 proof).
__global__ void __launch_bounds__(64) k_mat_affine(const ge *__restrict__ ext, uint32_t npts, uint32_t ptotal_small, ge_an *__restrict__ tab_small,
                                                    const ge_an *__restrict__ tab_main, uint32_t ptotal_main, uint32_t pB_main) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < npts) {
        fe pre[BPG_NWIN]; // pre[w] = Z_0 Z_1 ... Z_w
        ld_fe_nc(pre[0], &ext[q].Z);
#pragma unroll 1
        for (int w = 1; w < BPG_NWIN; w++) {
            fe z;
            ld_fe_nc(z, &ext[(size_t)w * npts + q].Z);
            fe_mul(pre[w], pre[w - 1], z);
        }
        fe inv;
        fe_invert(inv, pre[BPG_NWIN - 1]);
#pragma unroll 1
        for (int w = BPG_NWIN - 1; w >= 0; w--) {
            ge p;
            ld_ge(p, &ext[(size_t)w * npts + q]);
            fe zi;
            if (w) { fe_mul(zi, inv, pre[w - 1]); fe_mul(inv, inv, p.Z); } else zi = inv;
            fe x, y;
            fe_mul(x, p.X, zi);
            fe_mul(y, p.Y, zi);
            ge_an a;
            ge_affine_to_an(a, x, y);
            st_an(&tab_small[(size_t)w * ptotal_small + q], a);
        }
    } else if (q < npts + BPG_NWIN) {
        uint32_t w = q - npts;
        ge_an a;
        ld_an(a, &tab_main[(size_t)w * ptotal_main + pB_main]);
        st_an(&tab_small[(size_t)w * ptotal_small + npts], a);
    }
}
// out[k] = sum over ranks r of recv[r * K + k]   (partial results of a sharded MSM, gathered in rank order)
__global__ void __launch_bounds__(64) k_sum_ranks(const ge *__restrict__ recv, uint32_t K, uint32_t world, ge *__restrict__ out) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    ge acc, o;
    ld_ge(acc, &recv[k]);
#pragma unroll 1
    for (uint32_t r = 1; r < world; r++) { ld_ge(o, &recv[(size_t)r * K + k]); ge_add_ilp(acc, acc, o); }
    st_ge(&out[k], acc);
}
// ---- variable-base MSMs (bpg_msm, the verifier's own points): the same bucket engine with the 16 windows of a group as 16
// bucket groups (no tables, entry = the point itself); this kernel recombines them:  out[g] = sum_w 2^(16 w) S[16 g + w]
// (Horner from the top window: 240 doublings -- a fixed latency of every variable-base MSM; the points pay none).
__global__ void __launch_bounds__(32) k_msm_horner16(const ge *__restrict__ S, uint32_t G, ge *__restrict__ out) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    ge acc, t;
    ld_ge(acc, &S[16 * g + 15]);
#pragma unroll 1
    for (int w = 14; w >= 0; w--) {
#pragma unroll 1
        for (int k = 0; k < 16; k++) ge_dbl(acc, acc);
        ld_ge(t, &S[16 * g + w]);
        ge_add(acc, acc, t);
    }
    st_ge(&out[g], acc);
}
// ristretto255 decode -> affine Niels (the decoded point is affine: Z = 1, T = x y); ok &= every encoding was valid
__global__ void __launch_bounds__(128) k_decompress_an_kernel(const uint8_t *__restrict__ in32, uint32_t n, ge_an *__restrict__ out, uint32_t *ok) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t b[32];
    const uint4 *src = reinterpret_cast<const uint4 *>(in32 + 32ull * i);
    uint4 v0 = src[0], v1 = src[1];
    memcpy(b, &v0, 16); memcpy(b + 16, &v1, 16);
    ge p;
    if (!ristretto_decode(p, b)) { atomicAnd(ok, 0u); ge_identity(p); }
    ge_an a;
    ge_affine_to_an(a, p.X, p.Y);
    st_an(&out[i], a);
}
__global__ void __launch_bounds__(128) k_sc_fill_one(sc *__restrict__ v, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sc one;
    sc_set_u32(one, 1);
    st_sc(&v[i], one);
}
