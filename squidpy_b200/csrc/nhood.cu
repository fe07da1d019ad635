// nhood.cu — nhood_enrichment permutation test on B200 (sm_100a).
//
// Replaces the reference's per-permutation CPU loop (src/squidpy/gr/_nhood.py:516-547): for every permutation
//   shuffled = base.copy(); rng_p.shuffle(shuffled)        (numpy PCG64 Generator.shuffle, replayed bit-exactly)
//   perms[p] = count(indices, indptr, shuffled)            (_nenrich kernel, _nhood.py:54-141)
// with five kernels per chunk of permutations, all integer / byte work (HBM, L2 and shared-memory bound, no tensor
// cores):
//   1. nhood_fill          broadcast the base labels into one row per permutation            [P][stride]
//   2. nhood_jgen          one WARP per permutation replays the PCG64 stream (jump-ahead, one 64-bit output per lane
//                          and batch) and numpy's masked rejection sampling (ballots + prefix sums) and streams the
//                          Fisher-Yates target of every step to J[P][stride]
//      nhood_apply_list    one CTA per permutation applies the swaps in 2048-step windows: 2-bit duplicate filter,
//                          per-position lists instead of an ordered replay of conflicting swaps, low part of the array in
//                          shared memory, next window marked while the current one is resolved (sections 2c-2e)
//      nhood_shuffle_cta   replace the two kernels above for few permutations (one CTA each, 2a) or many permutations of
//      nhood_shuffle_warp  small arrays (one warp each, 2b): one kernel replays the stream and applies the swaps
//   3. nhood_transpose     [P][n] -> [PB/32][n + 1][32] (groups of 32 permutations, permutation-minor inside a group) so that
//                          one warp lane = one permutation and a CTA's labels of consecutive nodes are contiguous
//   4. nhood_count         CSR neighbour-pair histogram: lane = permutation, warp walks the CSR once for 32
//                          permutations; lane-private shared-memory histogram columns (bank = lane, no
//                          conflicts), one flush per CTA; symmetric graphs are walked over j >= i only (3b).
#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "pcg64_jump.h"

typedef unsigned __int128 u128;

// Block barriers (bar.sync / bar.red) are warp-ALIGNED instructions: every lane of a warp must execute them together.
// After data-dependent branches (hash probing, staging paths) the lanes are not guaranteed to have re-converged
// (compute-sanitizer synccheck: "Divergent thread(s) in warp" -> cudaErrorIllegalInstruction on sm_100), and the
// compiler elides a plain __syncwarp() it believes redundant, hence the volatile asm
// (and ptxas turns a `bar.warp.sync 0xffffffff` it considers redundant into a NOP, so the full mask is passed in
// at run time, as a kernel argument, which it cannot reason about).
#define SQB_CONVERGE() asm volatile("bar.warp.sync %0;" ::"r"(full_mask) : "memory")

__constant__ uint64_t c_jump_M[SQB_PCG_JUMP_BITS][2] = SQB_PCG_JUMP_M_INIT;
__constant__ uint64_t c_jump_C[SQB_PCG_JUMP_BITS][2] = SQB_PCG_JUMP_C_INIT;

// ------------------------------------------------------------------------------------------------
// numpy PCG64 (XSL-RR 128/64) on the device.  numpy/random/src/pcg64/pcg64.h: advance first, then output.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ u128 mk128(uint64_t hi, uint64_t lo) { return ((u128)hi << 64) | (u128)lo; }

__device__ __forceinline__ uint64_t pcg_output(u128 s) {
    uint64_t hi = (uint64_t)(s >> 64), lo = (uint64_t)s;
    uint64_t x = hi ^ lo;
    unsigned rot = (unsigned)(hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
}

// state_{k+d} = M * state_k + C * inc
__device__ __forceinline__ void pcg_jump_consts(uint64_t d, u128& M, u128& C) {
    M = 1;
    C = 0;
    for (int b = 0; d != 0; ++b, d >>= 1) {
        if (d & 1) {
            u128 Mb = mk128(c_jump_M[b][0], c_jump_M[b][1]);
            u128 Cb = mk128(c_jump_C[b][0], c_jump_C[b][1]);
            C = Mb * C + Cb;
            M = Mb * M;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// 1. fill: labels[p][0..stride) = base[0..stride)   (16-byte vectors; stride*sizeof(LT) % 16 == 0)
// ------------------------------------------------------------------------------------------------
__global__ void nhood_fill_kernel(uint4* __restrict__ dst, const uint4* __restrict__ base, int64_t vec_per_row,
                                  int64_t n_rows) {
    for (int64_t row = blockIdx.y; row < n_rows; row += gridDim.y) {
        uint4* __restrict__ d = dst + row * vec_per_row;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < vec_per_row;
             i += (int64_t)gridDim.x * blockDim.x)
            d[i] = base[i];
    }
}

// ------------------------------------------------------------------------------------------------
// 2a. CTA-parallel exact replay of numpy Generator.shuffle (see file header; validated step by step against
//     numpy by the Python emulation tests/emu_shuffle.py).
//
//  Raw stream: v_{2k} = lo32(out_k), v_{2k+1} = hi32(out_k)  (pcg64_next32 hands out the low half first).
//  Thread t owns out_{b*NT + t} of batch b (LCG jump-ahead by NT per batch), i.e. raw slots 2t, 2t+1.
//  A window of K raw values is examined at a time; value r is accepted for the current step iff
//      (v_r & mask) <= i_cur - (#accepted before r)
//  which is solved as a fixed point of ballots + prefix sums (converges in 1-2 rounds because
//  K <= min(i/4, 4 sqrt(i))).  The S accepted values are the swap targets j of steps i_cur, i_cur-1, ...
//  Swaps of one window commute unless they share a position; sharing is detected exactly (targets inside the
//  window's own index range; duplicate targets through a shared-memory hash table) and the few conflicting
//  swaps are replayed in step order by one thread on the staged copies.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int sqb_window_size(int64_t i_cur, int raw_left, int raw_total, float wfactor) {
    int64_t a = i_cur >> 2;
    int64_t b = (int64_t)(wfactor * sqrtf((float)i_cur));
    int64_t k = a < b ? a : b;
    if (k > raw_total) k = raw_total;
    if (k < 1) k = 1;
    if (k > raw_left) k = raw_left;
    return (int)k;
}

template <typename LT>
__device__ __forceinline__ LT ld_cg(const LT* p) {
    return __ldcg(p);
}
template <typename LT>
__device__ __forceinline__ LT ld_cs(const LT* p) {
    return __ldcs(p);
}
template <typename LT>
__device__ __forceinline__ void st_cs(LT* p, LT v) {
    __stcs(p, v);
}

// Start-up stagger (ns): unit u of U starts u/U * stagger_ns late, so that the persistent CTAs work on different
// phases of their Fisher-Yates replays.  The live part of a label array is [0, i]; with all permutations in lock step
// the combined working set swings between P MB and 0, with staggered phases it stays near P/2 MB, which is what
// lets ~150-250 label arrays stay resident in the 126 MB L2 instead of thrashing DRAM with 32-byte sectors.
__device__ __forceinline__ void sqb_stagger(uint64_t delay_ns) {
    if (delay_ns == 0) return;
    uint64_t t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    do {
        __nanosleep(4000);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    } while (t - t0 < delay_ns);
}

#define SQB_EMPTY64 0xFFFFFFFFFFFFFFFFULL

template <typename LT, int NT>
__global__ void __launch_bounds__(NT) nhood_shuffle_cta_kernel(LT* __restrict__ labels, int64_t stride,
                                                               const uint64_t* __restrict__ states, int64_t n_perms,
                                                               int nseg, const int64_t* __restrict__ seg_start,
                                                               const int64_t* __restrict__ seg_len, float wfactor,
                                                               uint32_t full_mask, uint64_t stagger_ns) {
    constexpr int RAW = 2 * NT;
    constexpr int HS = 4 * NT;  // hash slots (load factor <= 0.5)
    constexpr int NW = NT / 32;
    constexpr int HS_SHIFT = (NT == 128 ? 23 : NT == 256 ? 22 : NT == 512 ? 21 : 20);  // 32 - log2(HS)
    static_assert(NT == 128 || NT == 256 || NT == 512 || NT == 1024, "NT");

    extern __shared__ __align__(16) unsigned char sqb_shuffle_smem[];
    unsigned long long* s_tab = reinterpret_cast<unsigned long long*>(sqb_shuffle_smem);  // (target << 32) | owner step, or EMPTY
    uint32_t* s_sj = reinterpret_cast<uint32_t*>(s_tab + HS);
    uint32_t* s_flag = s_sj + RAW;
    int* s_wsum = reinterpret_cast<int*>(s_flag + RAW / 32);
    int& s_rstar = s_wsum[32];
    LT* s_own = reinterpret_cast<LT*>(s_wsum + 36);
    LT* s_hval = s_own + RAW;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;

    for (int h = tid; h < HS; h += NT) s_tab[h] = SQB_EMPTY64;
    if (tid < RAW / 32) s_flag[tid] = 0;
    if (tid < 32) s_wsum[tid] = 0;
    u128 Mn, Cn;
    pcg_jump_consts((uint64_t)NT, Mn, Cn);
    u128 Mt, Ct;
    pcg_jump_consts((uint64_t)tid + 1, Mt, Ct);
    sqb_stagger(stagger_ns * blockIdx.x / gridDim.x);
    __syncthreads();

    // persistent CTA: permutations blockIdx.x, blockIdx.x + gridDim.x, ...  (the grid size bounds how many label
    // arrays are live at once, i.e. the L2 working set)
    for (int64_t perm = blockIdx.x; perm < n_perms; perm += gridDim.x) {
        LT* __restrict__ a = labels + perm * stride;
        const uint64_t* st4 = states + perm * 4;
        // per-thread LCG: state of output index t is state_{t+1}
        const u128 inc = mk128(st4[2], st4[3]);
        u128 st = Mt * mk128(st4[0], st4[1]) + Ct * inc;
        const u128 Cn_inc = Cn * inc;
        uint32_t raw0 = 0, raw1 = 0;
        int pos = RAW;

        for (int seg = 0; seg < nseg; ++seg) {
            const int64_t base = seg_start[seg];
            int64_t i_cur = seg_len[seg] - 1;
            while (i_cur >= 1) {
                if (pos >= RAW) {
                    uint64_t o = pcg_output(st);
                    st = Mn * st + Cn_inc;
                    raw0 = (uint32_t)o;
                    raw1 = (uint32_t)(o >> 32);
                    pos = 0;
                }
                // ---- phase parameters (uniform) ----
                uint64_t mask64 = (uint64_t)i_cur;
                mask64 |= mask64 >> 1;
                mask64 |= mask64 >> 2;
                mask64 |= mask64 >> 4;
                mask64 |= mask64 >> 8;
                mask64 |= mask64 >> 16;
                mask64 |= mask64 >> 32;
                const uint32_t mask = (uint32_t)mask64;  // i_cur < 2^32 (n < 2^32 enforced on the host)
                const int64_t i_lo = (int64_t)(mask64 >> 1) + 1;
                const int64_t n_ph = i_cur - i_lo + 1;
                const int K = sqb_window_size(i_cur, RAW - pos, RAW, wfactor);
                const int r0 = 2 * tid, r1 = 2 * tid + 1;
                const bool in0 = (r0 >= pos) && (r0 < pos + K);
                const bool in1 = (r1 >= pos) && (r1 < pos + K);
                const uint32_t u0 = raw0 & mask, u1 = raw1 & mask;

                // ---- acceptance fixed point ----
                int c0 = 0, c1 = 0, total = 0;
                bool F0 = in0 && ((int64_t)u0 <= i_cur);
                bool F1 = in1 && ((int64_t)u1 <= i_cur);
                while (true) {
                    const uint32_t b0 = __ballot_sync(0xffffffffu, F0);
                    const uint32_t b1 = __ballot_sync(0xffffffffu, F1);
                    if (lane == 0) s_wsum[warp] = __popc(b0) + __popc(b1);
                    __syncthreads();
                    int v = (lane < NW) ? s_wsum[lane] : 0;
                    int incl = v;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        int t = __shfl_up_sync(0xffffffffu, incl, d);
                        if (lane >= d) incl += t;
                    }
                    const int woff = __shfl_sync(0xffffffffu, incl - v, warp);
                    total = __shfl_sync(0xffffffffu, incl, 31);
                    c0 = woff + __popc(b0 & lt_mask) + __popc(b1 & lt_mask);
                    c1 = c0 + (F0 ? 1 : 0);
                    const bool nF0 = in0 && ((int64_t)u0 <= i_cur - (int64_t)c0);
                    const bool nF1 = in1 && ((int64_t)u1 <= i_cur - (int64_t)c1);
                    const int changed = (nF0 != F0) || (nF1 != F1);
                    const int any = __syncthreads_or(changed);
                    if (!any) break;
                    F0 = nF0;
                    F1 = nF1;
                }
                int S;
                const bool phase_ends = ((int64_t)total >= n_ph);
                if (phase_ends) {
                    S = (int)n_ph;
                    if (F0 && c0 == S - 1) s_rstar = r0;
                    if (F1 && c1 == S - 1) s_rstar = r1;
                } else {
                    S = total;
                }
                if (F0 && c0 < S) s_sj[c0] = u0;
                if (F1 && c1 < S) s_sj[c1] = u1;
                __syncthreads();
                const int newpos = phase_ends ? (s_rstar + 1) : (pos + K);

                // ---- swap phase: steps s = 0..S-1, step s swaps positions (i_cur - s) and s_sj[s] ----
                if (S > 0) {
                    const int64_t own_lo = i_cur - (int64_t)S;  // targets j > own_lo lie inside the window's own range
                    int slot[2] = {-1, -1};
                    bool owner[2] = {false, false};
                    uint32_t jv[2] = {0, 0};
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const int s = tid + q * NT;
                        if (s < S) {
                            const uint32_t j = s_sj[s];
                            jv[q] = j;
                            if ((int64_t)j > own_lo) {
                                const int s2 = (int)(i_cur - (int64_t)j);
                                if (s2 != s) {
                                    atomicOr(&s_flag[s >> 5], 1u << (s & 31));
                                    atomicOr(&s_flag[s2 >> 5], 1u << (s2 & 31));
                                }
                            } else {
                                uint32_t h = (j * 2654435761u) >> HS_SHIFT;
                                const unsigned long long mine = ((unsigned long long)j << 32) | (unsigned)s;
                                while (true) {
                                    const unsigned long long prev = atomicCAS(&s_tab[h], SQB_EMPTY64, mine);
                                    if (prev == SQB_EMPTY64) {
                                        owner[q] = true;
                                        break;
                                    }
                                    if ((uint32_t)(prev >> 32) == j) {  // duplicate target: both steps conflict
                                        const int so = (int)(uint32_t)prev;
                                        atomicOr(&s_flag[s >> 5], 1u << (s & 31));
                                        atomicOr(&s_flag[so >> 5], 1u << (so & 31));
                                        break;
                                    }
                                    h = (h + 1) & (HS - 1);
                                }
                                slot[q] = (int)h;
                            }
                        }
                    }
                    // stage values: own range (coalesced, streaming) and distinct external targets (random, L2)
                    LT vo[2], vh[2];
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const int s = tid + q * NT;
                        vo[q] = (s < S) ? ld_cs<LT>(a + base + i_cur - s) : (LT)0;
                        vh[q] = owner[q] ? ld_cg<LT>(a + base + (int64_t)jv[q]) : (LT)0;
                    }
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const int s = tid + q * NT;
                        if (s < S) s_own[s] = vo[q];
                        if (owner[q]) s_hval[slot[q]] = vh[q];
                    }
                    SQB_CONVERGE();
                    __syncthreads();
                    // conflict-free swaps in parallel
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const int s = tid + q * NT;
                        if (s < S && slot[q] >= 0 && !((s_flag[s >> 5] >> (s & 31)) & 1u)) {
                            const LT t = s_own[s];
                            s_own[s] = s_hval[slot[q]];
                            s_hval[slot[q]] = t;
                        }
                    }
                    // conflicting swaps in step order (disjoint from the conflict-free set); warp 0 finds them with
                    // ballots, lane 0 replays them on the staged copies
                    if (warp == 0) {
                        const int nwords = (S + 31) >> 5;
                        for (int wb = 0; wb < nwords; wb += 32) {
                            const uint32_t myw = (wb + lane < nwords) ? s_flag[wb + lane] : 0u;
                            uint32_t nz = __ballot_sync(0xffffffffu, myw != 0u);
                            while (nz) {
                                const int wl = __ffs(nz) - 1;
                                nz &= nz - 1;
                                uint32_t bits = __shfl_sync(0xffffffffu, myw, wl);
                                if (lane == 0) {
                                    while (bits) {
                                        const int b = __ffs(bits) - 1;
                                        bits &= bits - 1;
                                        const int s = (wb + wl) * 32 + b;
                                        const uint32_t j = s_sj[s];
                                        const LT x = s_own[s];
                                        if ((int64_t)j > own_lo) {
                                            const int s2 = (int)(i_cur - (int64_t)j);
                                            const LT y = s_own[s2];
                                            s_own[s] = y;
                                            s_own[s2] = x;
                                        } else {
                                            uint32_t h = (j * 2654435761u) >> HS_SHIFT;
                                            while ((uint32_t)(s_tab[h] >> 32) != j) h = (h + 1) & (HS - 1);
                                            const LT y = s_hval[h];
                                            s_own[s] = y;
                                            s_hval[h] = x;
                                        }
                                    }
                                }
                            }
                        }
                    }
                    SQB_CONVERGE();
                    __syncthreads();
                    // write back + reset the tables for the next window
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const int s = tid + q * NT;
                        if (s < S) st_cs<LT>(a + base + i_cur - s, s_own[s]);  // final: never read again by this kernel
                        if (owner[q]) {
                            a[base + (int64_t)jv[q]] = s_hval[slot[q]];
                            s_tab[slot[q]] = SQB_EMPTY64;
                        }
                    }
                    if (tid < RAW / 32) s_flag[tid] = 0;
                    SQB_CONVERGE();
                    __syncthreads();
                }
                i_cur -= S;
                pos = newpos;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// 2b. WARP-per-permutation exact replay (the auto choice for many permutations of arrays under 65 536 elements).
//     Same algorithm as 2a, but every synchronisation is warp level (ballots, shuffles, __syncwarp): no block barriers
//     at all.  A lane owns Q consecutive-by-32 PCG64 outputs (2Q raw 32-bit values) per batch and executes the
//     Fisher-Yates steps of the values IT drew; the swaps act on global memory directly (L2): conflict-free steps in
//     parallel, conflicting ones (own-range targets, duplicate targets found through a per-warp shared-memory hash
//     table) afterwards by lane 0 in step order.
//     ~4 warp instructions per shuffle step instead of ~12 for the CTA version, and thousands of permutations in
//     flight per GPU, so the random label accesses of different permutations overlap.
// ------------------------------------------------------------------------------------------------
template <typename LT, int Q>
__global__ void __launch_bounds__(128) nhood_shuffle_warp_kernel(LT* __restrict__ labels, int64_t stride,
                                                                 const uint64_t* __restrict__ states, int64_t n_perms,
                                                                 int nseg, const int64_t* __restrict__ seg_start,
                                                                 const int64_t* __restrict__ seg_len, float wfactor,
                                                                 uint64_t stagger_ns) {
    constexpr int RAW = 64 * Q;   // raw 32-bit values per batch
    constexpr int HS = 256 * Q;   // hash slots per warp (load factor <= 0.25)
    constexpr int HS_SHIFT = (Q == 1 ? 24 : Q == 2 ? 23 : 22);
    static_assert(Q == 1 || Q == 2 || Q == 4, "Q");
    __shared__ unsigned long long s_tab_all[4][HS];
    __shared__ uint32_t s_sj_all[4][RAW];
    __shared__ uint32_t s_flag_all[4][2 * Q];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    unsigned long long* s_tab = s_tab_all[warp];
    uint32_t* s_sj = s_sj_all[warp];
    uint32_t* s_flag = s_flag_all[warp];
    for (int h = lane; h < HS; h += 32) s_tab[h] = SQB_EMPTY64;
    if (lane < 2 * Q) s_flag[lane] = 0;
    u128 M32, C32, Mt, Ct;
    pcg_jump_consts(32, M32, C32);
    pcg_jump_consts((uint64_t)lane + 1, Mt, Ct);
    __syncwarp();

    const int64_t warps_total = (int64_t)gridDim.x * 4;
    sqb_stagger(stagger_ns * (uint64_t)(blockIdx.x * 4 + warp) / (uint64_t)warps_total);
    __syncwarp();
    for (int64_t perm = (int64_t)blockIdx.x * 4 + warp; perm < n_perms; perm += warps_total) {
        LT* __restrict__ a = labels + perm * stride;
        const uint64_t* st4 = states + perm * 4;
        const u128 inc = mk128(st4[2], st4[3]);
        u128 st = Mt * mk128(st4[0], st4[1]) + Ct * inc;  // state of output index `lane`
        const u128 C32_inc = C32 * inc;
        uint32_t raw[2 * Q];
#pragma unroll
        for (int k = 0; k < 2 * Q; ++k) raw[k] = 0;
        int pos = RAW;

        for (int seg = 0; seg < nseg; ++seg) {
            const int64_t base = seg_start[seg];
            int i_cur = (int)(seg_len[seg] - 1);  // n < 2^31 enforced on the host for this kernel
            while (i_cur >= 1) {
                if (pos >= RAW) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) {  // outputs q*32 + lane of this batch
                        const uint64_t o = pcg_output(st);
                        st = M32 * st + C32_inc;
                        raw[2 * q] = (uint32_t)o;
                        raw[2 * q + 1] = (uint32_t)(o >> 32);
                    }
                    pos = 0;
                }
                // ---- phase parameters (warp uniform) ----
                const uint32_t mask = 0xFFFFFFFFu >> __clz(i_cur);
                const int i_lo = (int)(mask >> 1) + 1;
                const int n_ph = i_cur - i_lo + 1;
                const int K = sqb_window_size((int64_t)i_cur, RAW - pos, RAW, wfactor);
                // raw index of (q, h) on this lane: q*64 + 2*lane + h
                uint32_t u[2 * Q];
                bool inw[2 * Q], F[2 * Q];
                int c[2 * Q];
#pragma unroll
                for (int k = 0; k < 2 * Q; ++k) {
                    const int r = (k >> 1) * 64 + 2 * lane + (k & 1);
                    inw[k] = (r >= pos) && (r < pos + K);
                    u[k] = raw[k] & mask;
                    F[k] = inw[k] && (u[k] <= (uint32_t)i_cur);
                    c[k] = 0;
                }
                // ---- acceptance fixed point: (v_r & mask) <= i_cur - #accepted before r ----
                int total = 0;
                while (true) {
                    int run = 0;
#pragma unroll
                    for (int q = 0; q < Q; ++q) {
                        const uint32_t blo = __ballot_sync(0xffffffffu, F[2 * q]);
                        const uint32_t bhi = __ballot_sync(0xffffffffu, F[2 * q + 1]);
                        c[2 * q] = run + __popc(blo & lt_mask) + __popc(bhi & lt_mask);
                        c[2 * q + 1] = c[2 * q] + (F[2 * q] ? 1 : 0);
                        run += __popc(blo) + __popc(bhi);
                    }
                    total = run;
                    bool changed = false;
#pragma unroll
                    for (int k = 0; k < 2 * Q; ++k) {
                        const bool nf = inw[k] && ((int)u[k] <= i_cur - c[k]) && (u[k] <= (uint32_t)i_cur);
                        changed |= (nf != F[k]);
                        F[k] = nf;
                    }
                    if (!__any_sync(0xffffffffu, changed)) break;
                }
                int S, newpos;
                if (total >= n_ph) {  // the phase (same mask / same segment) ends inside this window
                    S = n_ph;
                    int myr = -1;
#pragma unroll
                    for (int k = 0; k < 2 * Q; ++k)
                        if (F[k] && c[k] == S - 1) myr = (k >> 1) * 64 + 2 * lane + (k & 1);
                    const uint32_t who = __ballot_sync(0xffffffffu, myr >= 0);
                    newpos = __shfl_sync(0xffffffffu, myr, __ffs(who) - 1) + 1;
                } else {
                    S = total;
                    newpos = pos + K;
                }
                if (S > 0) {
                    const int own_lo = i_cur - S;  // targets j > own_lo lie inside the window's own index range
                    bool act[2 * Q], ins[2 * Q];
                    int slot[2 * Q];
#pragma unroll
                    for (int k = 0; k < 2 * Q; ++k) {
                        act[k] = F[k] && c[k] < S;
                        ins[k] = false;
                        slot[k] = 0;
                        if (act[k]) {
                            const int s = c[k];
                            const uint32_t j = u[k];
                            s_sj[s] = j;
                            if ((int)j > own_lo) {
                                const int s2 = i_cur - (int)j;
                                if (s2 != s) {
                                    atomicOr(&s_flag[s >> 5], 1u << (s & 31));
                                    atomicOr(&s_flag[s2 >> 5], 1u << (s2 & 31));
                                } else {
                                    act[k] = false;  // self swap: nothing to do
                                }
                            } else {
                                uint32_t h = (j * 2654435761u) >> HS_SHIFT;
                                const unsigned long long mine = ((unsigned long long)j << 32) | (unsigned)s;
                                while (true) {
                                    const unsigned long long prev = atomicCAS(&s_tab[h], SQB_EMPTY64, mine);
                                    if (prev == SQB_EMPTY64) {
                                        ins[k] = true;
                                        slot[k] = (int)h;
                                        break;
                                    }
                                    if ((uint32_t)(prev >> 32) == j) {  // duplicate target: both steps conflict
                                        const int so = (int)(uint32_t)prev;
                                        atomicOr(&s_flag[s >> 5], 1u << (s & 31));
                                        atomicOr(&s_flag[so >> 5], 1u << (so & 31));
                                        break;
                                    }
                                    h = (h + 1) & (HS - 1);
                                }
                            }
                        }
                    }
                    __syncwarp();
                    // conflict-free swaps: loads first (memory-level parallelism), then stores
                    LT vi[2 * Q], vj[2 * Q];
#pragma unroll
                    for (int k = 0; k < 2 * Q; ++k) {
                        if (act[k]) act[k] = !((s_flag[c[k] >> 5] >> (c[k] & 31)) & 1u);
                        if (act[k]) {
                            vi[k] = ld_cs<LT>(a + base + (i_cur - c[k]));
                            vj[k] = ld_cg<LT>(a + base + (int64_t)u[k]);
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 2 * Q; ++k) {
                        if (act[k]) {
                            st_cs<LT>(a + base + (i_cur - c[k]), vj[k]);  // final: evict first
                            a[base + (int64_t)u[k]] = vi[k];
                        }
                    }
                    // conflicting swaps, in step order, straight on global memory (disjoint from the set above)
                    uint32_t fw = (lane < 2 * Q) ? s_flag[lane] : 0u;
                    uint32_t nz = __ballot_sync(0xffffffffu, fw != 0u);
                    if (nz) {
                        if (lane == 0) {
                            for (int w = 0; w < 2 * Q; ++w) {
                                uint32_t bits = s_flag[w];
                                while (bits) {
                                    const int b = __ffs(bits) - 1;
                                    bits &= bits - 1;
                                    const int s = w * 32 + b;
                                    const int64_t pi = base + (i_cur - s), pj = base + (int64_t)s_sj[s];
                                    const LT x = ld_cg<LT>(a + pi), y = ld_cg<LT>(a + pj);
                                    a[pi] = y;
                                    a[pj] = x;
                                }
                            }
                        }
                        __syncwarp();
                        if (lane < 2 * Q) s_flag[lane] = 0;
                    }
#pragma unroll
                    for (int k = 0; k < 2 * Q; ++k)
                        if (ins[k]) s_tab[slot[k]] = SQB_EMPTY64;
                    __syncwarp();  // orders this window's global stores before the next window's loads (same warp)
                }
                i_cur -= S;
                pos = newpos;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// 2c. List-based resolution of the conflicts inside a window of Fisher-Yates steps (used by the apply kernel, 2e).
//     Swaps of one window commute unless they share a position.  Instead of replaying the conflicting ones in step
//     order, every step pushes itself on the list of the position it targets (outside targets: shared-memory hash table
//     keyed by position; targets inside the window's own range: one list head per step).  With
//       T(s) = value of step s's top position just before step s
//            = T(latest earlier step targeting that top) or its ORIGINAL value,
//     step s writes a[top_s] = value of position j_s just before step s
//                            = T(latest earlier step targeting j_s) or the original a[j_s],
//     and the last step targeting an outside position p writes a[p] = T(that step).  Only original values are read, all
//     lists are immutable once built, so every step resolves independently (chains are almost always empty) and windows
//     can be several times larger than with an ordered replay (tests/emu_shuffle.py::resolve_window_lists is the
//     executable specification).
// ------------------------------------------------------------------------------------------------
#define SQB_NONE16 0xFFFFu
#define SQB_NONE32 0xFFFFFFFFu

template <typename LT>
__device__ __forceinline__ LT sqb_list_T(const uint32_t* __restrict__ s_ohead, const uint16_t* __restrict__ s_next,
                                         const LT* __restrict__ s_otop, int x) {
    // follow "latest earlier step targeting my top" until a step whose top nobody targeted before it
    while (true) {
        const uint32_t h = s_ohead[x];
        if (h == SQB_NONE32) break;
        int m = (int)h;
        for (uint32_t e = s_next[h]; e != SQB_NONE16; e = s_next[e]) m = max(m, (int)e);
        x = m;  // every element of the list of x is < x
    }
    return s_otop[x];
}

template <typename LT>
__device__ __forceinline__ LT sqb_list_T_own(const uint32_t* __restrict__ s_ohead, const uint16_t* __restrict__ s_next,
                                             const LT* __restrict__ s_otop, int s, LT own) {
    return (s_ohead[s] == SQB_NONE32) ? own : sqb_list_T<LT>(s_ohead, s_next, s_otop, s);
}

__device__ __forceinline__ int sqb_list_latest_before(const uint16_t* __restrict__ s_next, uint32_t head, int s, int* mx) {
    int best = -1, m = -1;
    for (uint32_t e = head; e != SQB_NONE16 && e != SQB_NONE32; e = s_next[e]) {
        const int ei = (int)e;
        m = max(m, ei);
        if (ei < s) best = max(best, ei);
    }
    *mx = m;
    return best;
}

// ------------------------------------------------------------------------------------------------
// 2d. Swap-target generation, the first half of the TWO-KERNEL replay (shuffle_algo 7).  ncu showed the one-kernel
//     replays (2a, 2b) to be bound by random DRAM row activations (1000 live 1 MB label arrays do not fit the 126 MB L2)
//     and, with fewer permutations in flight, by the dependent instruction chain RNG -> rejection -> swaps.  Splitting
//     the replay removes both:
//       nhood_jgen_kernel        one warp per permutation, ALL permutations in flight (pure ALU + ballots, no random
//                                memory traffic): replays PCG64 + masked rejection and streams the Fisher-Yates target
//                                of every step i to J[perm][i] (coalesced 4-byte stores, read once, evict-first);
//       nhood_apply_list_kernel  one CTA per permutation, few permutations in flight, applies the swaps (2e).
// ------------------------------------------------------------------------------------------------
template <int Q>
__global__ void __launch_bounds__(128) nhood_jgen_kernel(uint32_t* __restrict__ J, int64_t stride,
                                                         const uint64_t* __restrict__ states, int64_t n_perms, int nseg,
                                                         const int64_t* __restrict__ seg_start,
                                                         const int64_t* __restrict__ seg_len, float wfactor) {
    constexpr int RAW = 64 * Q;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    // Q independent LCG chains per lane (output q*32 + lane of every batch has its own state, advanced by 32*Q per batch)
    // instead of one chain stepped Q times: the 128-bit multiply-adds of a batch no longer depend on each other
    u128 M32, C32, MQ, CQ, Mt, Ct;
    pcg_jump_consts(32, M32, C32);
    pcg_jump_consts((uint64_t)32 * Q, MQ, CQ);
    pcg_jump_consts((uint64_t)lane + 1, Mt, Ct);
    const int wpb = (int)(blockDim.x >> 5);  // warps per block (1, 2 or 4)
    const int64_t warps_total = (int64_t)gridDim.x * wpb;
    for (int64_t perm = (int64_t)blockIdx.x * wpb + warp; perm < n_perms; perm += warps_total) {
        uint32_t* __restrict__ Jp = J + perm * stride;
        const uint64_t* st4 = states + perm * 4;
        const u128 inc = mk128(st4[2], st4[3]);
        u128 st[Q];
        st[0] = Mt * mk128(st4[0], st4[1]) + Ct * inc;
        const u128 C32_inc = C32 * inc;
        const u128 CQ_inc = CQ * inc;
#pragma unroll
        for (int q = 1; q < Q; ++q) st[q] = M32 * st[q - 1] + C32_inc;
        uint32_t raw[2 * Q];
#pragma unroll
        for (int k = 0; k < 2 * Q; ++k) raw[k] = 0;
        int pos = RAW;
        for (int seg = 0; seg < nseg; ++seg) {
            const int64_t base = seg_start[seg];
            int i_cur = (int)(seg_len[seg] - 1);
            while (i_cur >= 1) {
                if (pos >= RAW) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) {
                        const uint64_t o = pcg_output(st[q]);
                        st[q] = MQ * st[q] + CQ_inc;
                        raw[2 * q] = (uint32_t)o;
                        raw[2 * q + 1] = (uint32_t)(o >> 32);
                    }
                    pos = 0;
                }
                const uint32_t mask = 0xFFFFFFFFu >> __clz(i_cur);
                const int i_lo = (int)(mask >> 1) + 1;
                const int n_ph = i_cur - i_lo + 1;
                // no swaps here, hence no conflicts to bound: the window is the rest of the batch (capped at i/4, which keeps
                // the acceptance fixed point short at the small-i end); wfactor only matters to the kernels that swap
                int K = min(i_cur >> 2, RAW);
                K = min(max(K, 1), RAW - pos);
                (void)wfactor;
                uint32_t u[2 * Q];
                bool inw[2 * Q], F[2 * Q];
                int c[2 * Q];
#pragma unroll
                for (int k = 0; k < 2 * Q; ++k) {
                    const int r = (k >> 1) * 64 + 2 * lane + (k & 1);
                    inw[k] = (uint32_t)(r - pos) < (uint32_t)K;
                    u[k] = raw[k] & mask;
                    F[k] = inw[k] && (u[k] <= (uint32_t)i_cur);
                    c[k] = 0;
                }
                // A candidate (u <= i_cur) with u <= i_cur - K is accepted whatever its rank (rank < K).  Without any candidate
                // above that line in the whole window nothing depends on the ranks: one pass.  (Evaluated on the candidates,
                // not on the current flags: a value rejected in one round can come back in the next.)
                bool uncertain = false;
#pragma unroll
                for (int k = 0; k < 2 * Q; ++k) uncertain |= F[k] && ((int)u[k] > i_cur - K);
                const bool any_uncertain = __any_sync(0xffffffffu, uncertain);
                int total = 0;
                while (true) {
                    int run = 0;
#pragma unroll
                    for (int q = 0; q < Q; ++q) {
                        const uint32_t blo = __ballot_sync(0xffffffffu, F[2 * q]);
                        const uint32_t bhi = __ballot_sync(0xffffffffu, F[2 * q + 1]);
                        c[2 * q] = run + __popc(blo & lt_mask) + __popc(bhi & lt_mask);
                        c[2 * q + 1] = c[2 * q] + (F[2 * q] ? 1 : 0);
                        run += __popc(blo) + __popc(bhi);
                    }
                    total = run;
                    if (!any_uncertain) break;  // the optimistic flags, and the ranks just computed from them, are final
                    bool changed = false;
#pragma unroll
                    for (int k = 0; k < 2 * Q; ++k) {
                        const bool nf = inw[k] && ((int)u[k] <= i_cur - c[k]) && (u[k] <= (uint32_t)i_cur);
                        changed |= (nf != F[k]);
                        F[k] = nf;
                    }
                    if (!__any_sync(0xffffffffu, changed)) break;
                }
                int S, newpos;
                if (total >= n_ph) {
                    S = n_ph;
                    int myr = -1;
#pragma unroll
                    for (int k = 0; k < 2 * Q; ++k)
                        if (F[k] && c[k] == S - 1) myr = (k >> 1) * 64 + 2 * lane + (k & 1);
                    const uint32_t who = __ballot_sync(0xffffffffu, myr >= 0);
                    newpos = __shfl_sync(0xffffffffu, myr, __ffs(who) - 1) + 1;
                } else {
                    S = total;
                    newpos = pos + K;
                }
                // target of step i = i_cur - rank, streamed out (read exactly once by the apply kernel)
                uint32_t* __restrict__ Jtop = Jp + base + i_cur;
#pragma unroll
                for (int k = 0; k < 2 * Q; ++k)
                    if (F[k] && c[k] < S) __stcs(Jtop - c[k], u[k]);
                i_cur -= S;
                pos = newpos;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// 2e. TWO-KERNEL replay with list-based conflict resolution (shuffle_algo 7): nhood_jgen_kernel (2d, a warp per
//     permutation, warp-level synchronisation only) turns the PCG64 streams into the swap targets J[perm][i]; this kernel
//     applies them, one CTA per permutation, W = NT*SPT Fisher-Yates steps per window.  Few permutations are in flight:
//     measured on B200 (tools/micro/rmw_bench.cu), random byte swaps over label arrays that stay inside the 126 MB L2
//     run at ~55 G swaps/s, over 1000 arrays (1 GB) at ~20 G swaps/s, because every swap then costs two random 32-byte
//     DRAM sectors.  Step s of a window (top position i_cur - s) belongs to thread s % NT: the J values, the own range
//     and its write-back are fully coalesced, no ranks, ballots or acceptance barriers are left in this kernel, and
//     conflicts are resolved as in 2c (per-position lists, original values only, no ordered pass).  The next window's J
//     values are prefetched into registers.
//     ncu on the first version (every outside target inserted into the hash table): 43% of all instructions and most
//     short-scoreboard stalls were the dependent 64-bit CAS probe chains, and the barrier stalls (25%) their imbalance.
//     Duplicate targets are rare, so they are now FILTERED first: two bits per bucket (bucket = target mod 32W) in shared
//     memory, "seen" and "seen again", set with one atomicOr per step (independent across the steps of a thread).  After a
//     barrier a step whose bucket was not seen again is alone on its target: it writes the two values without touching
//     any list.  Only the steps of multiply-hit buckets (a few percent, false positives included) and the own-range
//     targets build lists.  Marking a window needs nothing but its targets, so window w+1 is marked while window w is
//     resolved: TWO barriers per window (lists complete -> resolve + mark next -> reset); filter, hash table, own-range
//     heads and links are double buffered (window parity) so that neither the overlap nor the reset needs a barrier.
// ------------------------------------------------------------------------------------------------
template <typename LT, int NT, int SPT>
__global__ void __launch_bounds__(NT, 1) nhood_apply_list_kernel(LT* __restrict__ labels, const uint32_t* __restrict__ J,
                                                                 int64_t stride, int64_t n_perms, int nseg,
                                                                 const int64_t* __restrict__ seg_start,
                                                                 const int64_t* __restrict__ seg_len, uint32_t full_mask,
                                                                 uint64_t stagger_ns, int low_cap) {
    // low_cap > 0: positions [0, min(low_cap, segment length)) of the current segment live in shared memory during the
    // replay.  The kernel is bound by the SM's rate of UNCOALESCED global requests (one random byte load and one random
    // byte store per step, ~1.8 cycles each, tools/micro/rmw_bench.cu); targets are uniform in [0, i], so a low part of
    // L elements takes (L + L ln(n/L)) / n of them (25% for L = n/16) off the LSU/L2 path.
    constexpr int W = NT * SPT;  // steps per window
    constexpr int HS = W;        // hash slots: only steps of multiply-hit buckets are inserted (<= W distinct keys always fit)
    constexpr int NWB = 2 * W;   // filter words (16 buckets of 2 bits each)
    constexpr int LOG_HS = (HS == 512 ? 9 : HS == 1024 ? 10 : HS == 2048 ? 11 : HS == 4096 ? 12 : HS == 8192 ? 13 : 14);
    static_assert(HS == (1 << LOG_HS), "HS must be a power of two");
    static_assert(W < 0xFFFF, "step indices are stored in 16 bits");
    constexpr int HS_SHIFT = 32 - LOG_HS;
    extern __shared__ __align__(16) unsigned char sqb_shuffle_smem[];
    // Everything a window's lists live in is DOUBLE BUFFERED by window parity: window w+1 is marked (filter bits, own-range
    // list pushes) while window w is still being resolved, and the entries of window w are reset after its last barrier,
    // ordered before their reuse by window w+2 through the barriers of window w+1.
    unsigned long long* s_tab0 = reinterpret_cast<unsigned long long*>(sqb_shuffle_smem);  // [2][HS] (target << 32) | list head
    uint32_t* s_bits0 = reinterpret_cast<uint32_t*>(s_tab0 + 2 * HS);                        // [2][NWB] duplicate filter
    uint32_t* s_ohead0 = s_bits0 + 2 * NWB;                                                  // [2][W] own-range list heads
    uint16_t* s_next0 = reinterpret_cast<uint16_t*>(s_ohead0 + 2 * W);                       // [2][W] list links
    LT* s_otop = reinterpret_cast<LT*>(s_next0 + 2 * W);                                     // [W] original own-range values
    LT* s_low = s_otop + W;                                                                  // [low_cap] low part of the segment
    const int tid = threadIdx.x;
    for (int h = tid; h < 2 * HS; h += NT) s_tab0[h] = SQB_EMPTY64;
    for (int w = tid; w < 2 * NWB; w += NT) s_bits0[w] = 0u;
    for (int w = tid; w < 2 * W; w += NT) s_ohead0[w] = SQB_NONE32;
    int par = 0;
    sqb_stagger(stagger_ns * blockIdx.x / gridDim.x);
    __syncthreads();

    // filter marking + own-range list pushes of one window (targets jm[], S_m steps from top i_m) into the tables of parity q
    auto mark = [&](const uint32_t (&jm)[SPT], int S_m, int i_m, int q) {
        uint32_t* bits = s_bits0 + q * NWB;
        uint32_t* ohead = s_ohead0 + q * W;
        uint16_t* next = s_next0 + q * W;
        const int lo_m = i_m - S_m;
        uint32_t old[SPT];
#pragma unroll
        for (int m = 0; m < SPT; ++m) {
            const int s = tid + m * NT;
            const bool out = (s < S_m) && !((int)jm[m] > lo_m);
            const uint32_t j = jm[m];
            old[m] = out ? atomicOr(&bits[(j >> 4) & (NWB - 1)], 1u << ((j & 15u) * 2u)) : 0u;
        }
#pragma unroll
        for (int m = 0; m < SPT; ++m) {
            const int s = tid + m * NT;
            const uint32_t j = jm[m];
            const bool ac = s < S_m;
            const bool ow = ac && ((int)j > lo_m);
            const uint32_t sh = (j & 15u) * 2u;
            if (ac && !ow && ((old[m] >> sh) & 1u)) atomicOr(&bits[(j >> 4) & (NWB - 1)], 2u << sh);  // seen again
            if (ow) {
                const int u = i_m - (int)j;  // u >= s
                if (u != s) {
                    const uint32_t prev = atomicExch(&ohead[u], (uint32_t)s);
                    next[s] = (uint16_t)prev;  // NONE32 truncates to NONE16
                }
            }
        }
    };

    for (int64_t perm = blockIdx.x; perm < n_perms; perm += gridDim.x) {
        LT* __restrict__ a = labels + perm * stride;
        const uint32_t* __restrict__ Jp = J + perm * stride;
        for (int seg = 0; seg < nseg; ++seg) {
            const int64_t base = seg_start[seg];
            int i_cur = (int)(seg_len[seg] - 1);  // n < 2^31
            const int Lc = min(low_cap, i_cur + 1);
            for (int x = tid; x < Lc; x += NT) s_low[x] = a[base + x];
            uint32_t jv[SPT], jn[SPT];  // targets of the current and of the next window
            {
                const int S0 = min(W, i_cur);
                const int i1 = i_cur - S0;
                const int S1 = min(W, i1);
#pragma unroll
                for (int m = 0; m < SPT; ++m) {
                    const int s = tid + m * NT;
                    const bool a0 = s < S0, a1 = s < S1;
                    jv[m] = a0 ? __ldcs(Jp + base + (i_cur - (a0 ? s : 0))) : 0u;
                    jn[m] = a1 ? __ldcs(Jp + base + (i1 - (a1 ? s : 0))) : 0u;
                }
                mark(jv, S0, i_cur, par);
            }
            SQB_CONVERGE();
            __syncthreads();
            while (i_cur >= 1) {
                const int S = min(W, i_cur);  // steps i_cur, i_cur-1, ..., i_cur-S+1 (>= 1)
                const int own_lo = i_cur - S;
                unsigned long long* s_tab = s_tab0 + par * HS;
                uint32_t* s_bits = s_bits0 + par * NWB;
                uint32_t* s_ohead = s_ohead0 + par * W;
                uint16_t* s_next = s_next0 + par * W;
                // original values: the global and the shared-memory (low part) copies are loaded into separate registers
                // and selected where they are USED, so that nothing waits for the global loads before the list phases
                LT vtg[SPT], vts[SPT], vjg[SPT], vjs[SPT];
                uint32_t act = 0, ownm = 0;  // bit m: step tid + m*NT exists / targets the window's own range
                uint32_t tgm = 0, jgm = 0;   // bit m: top / target of the step lives in global memory (not in the low part)
#pragma unroll
                for (int m = 0; m < SPT; ++m) {
                    const int s = tid + m * NT;
                    const bool ac = s < S;
                    const bool ow = ac && ((int)jv[m] > own_lo);
                    act |= (ac ? 1u : 0u) << m;
                    ownm |= (ow ? 1u : 0u) << m;
                    const int xt = i_cur - (ac ? s : 0);
                    const bool tg = ac && xt >= Lc;  // global / shared-memory copy of the position
                    vtg[m] = tg ? ld_cs<LT>(a + base + (tg ? xt : 0)) : (LT)0;
                    vts[m] = (ac && !tg) ? s_low[tg ? 0 : xt] : (LT)0;
                    const bool jo = ac && !ow;
                    const bool jg = jo && (int)jv[m] >= Lc;
                    vjg[m] = jg ? ld_cg<LT>(a + base + (int64_t)(jg ? jv[m] : 0u)) : (LT)0;
                    vjs[m] = (jo && !jg) ? s_low[jg ? 0u : (jo ? jv[m] : 0u)] : (LT)0;
                    tgm |= (tg ? 1u : 0u) << m;
                    jgm |= (jg ? 1u : 0u) << m;
                }
                // prefetch the targets of the window after the next one (same segment)
                const int i_nx = i_cur - S;
                const int S_nx = min(W, i_nx);
                uint32_t jnn[SPT];
                {
                    const int i_n2 = i_nx - max(S_nx, 0);
                    const int S_n2 = min(W, i_n2);
#pragma unroll
                    for (int m = 0; m < SPT; ++m) {
                        const int s = tid + m * NT;
                        const bool ac = s < S_n2;
                        jnn[m] = ac ? __ldcs(Jp + base + (i_n2 - (ac ? s : 0))) : 0u;
                    }
                }
                // ---- B: steps of multiply-hit buckets build per-target lists in the hash table (this window was marked
                //      during the previous one); stage the original own-range values ----
                uint32_t slowm = 0;
                uint32_t slotv[SPT];
#pragma unroll
                for (int m = 0; m < SPT; ++m) slotv[m] = 0;
#pragma unroll
                for (int m = 0; m < SPT; ++m) {
                    const int s = tid + m * NT;
                    const bool out = ((act >> m) & 1u) && !((ownm >> m) & 1u);
                    const uint32_t j = jv[m];
                    const uint32_t wbits = out ? s_bits[(j >> 4) & (NWB - 1)] : 0u;
                    if ((wbits >> ((j & 15u) * 2u + 1u)) & 1u) {
                        slowm |= 1u << m;
                        uint32_t h = (j * 2654435761u) >> HS_SHIFT;
                        const unsigned long long mine = ((unsigned long long)j << 32) | (unsigned)s;
                        uint32_t nxt = SQB_NONE16;
                        while (true) {
                            const unsigned long long prev = atomicCAS(&s_tab[h], SQB_EMPTY64, mine);
                            if (prev == SQB_EMPTY64) break;
                            if ((uint32_t)(prev >> 32) == j) {  // same target: push in front of the current head
                                if (atomicCAS(&s_tab[h], prev, mine) == prev) {
                                    nxt = (uint32_t)prev & 0xFFFFu;
                                    break;
                                }
                                continue;
                            }
                            h = (h + 1) & (HS - 1);
                        }
                        s_next[s] = (uint16_t)nxt;
                        slotv[m] = h;
                    }
                }
#pragma unroll
                for (int m = 0; m < SPT; ++m) {
                    const int s = tid + m * NT;
                    if ((act >> m) & 1u) s_otop[s] = ((tgm >> m) & 1u) ? vtg[m] : vts[m];
                }
                SQB_CONVERGE();
                __syncthreads();
                // ---- C: every step derives what it writes from the (now immutable) lists, original values only (2c) ----
#pragma unroll
                for (int m = 0; m < SPT; ++m) {
                    const int s = tid + m * NT;
                    if ((act >> m) & 1u) {
                        const uint32_t j = jv[m];
                        const LT vj = ((jgm >> m) & 1u) ? vjg[m] : vjs[m];
                        LT val;
                        if ((ownm >> m) & 1u) {
                            const int u = i_cur - (int)j;
                            if (u == s) {
                                val = sqb_list_T<LT>(s_ohead, s_next, s_otop, s);
                            } else {
                                int mx;
                                const int p = sqb_list_latest_before(s_next, s_ohead[u], s, &mx);
                                val = (p >= 0) ? sqb_list_T<LT>(s_ohead, s_next, s_otop, p) : s_otop[u];
                            }
                        } else {
                            bool last = true;  // the only (or the last) step of this window that touches position j
                            val = vj;
                            if ((slowm >> m) & 1u) {
                                const uint32_t head = (uint32_t)s_tab[slotv[m]] & 0xFFFFu;
                                int mx;
                                const int p = sqb_list_latest_before(s_next, head, s, &mx);
                                if (p >= 0) val = sqb_list_T<LT>(s_ohead, s_next, s_otop, p);
                                last = (mx == s);
                            }
                            if (last) {
                                const LT tv = sqb_list_T_own<LT>(s_ohead, s_next, s_otop, s, ((tgm >> m) & 1u) ? vtg[m] : vts[m]);
                                if ((int)j < Lc) s_low[j] = tv;
                                else a[base + (int64_t)j] = tv;
                            }
                        }
                        if (i_cur - s < Lc) s_low[i_cur - s] = val;
                        else st_cs<LT>(a + base + (i_cur - s), val);  // final position: never read again by this kernel
                    }
                }
                // ---- mark the next window in the other copy of the tables (needs nothing but its targets) ----
                mark(jn, S_nx, i_nx, par ^ 1);
                SQB_CONVERGE();
                __syncthreads();
                // ---- reset this window's copy of the tables (ordered before its reuse by the next window's barriers) ----
#pragma unroll
                for (int m = 0; m < SPT; ++m) {
                    const bool ac = (act >> m) & 1u, ow = (ownm >> m) & 1u, sl = (slowm >> m) & 1u;
                    const uint32_t j = jv[m];
                    if (ac && ow) s_ohead[i_cur - (int)j] = SQB_NONE32;
                    if (sl) s_tab[slotv[m]] = SQB_EMPTY64;
                }
                {  // the filter copy of this window only holds this window's marks: clear it wholesale (16-byte stores)
                    uint4* bz = reinterpret_cast<uint4*>(s_bits);
#pragma unroll
                    for (int x = tid; x < NWB / 4; x += NT) bz[x] = make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
                for (int m = 0; m < SPT; ++m) {
                    jv[m] = jn[m];
                    jn[m] = jnn[m];
                }
                i_cur = i_nx;
                par ^= 1;
            }
            __syncthreads();
            for (int x = tid; x < Lc; x += NT) a[base + x] = s_low[x];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// 3. transpose [P][stride] -> [PB/32][n + 1][32]  (32 permutations x 256 nodes per CTA), optional row scatter through
//    `order` (library-grouped position k -> original node id)
// ------------------------------------------------------------------------------------------------
template <typename LT>
__global__ void __launch_bounds__(256) nhood_transpose_kernel(const LT* __restrict__ lab, LT* __restrict__ labT, int64_t n,
                                                              int64_t stride, int P, int PB,
                                                              const uint32_t* __restrict__ order) {
    __shared__ LT tile[32][256 + 16 / sizeof(LT)];
    const int tx = threadIdx.x;
    const int64_t node = (int64_t)blockIdx.x * 256 + tx;
    const int pg = blockIdx.y * 32;
#pragma unroll 8
    for (int pp = 0; pp < 32; ++pp) {
        const int perm = pg + pp;
        tile[pp][tx] = (perm < P && node < n) ? lab[(int64_t)perm * stride + node] : (LT)0;
    }
    __syncthreads();
    if (node < n) {
        const int64_t row = order ? (int64_t)order[node] : node;
        constexpr int NV = (int)(32 * sizeof(LT) / 16);
        union {
            LT e[32];
            uint4 v[NV];
        } pack;
#pragma unroll
        for (int pp = 0; pp < 32; ++pp) pack.e[pp] = tile[pp][tx];
        uint4* dst = reinterpret_cast<uint4*>(labT + ((int64_t)(pg >> 5) * (n + 1) + row) * 32);  // group-major: [PB/32][n + 1][32]
#pragma unroll
        for (int k = 0; k < NV; ++k) dst[k] = pack.v[k];
    }
}

// ------------------------------------------------------------------------------------------------
// 2f. Fast RNG mode ("philox"): no replay of numpy's stream, no Fisher-Yates, no permutation-major label rows.
//     Permutation p of a segment of m labels is a KEYED BIJECTION pi_p on [0, m): a generalised Feistel network
//     (Black & Rogaway's FE2) on the mixed-radix domain [0, a) x [0, b), a = ceil(sqrt(m)), b = ceil(m / a), so that
//     a*b - m < a and cycle walking (re-encrypt while the value is >= m) practically never happens (m = 10^6: 1 value
//     in 1000);  x = L*b + R, six rounds alternate  L <- (L + mulhi(F(R ^ k_j), a)) mod a,
//     R <- (R + mulhi(F(L ^ k_j), b)) mod b  with the multiply-xorshift hash F and a Philox-style Weyl key schedule
//     k_j = k0 + j*k1, (k0, k1) = splitmix64(seed, global permutation index, segment).  The segment's labels are used
//     SORTED BY CLASS (cum[c] = number of labels below class c): the label of position r under permutation p is
//     class_of(pi_p(r)) = the last c with cum[c] <= pi_p(r), found through a shared-memory bucket table + a fixed
//     number of bisection steps instead of a random gather from a 1 MB array.  Shuffling the sorted vector has the same
//     distribution as shuffling the original.  One lane evaluates 4 consecutive permutations of one position (4
//     independent dependency chains) and stores 4 labels straight into the group-major matrix labT[PB/32][node][32] the
//     count kernel reads: fill + target generation + apply + transpose (21 of the 25 ms of the exact mode at 1M x 1000)
//     collapse into one streaming kernel.  tests/philox_ref.py is the executable specification (numpy, bit-identical);
//     results are validated statistically against the exact mode (SURVEY.md 8d).
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t sqb_philox_key(uint64_t seed, uint64_t perm, uint32_t seg, uint32_t which) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (perm + 1ull);
    z ^= (uint64_t)(seg * 2u + which + 1u) * 0xD1B54A32D192ED03ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (uint32_t)(z >> 32);
}

__device__ __forceinline__ uint32_t sqb_fe2_hash(uint32_t v) {
    v *= 0x9E3779B1u;
    v ^= v >> 15;
    v *= 0x85EBCA77u;
    return v;  // only the high bits are used (mulhi)
}

// one pass of the 6-round network over (L, R) in [0, a) x [0, b): every half is updated three times.  Four rounds are
// measurably too few (the same-class neighbour counts of a lattice come out 3.5 % high and twice as dispersed, caught by
// tests/test_gpu_philox.py::test_statistical_validation_against_exact_mode); six match numpy's shuffle in mean and variance.
__device__ __forceinline__ void sqb_fe2(uint32_t& L, uint32_t& R, uint32_t k0, uint32_t k1, uint32_t a, uint32_t b) {
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const uint32_t kj = k0 + (uint32_t)j * k1;
        if ((j & 1) == 0) {
            L += __umulhi(sqb_fe2_hash(R ^ kj), a);  // < 2a
            L = min(L, L - a);                       // mod a: L - a wraps to a huge value when L < a
        } else {
            R += __umulhi(sqb_fe2_hash(L ^ kj), b);
            R = min(R, R - b);
        }
    }
}

struct PhiloxSeg {
    int64_t start, len;   // segment in grouped order
    uint32_t a, b;        // Feistel radices
    int shift, tsize;     // bucket = value >> shift; table of tsize + 1 entries
    int steps;            // bisection steps after the bucket lookup
    int seg;
};

template <typename LT>
__global__ void __launch_bounds__(256) nhood_philox_labels_kernel(LT* __restrict__ labT, int PB, int64_t n_nodes, PhiloxSeg sg,
                                                                  const uint32_t* __restrict__ cum, int C,
                                                                  const uint32_t* __restrict__ bucket,
                                                                  const uint32_t* __restrict__ order, uint64_t seed, int64_t perm0,
                                                                  int64_t pos_per_cta) {
    extern __shared__ uint32_t s_tab[];  // [C + 1] class offsets, then [tsize + 1] class at the start of every bucket
    uint32_t* __restrict__ s_cum = s_tab;
    uint32_t* __restrict__ s_bkt = s_tab + (C + 1);
    for (int c = threadIdx.x; c <= C; c += blockDim.x) s_cum[c] = cum[c];
    for (int c = threadIdx.x; c <= sg.tsize; c += blockDim.x) s_bkt[c] = bucket[c];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int p4 = (blockIdx.y * 32 + lane) * 4;
    if (p4 >= PB) return;
    const uint32_t a = sg.a, b = sg.b, m = (uint32_t)sg.len;
    uint32_t k0[4], k1[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        k0[q] = sqb_philox_key(seed, (uint64_t)(perm0 + p4 + q), (uint32_t)sg.seg, 0u);
        k1[q] = sqb_philox_key(seed, (uint64_t)(perm0 + p4 + q), (uint32_t)sg.seg, 1u) | 1u;
    }
    int64_t r0 = (int64_t)blockIdx.x * pos_per_cta, r1 = r0 + pos_per_cta;
    if (r1 > sg.len) r1 = sg.len;
    for (int64_t r = r0 + warp; r < r1; r += nwarps) {
        const int64_t node = order ? (int64_t)order[sg.start + r] : sg.start + r;
        const uint32_t L0 = (uint32_t)r / b, R0 = (uint32_t)r - L0 * b;
        uint32_t y[4];
        bool walk = false;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t L = L0, R = R0;
            sqb_fe2(L, R, k0[q], k1[q], a, b);
            y[q] = L * b + R;
            walk |= y[q] >= m;
        }
        if (walk) {  // a*b - m < a values fall outside [0, m): rare
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                while (y[q] >= m) {
                    uint32_t L = y[q] / b, R = y[q] - L * b;
                    sqb_fe2(L, R, k0[q], k1[q], a, b);
                    y[q] = L * b + R;
                }
            }
        }
        uint32_t cls[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t bk = y[q] >> sg.shift;
            uint32_t lo = s_bkt[bk], hi = s_bkt[bk + 1];  // last class with cum <= first / last value of the bucket
            for (int s = 0; s < sg.steps; ++s) {           // invariant: cum[lo] <= y <  cum[hi + 1]
                const uint32_t mid = (lo + hi + 1u) >> 1;
                const bool le = s_cum[mid] <= y[q];
                lo = le ? mid : lo;
                hi = le ? hi : mid - 1u;
            }
            cls[q] = lo;
        }
        LT* dst = labT + ((int64_t)(p4 >> 5) * (n_nodes + 1) + node) * 32 + (p4 & 31);
        if (sizeof(LT) == 1) {
            *reinterpret_cast<uint32_t*>(dst) = cls[0] | (cls[1] << 8) | (cls[2] << 16) | (cls[3] << 24);
        } else {
            *reinterpret_cast<uint2*>(dst) = make_uint2(cls[0] | (cls[1] << 16), cls[2] | (cls[3] << 16));
        }
    }
}

// single label vector (uint32 from the host) -> column 0 of a [n][32] permutation-minor matrix
template <typename LT>
__global__ void nhood_single_to_T_kernel(const uint32_t* __restrict__ labels, LT* __restrict__ labT, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) labT[i * 32] = (LT)labels[i];
}

template <typename LT>
__global__ void nhood_u32_to_lt_kernel(const uint32_t* __restrict__ src, LT* __restrict__ dst, int64_t n, int64_t n_pad) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n_pad) dst[i] = (i < n) ? (LT)src[i] : (LT)0;
}

// ------------------------------------------------------------------------------------------------
// 3b. Symmetric graphs (what spatial_neighbors builds for grids and Delaunay graphs): when every stored entry (i -> j) has
//     exactly one mirror (j -> i) and no row holds a column twice, the count of all stored entries equals, per unordered
//     pair {i, j}: +1 on (l_i, l_j) and +1 on (l_j, l_i), and +1 on (l_i, l_i) per self loop.  The count kernel then walks
//     only the entries with j >= i: half the index and label loads for the same atomics.  The check and the upper CSR are
//     built once per graph on the device; anything else (kNN graphs, duplicates, rows longer than 64) keeps the full CSR.
// ------------------------------------------------------------------------------------------------
__global__ void nhood_symcheck_kernel(const uint32_t* __restrict__ indptr, const uint32_t* __restrict__ indices, int64_t n,
                                      uint32_t* __restrict__ flag, uint32_t* __restrict__ upper_cnt) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) {
        upper_cnt[n] = 0;
        return;
    }
    const uint32_t b = indptr[i], e = indptr[i + 1];
    if (e < b) {  // indptr not monotone: invalid CSR (flag bit 1), nothing else of this row is looked at
        upper_cnt[i] = 0;
        atomicOr(flag, 3u);
        return;
    }
    bool bad = (e - b > 64u);
    if (bad) {  // long row: no symmetric shortcut, but every column index is still validated
        bool oob = false;
        for (uint32_t k = b; k < e; ++k) oob |= ((int64_t)indices[k] >= n);
        if (oob) atomicOr(flag, 2u);
    }
    uint32_t up = 0;
    if (!bad) {
        for (uint32_t k = b; k < e; ++k) {
            const uint32_t j = indices[k];
            if ((int64_t)j >= n) {  // column index out of range (also what a negative int32 index looks like): invalid CSR
                atomicOr(flag, 2u);
                bad = true;
                break;
            }
            up += (j >= (uint32_t)i) ? 1u : 0u;
            for (uint32_t k2 = k + 1; k2 < e; ++k2) bad |= (indices[k2] == j);
            if (j != (uint32_t)i) {
                const uint32_t jb = indptr[j], je = indptr[j + 1];
                if (je < jb || je - jb > 64u) {
                    bad = true;
                } else {
                    uint32_t c = 0;
                    for (uint32_t t = jb; t < je; ++t) c += (indices[t] == (uint32_t)i) ? 1u : 0u;
                    bad |= (c != 1u);
                }
            }
        }
    }
    upper_cnt[i] = up;
    if (bad) atomicOr(flag, 1u);
}

__global__ void nhood_upper_fill_kernel(const uint32_t* __restrict__ indptr, const uint32_t* __restrict__ indices, int64_t n,
                                        const uint32_t* __restrict__ uptr, uint32_t* __restrict__ uidx) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w = uptr[i];
    for (uint32_t k = indptr[i]; k < indptr[i + 1]; ++k) {
        const uint32_t j = indices[k];
        if (j >= (uint32_t)i) uidx[w++] = j;
    }
}

// 3c. Row records for the count kernel: {i, j0, j1, j2} (16 bytes) = a row and up to three of its stored columns, unused
//     slots = n; a row with more entries continues in further records.  One 16-byte load then serves three
//     (pair x 32 permutations) units and the row label is fetched once per record.  Unused slots name node n: row n of every
//     group of the label matrix holds the label n_cls, whose histogram column is a spare that is never flushed -- the
//     kernel needs no predicate for them.  Built from the entries with j >= i of a
//     symmetric graph (self loops stay in: they are over-counted by one in the symmetrised flush and taken off again by
//     nhood_count_selfloops_kernel, which only runs for graphs that have any) or from all entries of any other graph.
__global__ void nhood_rec_count_kernel(const uint32_t* __restrict__ ptr, int64_t n, uint32_t* __restrict__ cnt) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i > n) return;
    cnt[i] = (i < n) ? (ptr[i + 1] - ptr[i] + 2u) / 3u : 0u;
}

__global__ void nhood_rec_fill_kernel(const uint32_t* __restrict__ ptr, const uint32_t* __restrict__ idx, int64_t n,
                                      const uint32_t* __restrict__ rptr, uint4* __restrict__ recs, uint32_t* __restrict__ n_self) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t b = ptr[i], e = ptr[i + 1];
    uint32_t w = rptr[i], self = 0;
    for (uint32_t k = b; k < e; k += 3) {
        uint4 r = make_uint4((uint32_t)i, idx[k], (uint32_t)n, (uint32_t)n);  // unused slot = the spare row n of the label matrix
        if (k + 1 < e) r.z = idx[k + 1];
        if (k + 2 < e) r.w = idx[k + 2];
        self += (r.y == (uint32_t)i) + (r.z == (uint32_t)i) + (r.w == (uint32_t)i);
        recs[w++] = r;
    }
    if (self) atomicAdd(n_self, self);
}

__global__ void nhood_self_fill_kernel(const uint32_t* __restrict__ uptr, const uint32_t* __restrict__ uidx, int64_t n,
                                       uint32_t* __restrict__ selfnodes, uint32_t* __restrict__ cursor) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (uint32_t k = uptr[i]; k < uptr[i + 1]; ++k)
        if (uidx[k] == (uint32_t)i) selfnodes[atomicAdd(cursor, 1u)] = (uint32_t)i;  // order is irrelevant (integer adds)
}

// ------------------------------------------------------------------------------------------------
// 4. count: hist[(a*C+b)*G + perm_in_group] over the nodes of this CTA's chunk.
//    G = permutations per CTA; lane = (edge slot = lane / G, perm = lane % G).  With G = 32 every lane owns
//    its own histogram column (bank == lane): shared-memory atomics never conflict inside a warp.
// ------------------------------------------------------------------------------------------------
template <typename LT, int G, int UNROWS = 8>
__global__ void __launch_bounds__(1024) nhood_count_kernel(const uint32_t* __restrict__ indptr, const uint32_t* __restrict__ indices,
                                                           const LT* __restrict__ labT, int PB, int64_t n, int C,
                                                           int64_t nodes_per_cta, int P, uint32_t* __restrict__ counts) {
    extern __shared__ uint32_t hist[];
    const int nb = C * C * G;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int64_t node_begin = (int64_t)blockIdx.x * nodes_per_cta;
    int64_t node_end = node_begin + nodes_per_cta;
    if (node_end > n) node_end = n;

    if (G == 32) {
        // lane = permutation; a warp walks UN consecutive CSR rows at once so that UN independent index loads, then UN
        // independent label gathers (one 32-byte sector each) are in flight before the UN shared-memory atomics:
        // ~7 instructions per (edge x 32 permutations), memory-level parallelism UN per warp.
        constexpr int UN = UNROWS;
        const int perm = blockIdx.y * 32 + lane;
        const LT* __restrict__ col = labT + (int64_t)blockIdx.y * (n + 1) * 32 + lane;  // group-major label matrix [PB/32][n + 1][32]
        // all element offsets are 32 x 32 -> 64 bit products (one IMAD.WIDE.U32 each): n < 2^31
        const uint32_t PBu = 32u, Cu = (uint32_t)C;
        (void)perm;
        const uint32_t nb32 = (uint32_t)node_begin, ne32 = (uint32_t)node_end;
        uint32_t* __restrict__ myhist = hist + lane;
        for (uint32_t i0 = nb32 + (uint32_t)warp * UN; i0 < ne32; i0 += (uint32_t)nwarps * UN) {
            uint32_t beg[UN], deg[UN], rowb[UN];
            uint32_t maxdeg = 0, mindeg = 0xFFFFFFFFu;
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const uint32_t i = i0 + u;
                beg[u] = 0;
                deg[u] = 0;
                rowb[u] = 0;
                if (i < ne32) {
                    beg[u] = indptr[i];
                    deg[u] = indptr[i + 1] - beg[u];
                    rowb[u] = (uint32_t)col[(uint64_t)i * PBu] * Cu;
                }
                maxdeg = deg[u] > maxdeg ? deg[u] : maxdeg;
                mindeg = deg[u] < mindeg ? deg[u] : mindeg;
            }
            // rows of a spatial graph have (nearly) equal degree: unpredicated fast path up to the smallest degree,
            // predicated tail for the rest.  Lanes of padded permutations (perm >= P) count into columns nobody reads.
            uint32_t k = 0;
            for (; k < mindeg; ++k) {
                uint32_t j[UN], bl[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) j[u] = indices[beg[u] + k];
#pragma unroll
                for (int u = 0; u < UN; ++u) bl[u] = (uint32_t)col[(uint64_t)j[u] * PBu];
#pragma unroll
                for (int u = 0; u < UN; ++u) atomicAdd(myhist + (rowb[u] + bl[u]) * 32u, 1u);
            }
            for (; k < maxdeg; ++k) {
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    if (k < deg[u]) {
                        const uint32_t j = indices[beg[u] + k];
                        const uint32_t bl = (uint32_t)col[(uint64_t)j * PBu];
                        atomicAdd(myhist + (rowb[u] + bl) * 32u, 1u);
                    }
                }
            }
        }
    } else {
        constexpr int EPW = 32 / G;
        const int sub = lane / G, pl = lane % G;
        const int perm = blockIdx.y * G + pl;
        const bool valid = perm < P;
        const LT* __restrict__ col = labT + (int64_t)(perm >> 5) * (n + 1) * 32 + (perm & 31);  // padded columns exist up to PB
        for (int64_t i = node_begin + warp; i < node_end; i += nwarps) {
            const uint32_t beg = indptr[i], end = indptr[i + 1];
            const uint32_t a = (uint32_t)col[i * 32];
            const uint32_t rowbase = a * (uint32_t)C;
#pragma unroll 4
            for (uint32_t e = beg + sub; e < end; e += EPW) {
                const uint32_t j = indices[e];
                const uint32_t b = (uint32_t)col[(int64_t)j * 32];
                if (valid) atomicAdd(&hist[(rowbase + b) * G + pl], 1u);
            }
        }
    }
    __syncthreads();
    const int CC = C * C;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) {
        const uint32_t v = hist[i];
        const int p = blockIdx.y * G + (i % G);
        if (v != 0 && p < P) atomicAdd(&counts[(int64_t)p * CC + (i / G)], v);
    }
}

// ------------------------------------------------------------------------------------------------
// 4b. count from the row records (3c).  Directed graphs: one increment (l_i, l_j) per stored entry (MIRROR = false).
//     Structurally symmetric graphs (MIRROR = true): per unordered pair {i, j} the full count is +1 on (l_i, l_j) and +1 on
//     (l_j, l_i): the kernel makes ONE increment, U[l_i][l_j], per stored entry with j >= i and adds the mirror when the
//     histogram is flushed (counts += U + U^T; a self loop lands twice on the diagonal and is taken off once by
//     nhood_count_selfloops_kernel).  lane = permutation, every lane owns its histogram column (bank == lane): the
//     shared-memory reductions of a warp never conflict.
//     What bounds it (tools/micro/smem_bench.cu, ncu): the SM's single load/store pipe takes ~1.85 cycles per warp
//     instruction, global load or shared-memory reduction alike -- not the reduction itself (1.87 cycles) and not DRAM.  So the
//     kernel minimises LSU instructions per (entry x 32 permutations): one 16-byte record load per three entries, the row
//     label once per record, one label load and one reduction per entry = 2.67 (CSR-row kernel of rounds 1-2: 2 reductions,
//     1.3 label loads and an index load per entry + a branch, 21 instructions, 4.2 ms at 1M spots x 1000 permutations;
//     flat (i, j) pairs: 3.5).  A warp takes UN records per pass, software-pipelined three deep: while the reductions of
//     group k issue, the label loads of group k+1 and the record loads of group k+2 are in flight (one CTA of 32 warps per
//     SM: without the pipeline 67% of the stall samples were label addresses waiting for the index load).
// ------------------------------------------------------------------------------------------------
// label load straight into a 32-bit register (ld.u8 / ld.u16 zero-extend: no cvt + mask after the load); the address is one
// 32 x 32 + 64 bit multiply-add (node_bytes is kept opaque by the caller so that it is not strength-reduced into two shifts)
template <typename LT>
__device__ __forceinline__ uint32_t sqb_ld_label_u32(unsigned long long base, uint32_t node, uint32_t node_bytes);
template <>
__device__ __forceinline__ uint32_t sqb_ld_label_u32<uint8_t>(unsigned long long base, uint32_t node, uint32_t node_bytes) {
    uint32_t v;
    asm volatile("{\n .reg .u64 a;\n mad.wide.u32 a, %1, %3, %2;\n ld.global.nc.u8 %0, [a];\n}" : "=r"(v) : "r"(node), "l"(base), "r"(node_bytes));
    return v;
}
template <>
__device__ __forceinline__ uint32_t sqb_ld_label_u32<uint16_t>(unsigned long long base, uint32_t node, uint32_t node_bytes) {
    uint32_t v;
    asm volatile("{\n .reg .u64 a;\n mad.wide.u32 a, %1, %3, %2;\n ld.global.nc.u16 %0, [a];\n}" : "=r"(v) : "r"(node), "l"(base), "r"(node_bytes));
    return v;
}
// one reduction on this lane's counter of bin (l_i, l_j): rowaddr = l_i * bytes per histogram row + the lane's column.  The
// histogram rows have C + 1 columns: unused record slots name the spare row of the label matrix, carry the label C and land
// in the spare column, which is never flushed -- no predicate anywhere (ptxas wraps a predicated ATOMS into a four-instruction
// convergence region).
__device__ __forceinline__ void sqb_hist_inc(uint32_t rowaddr, uint32_t lb) {
    asm volatile("{\n .reg .u32 a;\n mad.lo.u32 a, %1, 128, %0;\n red.shared.add.u32 [a], 1;\n}" ::"r"(rowaddr), "r"(lb));
}

template <typename LT, int UN, bool MIRROR>
__global__ void __launch_bounds__(1024) nhood_count_recs_kernel(const uint4* __restrict__ recs, int64_t n_recs,
                                                                const LT* __restrict__ labT, int64_t n, int C,
                                                                int64_t recs_per_cta, int P, uint32_t* __restrict__ counts) {
    extern __shared__ __align__(16) uint32_t hist[];
    const int C1 = C + 1;  // one spare column per histogram row (see sqb_hist_inc)
    const int nb = C * C1 * 32;
    {
        uint4* hz = reinterpret_cast<uint4*>(hist);
        for (int i = threadIdx.x; i < nb / 4; i += blockDim.x) hz[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    // lanes of padded permutations (blockIdx.y * 32 + lane >= P) count into columns nobody reads
    unsigned long long colp = reinterpret_cast<unsigned long long>(labT + (int64_t)blockIdx.y * (n + 1) * 32 + lane);  // [PB/32][n + 1][32]
    asm volatile("" : "+l"(colp));  // opaque: every label address stays ONE 32x32+64 multiply-add
    uint32_t NB = 32u * (uint32_t)sizeof(LT);  // bytes between the labels of consecutive nodes
    asm volatile("" : "+r"(NB));
    const uint32_t hbase = (uint32_t)__cvta_generic_to_shared(hist) + (uint32_t)lane * 4u;  // byte address of this lane's column
    const uint32_t rowmul = (uint32_t)C1 * 128u;                                           // bytes per histogram row ((C + 1) bins x 32 lanes)
    const int64_t r_begin = (int64_t)blockIdx.x * recs_per_cta;
    int64_t r_end = r_begin + recs_per_cta;
    if (r_end > n_recs) r_end = n_recs;
    const int64_t r_full = r_begin + ((r_end - r_begin) / UN) * UN;  // whole groups of UN records
    const int64_t step = (int64_t)nwarps * UN;
    const int64_t r_first = r_begin + (int64_t)warp * UN;
    const int n_it = r_first < r_full ? (int)((r_full - 1 - r_first) / step) + 1 : 0;  // groups of this warp
    const uint4* __restrict__ pp = recs + r_first;                                     // the group being fetched
    uint4 rc[UN];
    uint32_t la[UN], lb[UN][3];
    auto ld_recs = [&]() {
#pragma unroll
        for (int u = 0; u < UN; ++u)  // streamed once: keep the records out of L1, which holds the label sectors
            asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(rc[u].x), "=r"(rc[u].y), "=r"(rc[u].z), "=r"(rc[u].w)
                         : "l"(pp + u));
        pp += step;
    };
    auto ld_labels = [&](uint32_t(&xa)[UN], uint32_t(&xb)[UN][3]) {
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            xa[u] = sqb_ld_label_u32<LT>(colp, rc[u].x, NB);
            xb[u][0] = sqb_ld_label_u32<LT>(colp, rc[u].y, NB);
            xb[u][1] = sqb_ld_label_u32<LT>(colp, rc[u].z, NB);
            xb[u][2] = sqb_ld_label_u32<LT>(colp, rc[u].w, NB);
        }
    };
    auto reduce = [&](const uint32_t(&xa)[UN], const uint32_t(&xb)[UN][3]) {
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            const uint32_t rowaddr = xa[u] * rowmul + hbase;
            sqb_hist_inc(rowaddr, xb[u][0]);
            sqb_hist_inc(rowaddr, xb[u][1]);
            sqb_hist_inc(rowaddr, xb[u][2]);
        }
    };
    if (n_it > 0) {
        ld_recs();
        ld_labels(la, lb);
        if (n_it > 1) ld_recs();
        // steady state: all three stages are live; unrolled by two so that the label registers of consecutive groups swap
        // roles instead of being copied
#pragma unroll 2
        for (int k = 0; k < n_it - 2; ++k) {
            uint32_t na[UN], nb2[UN][3];
            ld_labels(na, nb2);  // group k+1
            ld_recs();           // group k+2
            reduce(la, lb);      // group k
#pragma unroll
            for (int u = 0; u < UN; ++u) la[u] = na[u], lb[u][0] = nb2[u][0], lb[u][1] = nb2[u][1], lb[u][2] = nb2[u][2];
        }
        if (n_it > 1) {
            uint32_t na[UN], nb2[UN][3];
            ld_labels(na, nb2);
            reduce(la, lb);
#pragma unroll
            for (int u = 0; u < UN; ++u) la[u] = na[u], lb[u][0] = nb2[u][0], lb[u][1] = nb2[u][1], lb[u][2] = nb2[u][2];
        }
        reduce(la, lb);
    }
    for (int64_t r = r_full + warp; r < r_end; r += nwarps) {  // fewer than UN records are left
        const uint4 v = __ldg(recs + r);
        const uint32_t rowaddr = sqb_ld_label_u32<LT>(colp, v.x, NB) * rowmul + hbase;
        sqb_hist_inc(rowaddr, sqb_ld_label_u32<LT>(colp, v.y, NB));
        sqb_hist_inc(rowaddr, sqb_ld_label_u32<LT>(colp, v.z, NB));
        sqb_hist_inc(rowaddr, sqb_ld_label_u32<LT>(colp, v.w, NB));
    }
    __syncthreads();
    const int CC = C * C;
    for (int i = threadIdx.x; i < CC * 32; i += blockDim.x) {
        const int bin = i >> 5, l = i & 31;
        const int a = bin / C, b = bin - a * C;
        const uint32_t v = MIRROR ? hist[((a * C1 + b) << 5) + l] + hist[((b * C1 + a) << 5) + l] : hist[((a * C1 + b) << 5) + l];  // U[a][b] + U[b][a]
        const int p = blockIdx.y * 32 + l;
        if (v != 0 && p < P) atomicAdd(&counts[(int64_t)p * CC + bin], v);
    }
}

// row n of every group of the label matrix = label n_cls ("no node": the unused slots of the row records point here)
template <typename LT>
__global__ void nhood_spare_row_kernel(LT* __restrict__ labT, int64_t n, int PB, int C) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < PB) labT[((int64_t)(p >> 5) * (n + 1) + n) * 32 + (p & 31)] = (LT)C;
}

// a self loop (i, i) is ONE stored entry: +1 on (l_i, l_i); the symmetrised flush above gave it 2
template <typename LT>
__global__ void nhood_count_selfloops_kernel(const uint32_t* __restrict__ selfnodes, uint32_t n_self, const LT* __restrict__ labT,
                                             int64_t n, int C, int P, uint32_t* __restrict__ counts) {
    const int p = blockIdx.y * blockDim.x + threadIdx.x;
    if (p >= P) return;
    for (uint32_t k = blockIdx.x; k < n_self; k += gridDim.x) {
        const uint32_t a = (uint32_t)labT[((int64_t)(p >> 5) * (n + 1) + selfnodes[k]) * 32 + (p & 31)];
        atomicAdd(&counts[(int64_t)p * C * C + a * C + a], 0xFFFFFFFFu);  // -1 (mod 2^32)
    }
}

// observed count (ONE label vector, uint32 as handed over by the host): a warp per CSR row, per-CTA C x C histogram in shared
// memory (global atomics when it does not fit).  The batched kernel above would zero and flush 32 histogram columns per CTA
// for a single permutation (13 ms at 1M spots); this one takes ~0.1 ms.
__global__ void __launch_bounds__(256) nhood_count_single_kernel(const uint32_t* __restrict__ indptr, const uint32_t* __restrict__ indices,
                                                                 const uint32_t* __restrict__ labels, int64_t n, int C, int hist_smem,
                                                                 uint32_t* __restrict__ counts) {
    extern __shared__ uint32_t hist[];
    const int CC = C * C;
    if (hist_smem) {
        for (int i = threadIdx.x; i < CC; i += blockDim.x) hist[i] = 0;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        const uint32_t b = indptr[i], e = indptr[i + 1];
        const uint32_t ra = labels[i] * (uint32_t)C;
        for (uint32_t k = b + lane; k < e; k += 32) {
            const uint32_t bin = ra + labels[indices[k]];
            if (hist_smem)
                atomicAdd(&hist[bin], 1u);
            else
                atomicAdd(&counts[bin], 1u);
        }
    }
    if (!hist_smem) return;
    __syncthreads();
    for (int i = threadIdx.x; i < CC; i += blockDim.x) {
        const uint32_t v = hist[i];
        if (v) atomicAdd(&counts[i], v);
    }
}

// fallback for very large n_cls: global atomics, lane = permutation
template <typename LT>
__global__ void nhood_count_global_kernel(const uint32_t* __restrict__ indptr, const uint32_t* __restrict__ indices,
                                          const LT* __restrict__ labT, int PB, int64_t n, int C, int64_t nodes_per_cta,
                                          int P, uint32_t* __restrict__ counts) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int perm = blockIdx.y * 32 + lane;
    const bool valid = perm < P;
    const int64_t node_begin = (int64_t)blockIdx.x * nodes_per_cta;
    int64_t node_end = node_begin + nodes_per_cta;
    if (node_end > n) node_end = n;
    const LT* __restrict__ col = labT + (int64_t)blockIdx.y * (n + 1) * 32 + lane;  // group-major label matrix [PB/32][n + 1][32]
    const int64_t CC = (int64_t)C * C;
    for (int64_t i = node_begin + warp; i < node_end; i += nwarps) {
        const uint32_t beg = indptr[i], end = indptr[i + 1];
        const uint32_t a = (uint32_t)col[i * 32];
        for (uint32_t e = beg; e < end; ++e) {
            const uint32_t b = (uint32_t)col[(int64_t)indices[e] * 32];
            if (valid) atomicAdd(&counts[(int64_t)perm * CC + (int64_t)a * C + b], 1u);
        }
    }
}

// ================================================================================================
// host side
// ================================================================================================
struct sqb_nhood {
    sqb_ctx* ctx = nullptr;
    int64_t n = 0, nnz = 0, stride = 0;
    int n_cls = 0;
    int lt_bytes = 1;  // 1: uint8 labels (n_cls <= 256), 2: uint16
    DevBuf<uint32_t> d_indptr, d_indices;
    DevBuf<uint32_t> d_uptr, d_uidx;  // entries with j >= i of a symmetric graph (see 3b): only while the pair list is built
    DevBuf<uint4> d_recs;              // row records (3c) of those entries (symmetric graph) or of all entries: what the count kernel walks
    DevBuf<uint32_t> d_selfnodes;      // nodes with a stored self loop (usually none)
    int64_t n_recs = 0;
    uint32_t n_self = 0;
    bool sym = false;
    int count_sym = -1;  // -1 auto (use the upper CSR when the graph is symmetric), 0 = always the full CSR
    int jgen_threads = 128;  // block size of the swap-target generation kernel (32 / 64 / 128: 1 / 2 / 4 permutations per block)
    int count_un = 4;    // records (of three entries) a warp takes per pass in the count kernel (1 / 2 / 3 / 4)
    DevBuf<uint8_t> d_base;   // stride * lt_bytes, library-grouped order
    DevBuf<uint32_t> d_order;  // grouped position -> node id (only with libraries)
    bool has_order = false;
    DevBuf<int64_t> d_seg_start, d_seg_len;
    int nseg = 0;
    bool base_set = false;
    DevBuf<uint64_t> d_states;  // P x 4
    int64_t n_perms = 0;
    bool uploaded = false, ran = false;
    int64_t chunk = 0;      // permutations resident at once, fixed by the upload that sized the scratch buffers
    int rng_mode = 0;       // 0: exact numpy PCG64 replay, 1: keyed-bijection ("philox") fast mode
    uint64_t philox_seed = 0;
    int64_t perm_first = 0;  // global index of permutation 0 of this handle (multi-GPU shards keep their global indices)
    DevBuf<uint32_t> d_cum;  // [nseg][n_cls + 1] class offsets of every segment's sorted labels (fast mode)
    DevBuf<uint32_t> d_bkt;  // per segment: class at the first value of every bucket (fast mode class lookup)
    std::vector<int64_t> h_seg_start, h_seg_len, h_bkt_off;
    bool philox_ready = false;
    std::vector<PhiloxSeg> h_pseg;
    // label matrices [chunk][stride] and [PB/32][n + 1][32] live in ctx->scratch[0..1]
    DevBuf<uint32_t> d_counts;  // [P][C*C]
    DevBuf<uint32_t> d_tmp_u32;
    std::vector<uint32_t> h_order;
    // options
    int shuffle_algo = -1;  // -1 auto (see launch_shuffle); 1 CTA per permutation (2a); 2 warp per permutation (2b);
                            // 7 swap-target generation + list apply (2d, 2e)
    int shuffle_q = 4;     // algos 2, 7: PCG64 outputs per lane per batch (window = 64*q raw values)
    int shuffle_r = 4;     // algo 7: Fisher-Yates steps per thread and window (window = r*threads steps)
    int64_t shuffle_low = 0;   // algo 7: elements of every label array kept in shared memory (-1 = as much as fits, 0 = off)
    int64_t shuffle_stagger_us = 0;  // start-up stagger of the persistent shuffle CTAs / warps (see sqb_stagger)
    int shuffle_threads = 512;
    int64_t perm_chunk = 0;  // 0 = auto
    int count_algo = 0;
    int count_single = 1;  // sqb_nhood_count: 1 = dedicated single-vector kernel, 0 = the batched kernels (test hook)
    int64_t shuffle_ctas = 0;          // persistent CTAs of the shuffle kernel (0 = occupancy x SM count)
    int shuffle_wfactor_x100 = 400;    // window = min(i/4, wfactor * sqrt(i)) raw values
};

template <typename LT>
static int launch_count(sqb_nhood* h, const LT* labT, int PB, int P, uint32_t* d_counts) {
    sqb_ctx* c = h->ctx;
    const int C = h->n_cls;
    const size_t smem_limit = c->smem_optin > 8192 ? c->smem_optin - 4096 : 40000;
    int G = 0;
    if (h->count_algo != 2) {
        for (int g = 32; g >= 1; g >>= 1) {
            if ((size_t)C * C * g * 4 <= smem_limit) {
                G = g;
                break;
            }
        }
    }
    const int ngroups_of = (G > 0) ? G : 32;
    const int ngroups = (P + ngroups_of - 1) / ngroups_of;
    int64_t nchunk = ceil_div64((int64_t)4 * c->sm_count, ngroups);
    const int64_t max_chunk = ceil_div64(h->n, 512);
    if (nchunk > max_chunk) nchunk = max_chunk;
    if (nchunk < 1) nchunk = 1;
    const int64_t nodes_per_cta = ceil_div64(h->n, nchunk);
    nchunk = ceil_div64(h->n, nodes_per_cta);
    dim3 grid((unsigned)nchunk, (unsigned)ngroups);
    SqbLaunchScope scope(c, SQB_K_NHOOD_COUNT);
    if (G == 0) {
        nhood_count_global_kernel<LT><<<grid, 256, 0, c->stream>>>(h->d_indptr.p, h->d_indices.p, labT, PB, h->n, C,
                                                                   nodes_per_cta, P, d_counts);
        SQB_POST_LAUNCH();
        return SQB_OK;
    }
    const size_t smem = (size_t)C * C * G * 4;
    const int threads = smem > 100 * 1024 ? 1024 : 512;
#define SQB_COUNT_CASE(GV)                                                                                        \
    case GV: {                                                                                                    \
        auto k = nhood_count_kernel<LT, GV>;                                                                      \
        SQB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));               \
        k<<<grid, threads, smem, c->stream>>>(h->d_indptr.p, h->d_indices.p, labT, PB, h->n, C, nodes_per_cta, P, \
                                              d_counts);                                                          \
    } break;
    if (G == 32 && h->n_recs > 0 && h->count_sym != 0 && (size_t)C * (C + 1) * 128 <= smem_limit) {  // record kernel (4b): mirrored flush for symmetric graphs
        void (*k)(const uint4*, int64_t, const LT*, int64_t, int, int64_t, int, uint32_t*) = nullptr;
#define SQB_RECS_PICK(UNV) (h->sym ? nhood_count_recs_kernel<LT, UNV, true> : nhood_count_recs_kernel<LT, UNV, false>)
        // records per warp pass, measured at 1M spots x 1000 permutations: 1 -> 2.38 ms, 2 -> 1.95, 3 -> 1.57, 4 -> 1.52
        k = SQB_RECS_PICK(4);
        if (h->count_un == 1) k = SQB_RECS_PICK(1);
        if (h->count_un == 2) k = SQB_RECS_PICK(2);
        if (h->count_un == 3) k = SQB_RECS_PICK(3);
#undef SQB_RECS_PICK
        // grid = pchunk x ngroups CTAs, one per SM at a time: aim at ~8 waves and, when a nearby pchunk makes the CTA count a
        // multiple of the SM count, take it (608 CTAs = 4.1 waves cost a fifth round for 10% of the work)
        int64_t pchunk = ((int64_t)8 * c->sm_count + ngroups / 2) / ngroups;
        if (pchunk < 1) pchunk = 1;
        for (int64_t q = pchunk; q <= 2 * pchunk; ++q)
            if ((q * ngroups) % c->sm_count == 0) {
                pchunk = q;
                break;
            }
        const int64_t max_pchunk = ceil_div64(h->n_recs, 1024);
        if (pchunk > max_pchunk) pchunk = max_pchunk;
        if (pchunk < 1) pchunk = 1;
        const int64_t recs_per_cta = ceil_div64(h->n_recs, pchunk);
        pchunk = ceil_div64(h->n_recs, recs_per_cta);
        if (pchunk < 1) pchunk = 1;
        dim3 pgrid((unsigned)pchunk, (unsigned)ngroups);
        const size_t rsmem = (size_t)C * (C + 1) * 128;  // one spare column per row
        nhood_spare_row_kernel<LT><<<(unsigned)((PB + 255) / 256), 256, 0, c->stream>>>(const_cast<LT*>(labT), h->n, PB, C);
        SQB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsmem));
        k<<<pgrid, threads, rsmem, c->stream>>>(h->d_recs.p, h->n_recs, labT, h->n, C, recs_per_cta, P, d_counts);
        SQB_POST_LAUNCH();
        if (h->sym && h->n_self > 0) {
            dim3 sgrid((unsigned)(h->n_self < 4096 ? h->n_self : 4096), (unsigned)((P + 127) / 128));
            nhood_count_selfloops_kernel<LT><<<sgrid, 128, 0, c->stream>>>(h->d_selfnodes.p, h->n_self, labT, h->n, C, P, d_counts);
            SQB_POST_LAUNCH();
        }
        return SQB_OK;
    }
    switch (G) {
        SQB_COUNT_CASE(32)
        SQB_COUNT_CASE(16)
        SQB_COUNT_CASE(8)
        SQB_COUNT_CASE(4)
        SQB_COUNT_CASE(2)
        SQB_COUNT_CASE(1)
    }
#undef SQB_COUNT_CASE
    SQB_POST_LAUNCH();
    return SQB_OK;
}

template <typename LT, int NT>
static int launch_shuffle_nt(sqb_nhood* h, LT* lab, const uint64_t* states, int64_t np) {
    sqb_ctx* c = h->ctx;
    auto k = nhood_shuffle_cta_kernel<LT, NT>;
    // [tab u64 x 4NT][sj u32 x 2NT][flag u32 x NT/16][wsum int x 36][own LT x 2NT][hval LT x 4NT]
    const size_t smem = (size_t)4 * NT * 8 + (size_t)2 * NT * 4 + (size_t)(NT / 16) * 4 + 36 * 4 + (size_t)6 * NT * sizeof(LT);
    SQB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t grid = h->shuffle_ctas;
    if (grid <= 0) {
        int per_sm = 1;
        SQB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, NT, smem));
        if (per_sm < 1) per_sm = 1;
        grid = (int64_t)per_sm * c->sm_count;
    }
    if (grid > np) grid = np;
    k<<<(unsigned)grid, NT, smem, c->stream>>>(lab, h->stride, states, np, h->nseg, h->d_seg_start.p, h->d_seg_len.p,
                                            (float)h->shuffle_wfactor_x100 / 100.0f, 0xFFFFFFFFu,
                                            (uint64_t)h->shuffle_stagger_us * 1000ull);
    return SQB_OK;
}

template <typename LT, int NT, int SPT>
static int launch_apply_list(sqb_nhood* h, LT* lab, const uint32_t* J, int64_t np, int64_t low) {
    sqb_ctx* c = h->ctx;
    auto k = nhood_apply_list_kernel<LT, NT, SPT>;
    constexpr size_t W = (size_t)NT * SPT, HS = W, NWB = 2 * W;
    // [tab u64 x 2*HS][bits u32 x 2*NWB][ohead u32 x 2*W][next u16 x 2*W][otop LT x W]
    const size_t tables = 2 * HS * 8 + 2 * NWB * 4 + 2 * W * 4 + 2 * W * 2 + W * sizeof(LT);
    SQB_CHECK(tables <= c->smem_optin, SQB_ERR_UNSUPPORTED, "shuffle_algo 7: %zu bytes of shared memory exceed the device limit", tables);
    // shared-memory resident low part (low: -1 = everything the SM has left, 0 = off, > 0 = at most that many elements)
    int64_t low_cap = 0;
    if (low != 0) {
        int64_t avail = ((int64_t)c->smem_optin - (int64_t)tables) / (int64_t)sizeof(LT);
        if (low > 0 && avail > low) avail = low;
        low_cap = avail > 0 ? (avail / 1024) * 1024 : 0;
    }
    const size_t smem = tables + (size_t)low_cap * sizeof(LT);
    SQB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t grid = h->shuffle_ctas;
    if (grid <= 0) {
        int per_sm = 1;
        SQB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, NT, smem));
        grid = (int64_t)(per_sm < 1 ? 1 : per_sm) * c->sm_count;
    }
    if (grid > np) grid = np;
    k<<<(unsigned)grid, NT, smem, c->stream>>>(lab, J, h->stride, np, h->nseg, h->d_seg_start.p, h->d_seg_len.p, 0xFFFFFFFFu,
                                               (uint64_t)h->shuffle_stagger_us * 1000ull, (int)low_cap);
    return SQB_OK;
}

// shuffle_algo 7: swap-target generation (2d), then the list apply (2e) with nt threads, r steps per thread and window and
// low elements of every label array in shared memory
template <typename LT>
static int launch_shuffle_two_kernel(sqb_nhood* h, LT* lab, const uint64_t* states, int64_t np, int nt, int r, int64_t low) {
    sqb_ctx* c = h->ctx;
    SQB_TRY(c->scratch[2].alloc((size_t)np * h->stride * sizeof(uint32_t)));
    uint32_t* J = reinterpret_cast<uint32_t*>(c->scratch[2].p);
    {
        SqbLaunchScope scope(c, SQB_K_MISC);  // J generation is accounted under "misc"
        // one warp per permutation; small blocks spread the (latency-bound) warps evenly over the SMs
        const int jt = (int)h->jgen_threads;
        int64_t ctas = (int64_t)c->sm_count * 8 * (128 / jt);
        if (ctas > ceil_div64(np, jt / 32)) ctas = ceil_div64(np, jt / 32);
        if (h->shuffle_q == 2)
            nhood_jgen_kernel<2><<<(unsigned)ctas, jt, 0, c->stream>>>(J, h->stride, states, np, h->nseg, h->d_seg_start.p, h->d_seg_len.p, 4.0f);
        else if (h->shuffle_q == 8)
            nhood_jgen_kernel<8><<<(unsigned)ctas, jt, 0, c->stream>>>(J, h->stride, states, np, h->nseg, h->d_seg_start.p, h->d_seg_len.p, 4.0f);
        else
            nhood_jgen_kernel<4><<<(unsigned)ctas, jt, 0, c->stream>>>(J, h->stride, states, np, h->nseg, h->d_seg_start.p, h->d_seg_len.p, 4.0f);
        SQB_POST_LAUNCH();
    }
    SqbLaunchScope scope(c, SQB_K_NHOOD_SHUFFLE);
    int rc = SQB_ERR_INVALID;
    if (nt == 1024 && r == 4) rc = launch_apply_list<LT, 1024, 4>(h, lab, J, np, low);
    else if (nt == 1024 && r == 2) rc = launch_apply_list<LT, 1024, 2>(h, lab, J, np, low);
    else if (nt == 512 && r == 8) rc = launch_apply_list<LT, 512, 8>(h, lab, J, np, low);
    else if (nt == 512 && r == 4) rc = launch_apply_list<LT, 512, 4>(h, lab, J, np, low);
    else if (nt == 512 && r == 2) rc = launch_apply_list<LT, 512, 2>(h, lab, J, np, low);
    else if (nt == 256 && r == 8) rc = launch_apply_list<LT, 256, 8>(h, lab, J, np, low);
    else if (nt == 256 && r == 4) rc = launch_apply_list<LT, 256, 4>(h, lab, J, np, low);
    else if (nt == 128 && r == 4) rc = launch_apply_list<LT, 128, 4>(h, lab, J, np, low);
    else sqb_set_error("shuffle_algo 7: unsupported (shuffle_threads, shuffle_r) = (%d, %d)", nt, r);
    SQB_TRY(rc);
    SQB_POST_LAUNCH();
    return SQB_OK;
}

template <typename LT>
static int launch_shuffle(sqb_nhood* h, LT* lab, const uint64_t* states, int64_t np) {
    sqb_ctx* c = h->ctx;
    if (h->shuffle_algo == 7) return launch_shuffle_two_kernel<LT>(h, lab, states, np, h->shuffle_threads, h->shuffle_r, h->shuffle_low);
    // auto (measured on B200, 1000 x 1M: two-kernel list replay 23 ms, warp per permutation 39 ms, CTA per permutation
    // 42 ms): many permutations of large arrays -> J generation + list apply with the tuned shape (1024 threads, 2048-step
    // windows, 96 K elements of every array in shared memory); few permutations -> one CTA each (finishes sooner);
    // many permutations of small arrays (L1/L2 resident) -> one warp each
    if (h->shuffle_algo < 0 && np > 2 * (int64_t)c->sm_count && h->n >= 65536)
        return launch_shuffle_two_kernel<LT>(h, lab, states, np, 1024, 2, 98304);
    SqbLaunchScope scope(c, SQB_K_NHOOD_SHUFFLE);
    const int algo = h->shuffle_algo >= 0 ? h->shuffle_algo : (np <= 2 * (int64_t)c->sm_count ? 1 : 2);
    if (algo == 2) {
        const float wf = (float)h->shuffle_wfactor_x100 / 100.0f;
        int64_t ctas = h->shuffle_ctas > 0 ? h->shuffle_ctas : (int64_t)c->sm_count * 8;
        if (ctas > ceil_div64(np, 4)) ctas = ceil_div64(np, 4);
        switch (h->shuffle_q) {
            case 1:
                nhood_shuffle_warp_kernel<LT, 1><<<(unsigned)ctas, 128, 0, c->stream>>>(lab, h->stride, states, np, h->nseg,
                                                                                       h->d_seg_start.p, h->d_seg_len.p, wf,
                                                                                       (uint64_t)h->shuffle_stagger_us * 1000ull);
                break;
            case 2:
                nhood_shuffle_warp_kernel<LT, 2><<<(unsigned)ctas, 128, 0, c->stream>>>(lab, h->stride, states, np, h->nseg,
                                                                                       h->d_seg_start.p, h->d_seg_len.p, wf,
                                                                                       (uint64_t)h->shuffle_stagger_us * 1000ull);
                break;
            default:
                nhood_shuffle_warp_kernel<LT, 4><<<(unsigned)ctas, 128, 0, c->stream>>>(lab, h->stride, states, np, h->nseg,
                                                                                       h->d_seg_start.p, h->d_seg_len.p, wf,
                                                                                       (uint64_t)h->shuffle_stagger_us * 1000ull);
                break;
        }
    } else {
        switch (h->shuffle_threads) {
            case 128:
                SQB_TRY((launch_shuffle_nt<LT, 128>(h, lab, states, np)));
                break;
            case 256:
                SQB_TRY((launch_shuffle_nt<LT, 256>(h, lab, states, np)));
                break;
            case 1024:
                SQB_TRY((launch_shuffle_nt<LT, 1024>(h, lab, states, np)));
                break;
            default:
                SQB_TRY((launch_shuffle_nt<LT, 512>(h, lab, states, np)));
                break;
        }
    }
    SQB_POST_LAUNCH();
    return SQB_OK;
}

static int64_t auto_chunk(sqb_nhood* h) {
    if (h->perm_chunk > 0) return ((h->perm_chunk + 31) / 32) * 32;
    // keep [chunk][stride] + [n][chunk] under ~8 GB
    int64_t per_perm = 2 * h->stride * h->lt_bytes + 4 * h->stride;  // label matrices + uint32 target lists (algo 7)
    int64_t ch = (int64_t)8e9 / (per_perm > 0 ? per_perm : 1);
    if (ch < 32) ch = 32;
    if (ch > 16384) ch = 16384;
    return (ch / 32) * 32;
}

template <typename LT>
static int run_chunk(sqb_nhood* h, int64_t p0, int64_t np, bool do_count) {
    sqb_ctx* c = h->ctx;
    LT* lab = reinterpret_cast<LT*>(c->scratch[0].p);
    LT* labT = reinterpret_cast<LT*>(c->scratch[1].p);
    const int64_t vec_per_row = h->stride * (int64_t)sizeof(LT) / 16;
    {
        SqbLaunchScope scope(c, SQB_K_NHOOD_FILL);
        unsigned gx = (unsigned)ceil_div64(vec_per_row, 256 * 4);
        if (gx < 1) gx = 1;
        if (gx > 64) gx = 64;
        dim3 fgrid(gx, (unsigned)(np < 4096 ? np : 4096));
        nhood_fill_kernel<<<fgrid, 256, 0, c->stream>>>(reinterpret_cast<uint4*>(lab),
                                                                  reinterpret_cast<const uint4*>(h->d_base.p),
                                                                  vec_per_row, np);
        SQB_POST_LAUNCH();
    }
    SQB_TRY(launch_shuffle<LT>(h, lab, h->d_states.p + p0 * 4, np));
    if (!do_count) return SQB_OK;
    const int PB = (int)(((np + 31) / 32) * 32);
    {
        SqbLaunchScope scope(c, SQB_K_NHOOD_TRANSPOSE);
        dim3 grid((unsigned)ceil_div64(h->n, 256), (unsigned)(PB / 32));
        nhood_transpose_kernel<LT><<<grid, 256, 0, c->stream>>>(lab, labT, h->n, h->stride, (int)np, PB,
                                                                h->has_order ? h->d_order.p : nullptr);
        SQB_POST_LAUNCH();
    }
    SQB_TRY(launch_count<LT>(h, labT, PB, (int)np, h->d_counts.p + p0 * (int64_t)h->n_cls * h->n_cls));
    return SQB_OK;
}

// fast RNG mode: labels of permutations [p0, p0 + np) straight into labT[PB/32][n + 1][32] (one launch per library segment)
template <typename LT>
static int philox_labels(sqb_nhood* h, int64_t p0, int64_t np, LT* labT, int PB) {
    sqb_ctx* c = h->ctx;
    const int C = h->n_cls;
    for (int sgm = 0; sgm < h->nseg; ++sgm) {
        const PhiloxSeg& ps = h->h_pseg[sgm];
        const int64_t m = ps.len;
        if (m <= 0) continue;
        const size_t smem = ((size_t)(C + 1) + (size_t)ps.tsize + 1) * sizeof(uint32_t);
        SQB_CHECK(smem <= h->ctx->smem_optin, SQB_ERR_UNSUPPORTED, "fast RNG mode: %d classes do not fit the shared-memory class table", C);
        if (smem > 48 * 1024)
            SQB_CUDA(cudaFuncSetAttribute(nhood_philox_labels_kernel<LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int gy = (PB / 4 + 31) / 32;
        int64_t gx = ceil_div64((int64_t)c->sm_count * 8, gy);
        if (gx > ceil_div64(m, 8)) gx = ceil_div64(m, 8);
        if (gx < 1) gx = 1;
        const int64_t pos_per_cta = ceil_div64(m, gx);
        gx = ceil_div64(m, pos_per_cta);
        SqbLaunchScope scope(c, SQB_K_NHOOD_SHUFFLE);
        nhood_philox_labels_kernel<LT><<<dim3((unsigned)gx, (unsigned)gy), 256, smem, c->stream>>>(
            labT, PB, h->n, ps, h->d_cum.p + (size_t)sgm * (C + 1), C, h->d_bkt.p + h->h_bkt_off[sgm], h->has_order ? h->d_order.p : nullptr,
            h->philox_seed, h->perm_first + p0, pos_per_cta);
        SQB_POST_LAUNCH();
    }
    (void)np;
    return SQB_OK;
}

template <typename LT>
static int run_chunk_philox(sqb_nhood* h, int64_t p0, int64_t np) {
    LT* labT = reinterpret_cast<LT*>(h->ctx->scratch[1].p);
    const int PB = (int)(((np + 31) / 32) * 32);
    SQB_TRY(philox_labels<LT>(h, p0, np, labT, PB));
    return launch_count<LT>(h, labT, PB, (int)np, h->d_counts.p + p0 * (int64_t)h->n_cls * h->n_cls);
}

// class histogram of one segment of the (library-grouped) base labels, for the fast-mode class tables
template <typename LT>
__global__ void nhood_class_hist_kernel(const LT* __restrict__ base, int64_t start, int64_t len, int C, uint32_t* __restrict__ out) {
    extern __shared__ uint32_t s_h[];
    const bool priv = C <= 4096;
    if (priv) {
        for (int c = threadIdx.x; c < C; c += blockDim.x) s_h[c] = 0u;
        __syncthreads();
    }
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < len; k += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t l = (uint32_t)base[start + k];
        if (priv) atomicAdd(&s_h[l], 1u);
        else atomicAdd(&out[l], 1u);
    }
    if (priv) {
        __syncthreads();
        for (int c = threadIdx.x; c < C; c += blockDim.x)
            if (s_h[c]) atomicAdd(&out[c], s_h[c]);
    }
}

// fast RNG mode tables (built lazily: the exact mode never needs them)
static int philox_prepare(sqb_nhood* h) {
    if (h->philox_ready) return SQB_OK;
    sqb_ctx* c = h->ctx;
    const std::vector<int64_t>& seg_start = h->h_seg_start;
    const std::vector<int64_t>& seg_len = h->h_seg_len;
    // class counts of every segment, from the grouped base labels on the device (the host keeps no copy of the labels)
    const int64_t C1h = (int64_t)h->n_cls + 1;
    std::vector<uint32_t> hcnt((size_t)h->nseg * C1h, 0u);
    {
        DevBuf<uint32_t> d_hist;
        d_hist.bind(c->stream);
        SQB_TRY(d_hist.alloc(hcnt.size()));
        cudaError_t e = cudaMemsetAsync(d_hist.p, 0, hcnt.size() * sizeof(uint32_t), c->stream);
        for (int sgm = 0; sgm < h->nseg && e == cudaSuccess; ++sgm) {
            const int64_t m = seg_len[sgm];
            if (m <= 0) continue;
            const unsigned g = (unsigned)(m < 256 * 296 ? ceil_div64(m, 256) : 296);
            const size_t sm = h->n_cls <= 4096 ? (size_t)h->n_cls * 4 : 0;
            if (h->lt_bytes == 1)
                nhood_class_hist_kernel<uint8_t><<<g, 256, sm, c->stream>>>(h->d_base.p, seg_start[sgm], m, h->n_cls, d_hist.p + (size_t)sgm * C1h + 1);
            else
                nhood_class_hist_kernel<uint16_t><<<g, 256, sm, c->stream>>>(reinterpret_cast<const uint16_t*>(h->d_base.p), seg_start[sgm], m,
                                                                              h->n_cls, d_hist.p + (size_t)sgm * C1h + 1);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(hcnt.data(), d_hist.p, hcnt.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        d_hist.release();
        if (e != cudaSuccess) {
            sqb_set_error("fast RNG mode: class histogram failed: %s", cudaGetErrorString(e));
            return SQB_ERR_CUDA;
        }
    }
    {  // fast RNG mode: per segment the class offsets of its labels sorted by class, the Feistel radices and a bucket table
       // (class at the first value of every bucket of 2^shift values) that shortens the class search to `steps` bisections
        const int64_t C1 = (int64_t)h->n_cls + 1;
        std::vector<uint32_t> cum((size_t)h->nseg * C1, 0u), bkt;
        h->h_pseg.assign(h->nseg, PhiloxSeg());
        h->h_bkt_off.assign(h->nseg, 0);
        for (int sgm = 0; sgm < h->nseg; ++sgm) {
            uint32_t* row = cum.data() + (size_t)sgm * C1;
            const int64_t m = seg_len[sgm];
            for (int64_t cc = 0; cc <= h->n_cls; ++cc) row[cc] = hcnt[(size_t)sgm * C1 + cc];  // row[c + 1] = labels of class c
            for (int64_t cc = 0; cc < h->n_cls; ++cc) row[cc + 1] += row[cc];
            PhiloxSeg& ps = h->h_pseg[sgm];
            ps.start = seg_start[sgm];
            ps.len = m;
            ps.seg = sgm;
            uint64_t a = (uint64_t)sqrt((double)(m > 0 ? m : 1));
            while (a * a < (uint64_t)m) ++a;
            while (a > 1 && (a - 1) * (a - 1) >= (uint64_t)m) --a;
            if (a < 1) a = 1;
            ps.a = (uint32_t)a;
            ps.b = (uint32_t)((m + (int64_t)a - 1) / (int64_t)a);
            if (ps.b < 1) ps.b = 1;
            int bits = 0;
            while (bits < 32 && ((uint64_t)(m > 0 ? m - 1 : 0) >> bits) != 0) ++bits;
            ps.shift = bits > 11 ? bits - 11 : 0;  // <= 2048 buckets
            ps.tsize = (int)((((uint64_t)(m > 0 ? m - 1 : 0)) >> ps.shift) + 1);
            h->h_bkt_off[sgm] = (int64_t)bkt.size();
            auto class_of = [&](uint64_t v) {  // last c in [0, n_cls) with row[c] <= v
                int lo = 0, hi = h->n_cls - 1;
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if ((uint64_t)row[mid] <= v) lo = mid; else hi = mid - 1;
                }
                return (uint32_t)lo;
            };
            for (int t = 0; t <= ps.tsize; ++t) bkt.push_back(class_of((uint64_t)t << ps.shift));
            // the kernel searches [table[bucket], table[bucket + 1]] (class at the first value of this / of the next bucket)
            uint32_t maxrange = 0;
            for (int t = 0; t < ps.tsize; ++t) {
                const uint32_t d = bkt[h->h_bkt_off[sgm] + t + 1] - bkt[h->h_bkt_off[sgm] + t];
                if (d > maxrange) maxrange = d;
            }
            int steps = 0;
            while ((1u << steps) < maxrange + 1u) ++steps;
            ps.steps = steps;
        }
        SQB_TRY(h->d_cum.alloc(cum.size()));
        SQB_TRY(h->d_bkt.alloc(bkt.size() > 0 ? bkt.size() : 1));
        SQB_CUDA(cudaMemcpyAsync(h->d_cum.p, cum.data(), cum.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        SQB_CUDA(cudaMemcpyAsync(h->d_bkt.p, bkt.data(), bkt.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        SQB_CUDA(cudaStreamSynchronize(c->stream));  // cum / bkt are locals
    }
    h->philox_ready = true;
    return SQB_OK;
}

// observed count through the BATCHED kernels (lane = permutation, symmetric shortcut): test hook, option count_single = 0
static int nhood_count_batched_path(sqb_nhood* h, const uint32_t* labels, uint32_t* out) {
    SQB_CHECK(h && labels && out, SQB_ERR_INVALID, "sqb_nhood_count: null argument");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    for (int64_t i = 0; i < h->n; ++i)
        SQB_CHECK(labels[i] < (uint32_t)h->n_cls, SQB_ERR_INVALID, "sqb_nhood_count: labels[%lld]=%u >= n_cls=%d",
                  (long long)i, labels[i], h->n_cls);
    const int64_t CC = (int64_t)h->n_cls * h->n_cls;
    DevBuf<uint8_t> labT;
    DevBuf<uint32_t> cnt;
    labT.bind(c->stream);
    cnt.bind(c->stream);
    int rc = SQB_OK;
    if ((rc = h->d_tmp_u32.alloc(h->n)) != SQB_OK) return rc;
    if ((rc = labT.alloc((size_t)(h->n + 1) * 32 * h->lt_bytes)) != SQB_OK) return rc;
    if ((rc = cnt.alloc(CC)) != SQB_OK) {
        labT.release();
        return rc;
    }
    auto cleanup = [&]() {
        labT.release();
        cnt.release();
    };
    cudaError_t e;
    e = cudaMemcpyAsync(h->d_tmp_u32.p, labels, h->n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(labT.p, 0, (size_t)(h->n + 1) * 32 * h->lt_bytes, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(cnt.p, 0, CC * sizeof(uint32_t), c->stream);
    if (e != cudaSuccess) {
        cleanup();
        sqb_set_error("sqb_nhood_count: %s", cudaGetErrorString(e));
        return SQB_ERR_CUDA;
    }
    {
        SqbLaunchScope scope(c, SQB_K_MISC);
        unsigned g = (unsigned)ceil_div64(h->n, 256);
        if (h->lt_bytes == 1)
            nhood_single_to_T_kernel<uint8_t><<<g, 256, 0, c->stream>>>(h->d_tmp_u32.p, labT.p, h->n);
        else
            nhood_single_to_T_kernel<uint16_t><<<g, 256, 0, c->stream>>>(h->d_tmp_u32.p, reinterpret_cast<uint16_t*>(labT.p), h->n);
    }
    rc = (h->lt_bytes == 1) ? launch_count<uint8_t>(h, labT.p, 32, 1, cnt.p)
                            : launch_count<uint16_t>(h, reinterpret_cast<uint16_t*>(labT.p), 32, 1, cnt.p);
    if (rc == SQB_OK) {
        e = cudaMemcpyAsync(out, cnt.p, CC * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) {
            sqb_set_error("sqb_nhood_count: %s", cudaGetErrorString(e));
            rc = SQB_ERR_CUDA;
        }
    }
    cleanup();
    return rc;
}


static int ensure_buffers(sqb_nhood* h, int64_t chunk) {
    SQB_TRY(h->ctx->scratch[0].alloc((size_t)chunk * h->stride * h->lt_bytes));
    SQB_TRY(h->ctx->scratch[1].alloc((size_t)(h->n + 1) * chunk * h->lt_bytes));
    return SQB_OK;
}

// row records (3c) of the CSR (ptr, idx) into h->d_recs; *n_self = number of stored (i, i) among them
static int nhood_build_records(sqb_nhood* h, const uint32_t* ptr, const uint32_t* idx, uint32_t* n_self_out) {
    sqb_ctx* ctx = h->ctx;
    const int64_t n = h->n;
    DevBuf<uint32_t> cnt, rptr, cnt_self;
    DevBuf<uint8_t> tmp;
    cnt.bind(ctx->stream), rptr.bind(ctx->stream), cnt_self.bind(ctx->stream), tmp.bind(ctx->stream);
    auto cleanup = [&]() { cnt.release(), rptr.release(), cnt_self.release(), tmp.release(); };
    int rc;
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)(n + 1), ctx->stream);
    if ((rc = cnt.alloc(n + 1)) != SQB_OK || (rc = rptr.alloc(n + 1)) != SQB_OK || (rc = cnt_self.alloc(1)) != SQB_OK ||
        (rc = tmp.alloc(tmp_bytes > 0 ? tmp_bytes : 1)) != SQB_OK) {
        cleanup();
        return rc;
    }
    nhood_rec_count_kernel<<<(unsigned)ceil_div64(n + 1, 256), 256, 0, ctx->stream>>>(ptr, n, cnt.p);
    cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, cnt.p, rptr.p, (int)(n + 1), ctx->stream);
    uint32_t total = 0, h_self = 0;
    cudaMemcpyAsync(&total, rptr.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess && total > 0 && (rc = h->d_recs.alloc(total)) == SQB_OK) {
        cudaMemsetAsync(cnt_self.p, 0, sizeof(uint32_t), ctx->stream);
        nhood_rec_fill_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(ptr, idx, n, rptr.p, h->d_recs.p, cnt_self.p);
        cudaMemcpyAsync(&h_self, cnt_self.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream);
        e = cudaStreamSynchronize(ctx->stream);
    }
    cleanup();
    if (e != cudaSuccess) {
        sqb_set_error("sqb_nhood_create: building the row records failed: %s", cudaGetErrorString(e));
        return SQB_ERR_CUDA;
    }
    if (rc != SQB_OK) return rc;
    h->n_recs = total;
    *n_self_out = h_self;
    return SQB_OK;
}

extern "C" {

int sqb_nhood_create(sqb_ctx* ctx, int64_t n, int64_t nnz, const uint32_t* indptr, const uint32_t* indices, int n_cls,
                     sqb_nhood** out) {
    SQB_CHECK(ctx && out, SQB_ERR_INVALID, "sqb_nhood_create: null ctx/out");
    SQB_CHECK(n >= 1 && n < 0x7FFFFFFFLL, SQB_ERR_INVALID, "sqb_nhood_create: n=%lld out of range [1, 2^31-1)", (long long)n);
    SQB_CHECK(nnz >= 0 && nnz < 0xFFFFFFFFLL, SQB_ERR_INVALID, "sqb_nhood_create: nnz=%lld does not fit uint32",
              (long long)nnz);
    // same message as the reference (_nhood.py:107-108)
    SQB_CHECK(n_cls >= 2, SQB_ERR_INVALID, "Expected at least `2` clusters, found `%d`.", n_cls);
    SQB_CHECK(n_cls <= 65535, SQB_ERR_UNSUPPORTED, "sqb_nhood_create: n_cls=%d > 65535 unsupported", n_cls);
    SQB_CHECK(indptr && (indices || nnz == 0), SQB_ERR_INVALID, "sqb_nhood_create: null CSR arrays");
    SQB_CHECK(indptr[0] == 0 && (int64_t)indptr[n] == nnz, SQB_ERR_INVALID,
              "sqb_nhood_create: indptr[0]=%u indptr[n]=%u inconsistent with nnz=%lld", indptr[0], indptr[n],
              (long long)nnz);
    SQB_CUDA(cudaSetDevice(ctx->device));
    sqb_nhood* h = new sqb_nhood();
    h->ctx = ctx;
    // all handle buffers are allocated, used and freed in ctx->stream order
    h->d_indptr.bind(ctx->stream);
    h->d_indices.bind(ctx->stream);
    h->d_uptr.bind(ctx->stream);
    h->d_uidx.bind(ctx->stream);
    h->d_recs.bind(ctx->stream);
    h->d_selfnodes.bind(ctx->stream);
    h->d_base.bind(ctx->stream);
    h->d_order.bind(ctx->stream);
    h->d_seg_start.bind(ctx->stream);
    h->d_seg_len.bind(ctx->stream);
    h->d_states.bind(ctx->stream);
    h->d_counts.bind(ctx->stream);
    h->d_tmp_u32.bind(ctx->stream);
    h->d_cum.bind(ctx->stream);
    h->d_bkt.bind(ctx->stream);
    h->n = n;
    h->nnz = nnz;
    h->n_cls = n_cls;
    h->lt_bytes = n_cls <= 256 ? 1 : 2;
    h->stride = ((n + 15) / 16) * 16;
    int rc;
    if ((rc = h->d_indptr.alloc(n + 1)) != SQB_OK || (rc = h->d_indices.alloc(nnz > 0 ? nnz : 1)) != SQB_OK) {
        sqb_nhood_destroy(h);
        return rc;
    }
    SQB_CUDA(cudaMemcpyAsync(h->d_indptr.p, indptr, (n + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    if (nnz > 0)
        SQB_TRY(sqb_h2d(ctx, h->d_indices.p, indices, nnz * sizeof(uint32_t)));
    // symmetric structure? then keep the entries with j >= i as a second CSR (3b)
    if (nnz > 0) {
        DevBuf<uint32_t> flag, ucnt;
        DevBuf<uint8_t> tmp;
        flag.bind(ctx->stream);
        ucnt.bind(ctx->stream);
        tmp.bind(ctx->stream);
        uint32_t hflag = 1;
        auto cleanup = [&]() {
            flag.release();
            ucnt.release();
            tmp.release();
        };
        rc = flag.alloc(1);
        if (rc == SQB_OK) rc = ucnt.alloc(n + 1);
        if (rc == SQB_OK) rc = h->d_uptr.alloc(n + 1);
        size_t tmp_bytes = 0;
        if (rc == SQB_OK) {
            cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, ucnt.p, h->d_uptr.p, (int)(n + 1), ctx->stream);
            rc = tmp.alloc(tmp_bytes > 0 ? tmp_bytes : 1);
        }
        if (rc != SQB_OK) {
            cleanup();
            sqb_nhood_destroy(h);
            return rc;
        }
        cudaMemsetAsync(flag.p, 0, sizeof(uint32_t), ctx->stream);
        nhood_symcheck_kernel<<<(unsigned)ceil_div64(n + 1, 256), 256, 0, ctx->stream>>>(h->d_indptr.p, h->d_indices.p, n, flag.p, ucnt.p);
        cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, ucnt.p, h->d_uptr.p, (int)(n + 1), ctx->stream);
        cudaMemcpyAsync(&hflag, flag.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e == cudaSuccess && (hflag & 2u)) {  // the kernels index the label arrays with these values: refuse
            cleanup();
            sqb_nhood_destroy(h);
            sqb_set_error("sqb_nhood_create: invalid CSR (column index outside [0, %lld) or indptr not monotone)", (long long)n);
            return SQB_ERR_INVALID;
        }
        if (e == cudaSuccess && hflag == 0) {
            uint32_t total = 0;
            cudaMemcpyAsync(&total, h->d_uptr.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream);
            e = cudaStreamSynchronize(ctx->stream);
            if (e == cudaSuccess && (rc = h->d_uidx.alloc(total > 0 ? total : 1)) == SQB_OK) {
                nhood_upper_fill_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(h->d_indptr.p, h->d_indices.p, n,
                                                                                              h->d_uptr.p, h->d_uidx.p);
                // the same entries as row records (3c) + the nodes with a self loop
                uint32_t h_self = 0;
                e = cudaStreamSynchronize(ctx->stream);
                if (e == cudaSuccess && (rc = nhood_build_records(h, h->d_uptr.p, h->d_uidx.p, &h_self)) == SQB_OK) {
                    if (h_self > 0 && (rc = h->d_selfnodes.alloc(h_self)) == SQB_OK) {
                        cudaMemsetAsync(flag.p, 0, sizeof(uint32_t), ctx->stream);
                        nhood_self_fill_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(h->d_uptr.p, h->d_uidx.p, n,
                                                                                                     h->d_selfnodes.p, flag.p);
                        e = cudaStreamSynchronize(ctx->stream);
                    }
                    h->n_self = h_self;
                    h->sym = (e == cudaSuccess && rc == SQB_OK);
                }
            }
        }
        cleanup();
        if (e != cudaSuccess || rc != SQB_OK) {
            if (e != cudaSuccess) sqb_set_error("sqb_nhood_create: symmetric-graph preparation failed: %s", cudaGetErrorString(e));
            sqb_nhood_destroy(h);
            return e != cudaSuccess ? SQB_ERR_CUDA : rc;
        }
        h->d_uptr.release();  // the count kernel walks the row records; the upper CSR was only their scaffolding
        h->d_uidx.release();
        const size_t smem_limit = ctx->smem_optin > 8192 ? ctx->smem_optin - 4096 : 40000;
        if (!h->sym && (size_t)n_cls * n_cls * 128 <= smem_limit && nnz < ((int64_t)1 << 31)) {
            // directed / irregular graph: row records of every stored entry, same kernel without the mirrored flush
            uint32_t unused = 0;
            if (nhood_build_records(h, h->d_indptr.p, h->d_indices.p, &unused) != SQB_OK) {
                h->d_recs.release();  // not fatal: the CSR-row kernel counts without them
                h->n_recs = 0;
            }
        }
    }
    SQB_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = h;
    return SQB_OK;
}

int sqb_nhood_destroy(sqb_nhood* h) {
    if (!h) return SQB_OK;
    cudaSetDevice(h->ctx->device);
    h->d_indptr.release();
    h->d_indices.release();
    h->d_uptr.release();
    h->d_uidx.release();
    h->d_recs.release();
    h->d_selfnodes.release();
    h->d_base.release();
    h->d_order.release();
    h->d_seg_start.release();
    h->d_seg_len.release();
    h->d_states.release();
    h->d_counts.release();
    h->d_cum.release();
    h->d_bkt.release();
    h->d_tmp_u32.release();
    delete h;
    return SQB_OK;
}

int sqb_nhood_set_option(sqb_nhood* h, const char* key, int64_t value) {
    SQB_CHECK(h && key, SQB_ERR_INVALID, "sqb_nhood_set_option: null argument");
    if (!strcmp(key, "shuffle_algo")) {
        SQB_CHECK(value == -1 || value == 1 || value == 2 || value == 7, SQB_ERR_INVALID, "shuffle_algo must be -1 (auto), 1, 2 or 7");
        h->shuffle_algo = (int)value;
    } else if (!strcmp(key, "jgen_threads")) {
        SQB_CHECK(value == 32 || value == 64 || value == 128, SQB_ERR_INVALID, "jgen_threads must be 32, 64 or 128");
        h->jgen_threads = (int)value;
    } else if (!strcmp(key, "count_un")) {
        SQB_CHECK(value >= 1 && value <= 4, SQB_ERR_INVALID, "count_un must be 1, 2, 3 or 4");
        h->count_un = (int)value;
    } else if (!strcmp(key, "count_single")) {
        h->count_single = value != 0;
    } else if (!strcmp(key, "count_sym")) {
        SQB_CHECK(value == -1 || value == 0, SQB_ERR_INVALID, "count_sym must be -1 (auto) or 0 (full CSR)");
        h->count_sym = (int)value;
    } else if (!strcmp(key, "shuffle_stagger_us")) {
        SQB_CHECK(value >= 0 && value <= 1000000, SQB_ERR_INVALID, "shuffle_stagger_us must be in [0, 1e6]");
        h->shuffle_stagger_us = value;
    } else if (!strcmp(key, "shuffle_low")) {
        SQB_CHECK(value >= -1, SQB_ERR_INVALID, "shuffle_low must be >= -1");
        h->shuffle_low = value;
    } else if (!strcmp(key, "shuffle_r")) {
        SQB_CHECK(value == 2 || value == 4 || value == 8, SQB_ERR_INVALID, "shuffle_r must be 2, 4 or 8");
        h->shuffle_r = (int)value;
    } else if (!strcmp(key, "shuffle_q")) {
        SQB_CHECK(value == 1 || value == 2 || value == 4 || value == 8, SQB_ERR_INVALID, "shuffle_q must be 1, 2, 4 or 8 (8: algo 7 only)");
        h->shuffle_q = (int)value;
    } else if (!strcmp(key, "shuffle_threads")) {
        SQB_CHECK(value == 128 || value == 256 || value == 512 || value == 1024, SQB_ERR_INVALID,
                  "shuffle_threads must be 128, 256, 512 or 1024");
        h->shuffle_threads = (int)value;
    } else if (!strcmp(key, "perm_chunk")) {
        SQB_CHECK(value >= 0, SQB_ERR_INVALID, "perm_chunk must be >= 0");
        h->perm_chunk = value;
    } else if (!strcmp(key, "shuffle_ctas")) {
        SQB_CHECK(value >= 0 && value <= 1000000, SQB_ERR_INVALID, "shuffle_ctas must be in [0, 1e6]");
        h->shuffle_ctas = value;
    } else if (!strcmp(key, "shuffle_wfactor_x100")) {
        SQB_CHECK(value >= 25 && value <= 6400, SQB_ERR_INVALID, "shuffle_wfactor_x100 must be in [25, 6400]");
        h->shuffle_wfactor_x100 = (int)value;
    } else if (!strcmp(key, "count_algo")) {
        SQB_CHECK(value >= 0 && value <= 2, SQB_ERR_INVALID, "count_algo must be 0, 1 or 2");
        h->count_algo = (int)value;
    } else {
        sqb_set_error("sqb_nhood_set_option: unknown key '%s'", key);
        return SQB_ERR_INVALID;
    }
    return SQB_OK;
}

int sqb_nhood_bytes_per_perm(sqb_nhood* h, int64_t* bytes) {
    SQB_CHECK(h && bytes, SQB_ERR_INVALID, "sqb_nhood_bytes_per_perm: null argument");
    *bytes = 4 * h->nnz + 4 * (h->n + 1) + 8 * h->n + 4 * (int64_t)h->n_cls * h->n_cls;
    return SQB_OK;
}

int sqb_nhood_count(sqb_nhood* h, const uint32_t* labels, uint32_t* out) {
    SQB_CHECK(h && labels && out, SQB_ERR_INVALID, "sqb_nhood_count: null argument");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    for (int64_t i = 0; i < h->n; ++i)
        SQB_CHECK(labels[i] < (uint32_t)h->n_cls, SQB_ERR_INVALID, "sqb_nhood_count: labels[%lld]=%u >= n_cls=%d",
                  (long long)i, labels[i], h->n_cls);
    if (!h->count_single) return nhood_count_batched_path(h, labels, out);
    const int64_t CC = (int64_t)h->n_cls * h->n_cls;
    DevBuf<uint32_t> cnt;
    cnt.bind(c->stream);
    int rc = SQB_OK;
    if ((rc = h->d_tmp_u32.alloc(h->n)) != SQB_OK) return rc;
    if ((rc = cnt.alloc(CC)) != SQB_OK) return rc;
    cudaError_t e = cudaMemcpyAsync(h->d_tmp_u32.p, labels, h->n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(cnt.p, 0, CC * sizeof(uint32_t), c->stream);
    if (e == cudaSuccess) {
        const size_t smem = (size_t)CC * sizeof(uint32_t);
        const int hist_smem = smem <= 160 * 1024 ? 1 : 0;
        if (hist_smem && smem > 48 * 1024) e = cudaFuncSetAttribute(nhood_count_single_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) {
            SqbLaunchScope scope(c, SQB_K_NHOOD_COUNT);
            int64_t ctas = ceil_div64(h->n, 8 * 16);  // >= 16 rows per warp
            const int64_t cap = (int64_t)c->sm_count * (smem > 32 * 1024 ? 2 : 8);
            if (ctas > cap) ctas = cap;
            if (ctas < 1) ctas = 1;
            nhood_count_single_kernel<<<(unsigned)ctas, 256, hist_smem ? smem : 0, c->stream>>>(h->d_indptr.p, h->d_indices.p, h->d_tmp_u32.p, h->n,
                                                                                                 h->n_cls, hist_smem, cnt.p);
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, cnt.p, CC * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cnt.release();
    if (e != cudaSuccess) {
        sqb_set_error("sqb_nhood_count: %s", cudaGetErrorString(e));
        return SQB_ERR_CUDA;
    }
    return SQB_OK;
}

int sqb_nhood_set_base(sqb_nhood* h, const uint32_t* base_labels, const int32_t* lib_codes, int n_libs) {
    SQB_CHECK(h && base_labels, SQB_ERR_INVALID, "sqb_nhood_set_base: null argument");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int64_t n = h->n;
    {  // one branch-free pass (this runs inside the end-to-end call: 1M labels)
        uint32_t mx = 0;
        for (int64_t i = 0; i < n; ++i) mx = base_labels[i] > mx ? base_labels[i] : mx;
        if (mx >= (uint32_t)h->n_cls)
            for (int64_t i = 0; i < n; ++i)
                SQB_CHECK(base_labels[i] < (uint32_t)h->n_cls, SQB_ERR_INVALID, "sqb_nhood_set_base: labels[%lld]=%u >= n_cls=%d",
                          (long long)i, base_labels[i], h->n_cls);
    }
    std::vector<int64_t> seg_start, seg_len;
    std::vector<uint32_t> grouped;
    const uint32_t* grouped_src = base_labels;  // no libraries: the labels are uploaded from the caller's buffer as they are
    h->h_order.clear();
    h->has_order = false;
    if (lib_codes && n_libs > 0) {
        // category order, ascending index inside a category: np.where(libraries == c)[0]  (gr/_utils.py:208-209)
        std::vector<int64_t> cnt(n_libs + 1, 0);
        for (int64_t i = 0; i < n; ++i) {
            SQB_CHECK(lib_codes[i] >= 0 && lib_codes[i] < n_libs, SQB_ERR_INVALID,
                      "sqb_nhood_set_base: lib_codes[%lld]=%d outside [0,%d) (NaN libraries are unsupported)",
                      (long long)i, lib_codes[i], n_libs);
            cnt[lib_codes[i] + 1]++;
        }
        for (int l = 0; l < n_libs; ++l) cnt[l + 1] += cnt[l];
        h->h_order.resize(n);
        grouped.resize(n);
        grouped_src = grouped.data();
        std::vector<int64_t> cur(cnt.begin(), cnt.end() - 1);
        for (int64_t i = 0; i < n; ++i) {
            int64_t k = cur[lib_codes[i]]++;
            h->h_order[k] = (uint32_t)i;
            grouped[k] = base_labels[i];
        }
        for (int l = 0; l < n_libs; ++l) {
            seg_start.push_back(cnt[l]);
            seg_len.push_back(cnt[l + 1] - cnt[l]);
        }
        h->has_order = true;
    } else {
        seg_start.push_back(0);
        seg_len.push_back(n);
    }
    h->nseg = (int)seg_start.size();
    h->h_seg_start = seg_start;
    h->h_seg_len = seg_len;
    h->philox_ready = false;
    SQB_TRY(h->d_seg_start.alloc(h->nseg));
    SQB_TRY(h->d_seg_len.alloc(h->nseg));
    SQB_TRY(h->d_tmp_u32.alloc(n));
    SQB_TRY(h->d_base.alloc((size_t)h->stride * h->lt_bytes));
    SQB_CUDA(cudaMemcpyAsync(h->d_seg_start.p, seg_start.data(), h->nseg * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    SQB_CUDA(cudaMemcpyAsync(h->d_seg_len.p, seg_len.data(), h->nseg * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    SQB_CUDA(cudaMemcpyAsync(h->d_tmp_u32.p, grouped_src, n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    if (h->has_order) {
        SQB_TRY(h->d_order.alloc(n));
        SQB_CUDA(cudaMemcpyAsync(h->d_order.p, h->h_order.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    }
    {
        SqbLaunchScope scope(c, SQB_K_MISC);
        unsigned g = (unsigned)ceil_div64(h->stride, 256);
        if (h->lt_bytes == 1)
            nhood_u32_to_lt_kernel<uint8_t><<<g, 256, 0, c->stream>>>(h->d_tmp_u32.p, h->d_base.p, n, h->stride);
        else
            nhood_u32_to_lt_kernel<uint16_t><<<g, 256, 0, c->stream>>>(h->d_tmp_u32.p, reinterpret_cast<uint16_t*>(h->d_base.p), n, h->stride);
        SQB_POST_LAUNCH();
    }
    SQB_CUDA(cudaStreamSynchronize(c->stream));  // host vectors go out of scope
    h->base_set = true;
    return SQB_OK;
}

int sqb_nhood_permute_upload(sqb_nhood* h, const uint64_t* states, int64_t n_perms) {
    SQB_CHECK(h && states, SQB_ERR_INVALID, "sqb_nhood_permute_upload: null argument");
    SQB_CHECK(n_perms >= 1, SQB_ERR_INVALID, "sqb_nhood_permute_upload: n_perms=%lld must be positive", (long long)n_perms);
    SQB_CHECK(h->base_set, SQB_ERR_STATE, "sqb_nhood_permute_upload: call sqb_nhood_set_base first");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    std::vector<uint64_t> packed((size_t)n_perms * 4);
    for (int64_t p = 0; p < n_perms; ++p) {
        SQB_CHECK(states[p * 6 + 4] == 0, SQB_ERR_UNSUPPORTED,
                  "sqb_nhood_permute: generator %lld has a buffered uint32 (has_uint32=1); only fresh generators are supported",
                  (long long)p);
        for (int k = 0; k < 4; ++k) packed[p * 4 + k] = states[p * 6 + k];
    }
    SQB_TRY(h->d_states.alloc((size_t)n_perms * 4));
    SQB_TRY(h->d_counts.alloc((size_t)n_perms * h->n_cls * h->n_cls));
    int64_t chunk = auto_chunk(h);
    if (chunk > ((n_perms + 31) / 32) * 32) chunk = ((n_perms + 31) / 32) * 32;
    SQB_TRY(ensure_buffers(h, chunk));
    SQB_CUDA(cudaMemcpyAsync(h->d_states.p, packed.data(), packed.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
    SQB_CUDA(cudaStreamSynchronize(c->stream));
    h->n_perms = n_perms;
    h->chunk = chunk;
    h->rng_mode = 0;
    h->uploaded = true;
    h->ran = false;
    return SQB_OK;
}

int sqb_nhood_permute_upload_philox(sqb_nhood* h, uint64_t seed, int64_t first_perm, int64_t n_perms) {
    SQB_CHECK(h, SQB_ERR_INVALID, "sqb_nhood_permute_upload_philox: null handle");
    SQB_CHECK(n_perms >= 1 && first_perm >= 0, SQB_ERR_INVALID, "sqb_nhood_permute_upload_philox: bad permutation range");
    SQB_CHECK(h->base_set, SQB_ERR_STATE, "sqb_nhood_permute_upload_philox: call sqb_nhood_set_base first");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    SQB_TRY(philox_prepare(h));
    SQB_TRY(h->d_counts.alloc((size_t)n_perms * h->n_cls * h->n_cls));
    int64_t chunk = auto_chunk(h);
    if (chunk > ((n_perms + 31) / 32) * 32) chunk = ((n_perms + 31) / 32) * 32;
    SQB_TRY(c->scratch[1].alloc((size_t)(h->n + 1) * chunk * h->lt_bytes));  // labT only: nothing permutation-major exists in this mode
    h->n_perms = n_perms;
    h->chunk = chunk;
    h->rng_mode = 1;
    h->philox_seed = seed;
    h->perm_first = first_perm;
    h->uploaded = true;
    h->ran = false;
    return SQB_OK;
}

int sqb_nhood_permute_run_async(sqb_nhood* h) {
    SQB_CHECK(h, SQB_ERR_INVALID, "sqb_nhood_permute_run_async: null handle");
    SQB_CHECK(h->uploaded, SQB_ERR_STATE, "sqb_nhood_permute_run_async: call sqb_nhood_permute_upload first");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int64_t CC = (int64_t)h->n_cls * h->n_cls;
    SQB_CUDA(cudaMemsetAsync(h->d_counts.p, 0, (size_t)h->n_perms * CC * sizeof(uint32_t), c->stream));
    // the chunk the upload sized the (context-owned) scratch buffers for; another plan on the same context may have
    // replaced them since: re-establish the sizes (no-op when they still fit)
    const int64_t chunk = h->chunk;
    if (h->rng_mode == 0)
        SQB_TRY(ensure_buffers(h, chunk));
    else
        SQB_TRY(c->scratch[1].alloc((size_t)(h->n + 1) * chunk * h->lt_bytes));
    for (int64_t p0 = 0; p0 < h->n_perms; p0 += chunk) {
        int64_t np = h->n_perms - p0 < chunk ? h->n_perms - p0 : chunk;
        if (h->rng_mode == 1) {
            if (h->lt_bytes == 1)
                SQB_TRY(run_chunk_philox<uint8_t>(h, p0, np));
            else
                SQB_TRY(run_chunk_philox<uint16_t>(h, p0, np));
        } else if (h->lt_bytes == 1) {
            SQB_TRY(run_chunk<uint8_t>(h, p0, np, true));
        } else {
            SQB_TRY(run_chunk<uint16_t>(h, p0, np, true));
        }
    }
    h->ran = true;
    return SQB_OK;
}

int sqb_nhood_permute_download(sqb_nhood* h, uint32_t* out_counts) {
    SQB_CHECK(h && out_counts, SQB_ERR_INVALID, "sqb_nhood_permute_download: null argument");
    SQB_CHECK(h->ran, SQB_ERR_STATE, "sqb_nhood_permute_download: nothing has run");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int64_t CC = (int64_t)h->n_cls * h->n_cls;
    SQB_CUDA(cudaMemcpyAsync(out_counts, h->d_counts.p, (size_t)h->n_perms * CC * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    SQB_CUDA(cudaStreamSynchronize(c->stream));
    return SQB_OK;
}

// ------------------------------------------------------------------------------------------------
// 5. per-bin mean and standard deviation over the permutations, in the exact operation order of the reference's
//    `perms.mean(axis=0)` / `perms.std(axis=0)` on the float64 copy of the counts (_nhood.py:231): numpy reduces axis 0 of a
//    C-contiguous array row by row (sequential adds per output element), std = sqrt(sum((x - mean)^2) / P).  Explicit
//    round-to-nearest intrinsics: no FMA contraction, so the doubles are bit-identical to numpy's.
// ------------------------------------------------------------------------------------------------
__global__ void nhood_stats_kernel(const uint32_t* __restrict__ counts, int64_t P, int CC, double* __restrict__ mean,
                                   double* __restrict__ stdv) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= CC) return;
    double s = 0.0;
    for (int64_t p = 0; p < P; ++p) s = __dadd_rn(s, (double)counts[p * CC + b]);
    const double m = __ddiv_rn(s, (double)P);
    double v = 0.0;
    for (int64_t p = 0; p < P; ++p) {
        const double x = __dsub_rn((double)counts[p * CC + b], m);
        v = __dadd_rn(v, __dmul_rn(x, x));
    }
    mean[b] = m;
    stdv[b] = __dsqrt_rn(__ddiv_rn(v, (double)P));
}

int sqb_nhood_permute_stats(sqb_nhood* h, double* mean_out, double* std_out) {
    SQB_CHECK(h && mean_out && std_out, SQB_ERR_INVALID, "sqb_nhood_permute_stats: null argument");
    SQB_CHECK(h->ran, SQB_ERR_STATE, "sqb_nhood_permute_stats: nothing has run");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int CC = h->n_cls * h->n_cls;
    DevBuf<double> d;
    d.bind(c->stream);
    SQB_TRY(d.alloc((size_t)2 * CC));
    {
        SqbLaunchScope scope(c, SQB_K_MISC);
        nhood_stats_kernel<<<(unsigned)ceil_div64(CC, 64), 64, 0, c->stream>>>(h->d_counts.p, h->n_perms, CC, d.p, d.p + CC);
    }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(mean_out, d.p, CC * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(std_out, d.p + CC, CC * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    d.release();
    if (e != cudaSuccess) {
        sqb_set_error("sqb_nhood_permute_stats: %s", cudaGetErrorString(e));
        return SQB_ERR_CUDA;
    }
    return SQB_OK;
}

// Multi-GPU form of the same statistics: the permutations are sharded contiguously over the ranks, so
//   * the per-bin SUMS are integers (< 2^53): exact in any order, all-reduced as int64 by the caller;
//   * the variance accumulation sum((x - mean)^2) is order dependent: every rank continues numpy's sequential accumulation
//     from the running value of the rank before it (one [C*C] float64 message per hop).
__global__ void nhood_sums_kernel(const uint32_t* __restrict__ counts, int64_t P, int CC, unsigned long long* __restrict__ sums) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= CC) return;
    unsigned long long s = 0ull;
    for (int64_t p = 0; p < P; ++p) s += counts[p * CC + b];
    sums[b] = s;
}

__global__ void nhood_var_chain_kernel(const uint32_t* __restrict__ counts, int64_t P, int CC, const double* __restrict__ mean,
                                       const double* __restrict__ acc_in, double* __restrict__ acc_out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= CC) return;
    const double m = mean[b];
    double v = acc_in[b];
    for (int64_t p = 0; p < P; ++p) {
        const double x = __dsub_rn((double)counts[p * CC + b], m);
        v = __dadd_rn(v, __dmul_rn(x, x));
    }
    acc_out[b] = v;
}

int sqb_nhood_permute_sums(sqb_nhood* h, int64_t* sums_out) {
    SQB_CHECK(h && sums_out, SQB_ERR_INVALID, "sqb_nhood_permute_sums: null argument");
    SQB_CHECK(h->ran, SQB_ERR_STATE, "sqb_nhood_permute_sums: nothing has run");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int CC = h->n_cls * h->n_cls;
    DevBuf<unsigned long long> d;
    d.bind(c->stream);
    SQB_TRY(d.alloc(CC));
    {
        SqbLaunchScope scope(c, SQB_K_MISC);
        nhood_sums_kernel<<<(unsigned)ceil_div64(CC, 64), 64, 0, c->stream>>>(h->d_counts.p, h->n_perms, CC, d.p);
    }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(sums_out, d.p, CC * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    d.release();
    if (e != cudaSuccess) {
        sqb_set_error("sqb_nhood_permute_sums: %s", cudaGetErrorString(e));
        return SQB_ERR_CUDA;
    }
    return SQB_OK;
}

int sqb_nhood_permute_var_chain(sqb_nhood* h, const double* mean, const double* acc_in, double* acc_out) {
    SQB_CHECK(h && mean && acc_in && acc_out, SQB_ERR_INVALID, "sqb_nhood_permute_var_chain: null argument");
    SQB_CHECK(h->ran, SQB_ERR_STATE, "sqb_nhood_permute_var_chain: nothing has run");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int CC = h->n_cls * h->n_cls;
    DevBuf<double> d;
    d.bind(c->stream);
    SQB_TRY(d.alloc((size_t)3 * CC));
    cudaError_t e = cudaMemcpyAsync(d.p, mean, CC * sizeof(double), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d.p + CC, acc_in, CC * sizeof(double), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        SqbLaunchScope scope(c, SQB_K_MISC);
        nhood_var_chain_kernel<<<(unsigned)ceil_div64(CC, 64), 64, 0, c->stream>>>(h->d_counts.p, h->n_perms, CC, d.p, d.p + CC, d.p + 2 * CC);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(acc_out, d.p + 2 * CC, CC * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    d.release();
    if (e != cudaSuccess) {
        sqb_set_error("sqb_nhood_permute_var_chain: %s", cudaGetErrorString(e));
        return SQB_ERR_CUDA;
    }
    return SQB_OK;
}

// Device-pointer forms of the statistics (asynchronous on the ctx stream; the caller owns the device buffers, e.g. torch
// tensors handed to NCCL): nothing crosses the PCIe bus between the count kernel and the collective.
int sqb_nhood_permute_stats_dev(sqb_nhood* h, double* d_mean, double* d_std) {
    SQB_CHECK(h && d_mean && d_std, SQB_ERR_INVALID, "sqb_nhood_permute_stats_dev: null argument");
    SQB_CHECK(h->ran, SQB_ERR_STATE, "sqb_nhood_permute_stats_dev: nothing has run");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int CC = h->n_cls * h->n_cls;
    SqbLaunchScope scope(c, SQB_K_MISC);
    nhood_stats_kernel<<<(unsigned)ceil_div64(CC, 64), 64, 0, c->stream>>>(h->d_counts.p, h->n_perms, CC, d_mean, d_std);
    SQB_POST_LAUNCH();
    return SQB_OK;
}

// Multi-GPU statistics by gathering: the per-permutation counts of this handle as a device array (asynchronous copy on the ctx
// stream into a caller-owned buffer, e.g. the padded block a torch all_gather_into_tensor sends) ...
int sqb_nhood_permute_counts_dev(sqb_nhood* h, uint32_t* d_dst) {
    SQB_CHECK(h && d_dst, SQB_ERR_INVALID, "sqb_nhood_permute_counts_dev: null argument");
    SQB_CHECK(h->ran, SQB_ERR_STATE, "sqb_nhood_permute_counts_dev: nothing has run");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const size_t bytes = (size_t)h->n_perms * h->n_cls * h->n_cls * sizeof(uint32_t);
    SQB_CUDA(cudaMemcpyAsync(d_dst, h->d_counts.p, bytes, cudaMemcpyDeviceToDevice, c->stream));
    return SQB_OK;
}

// ... and mean / std over the rows of ANY device array of counts [rows][n_cls * n_cls] (the gathered blocks of all ranks, rows in
// global permutation order): the same kernel as the single-GPU statistics, hence numpy's operation order.
int sqb_nhood_stats_rows_dev(sqb_ctx* ctx, const uint32_t* d_counts, int64_t rows, int n_cls, double* d_mean, double* d_std) {
    SQB_CHECK(ctx && d_counts && d_mean && d_std, SQB_ERR_INVALID, "sqb_nhood_stats_rows_dev: null argument");
    SQB_CHECK(rows >= 1 && n_cls >= 1, SQB_ERR_INVALID, "sqb_nhood_stats_rows_dev: rows=%lld, n_cls=%d", (long long)rows, n_cls);
    SQB_CUDA(cudaSetDevice(ctx->device));
    const int CC = n_cls * n_cls;
    SqbLaunchScope scope(ctx, SQB_K_MISC);
    nhood_stats_kernel<<<(unsigned)ceil_div64(CC, 64), 64, 0, ctx->stream>>>(d_counts, rows, CC, d_mean, d_std);
    SQB_POST_LAUNCH();
    return SQB_OK;
}

int sqb_nhood_permute_sums_dev(sqb_nhood* h, int64_t* d_sums) {
    SQB_CHECK(h && d_sums, SQB_ERR_INVALID, "sqb_nhood_permute_sums_dev: null argument");
    SQB_CHECK(h->ran, SQB_ERR_STATE, "sqb_nhood_permute_sums_dev: nothing has run");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int CC = h->n_cls * h->n_cls;
    SqbLaunchScope scope(c, SQB_K_MISC);
    nhood_sums_kernel<<<(unsigned)ceil_div64(CC, 64), 64, 0, c->stream>>>(h->d_counts.p, h->n_perms, CC,
                                                                           reinterpret_cast<unsigned long long*>(d_sums));
    SQB_POST_LAUNCH();
    return SQB_OK;
}

int sqb_nhood_permute_var_chain_dev(sqb_nhood* h, const double* d_mean, const double* d_acc_in, double* d_acc_out) {
    SQB_CHECK(h && d_mean && d_acc_in && d_acc_out, SQB_ERR_INVALID, "sqb_nhood_permute_var_chain_dev: null argument");
    SQB_CHECK(h->ran, SQB_ERR_STATE, "sqb_nhood_permute_var_chain_dev: nothing has run");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int CC = h->n_cls * h->n_cls;
    SqbLaunchScope scope(c, SQB_K_MISC);
    nhood_var_chain_kernel<<<(unsigned)ceil_div64(CC, 64), 64, 0, c->stream>>>(h->d_counts.p, h->n_perms, CC, d_mean, d_acc_in, d_acc_out);
    SQB_POST_LAUNCH();
    return SQB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// 6. ligrec permutation test (src/squidpy/gr/_ligrec.py:616-676 `_score_permutations`): per permutation the cluster labels
//    are shuffled with the SAME exact numpy-stream replay as above (numba's Generator.shuffle is numpy's), the per-cluster
//    mean expression of every gene is re-formed and every (interaction, cluster pair) whose shuffled score exceeds the
//    observed one counts one.  The reference accumulates groups[cl, g] += data[cell, g] over the cells in ascending order in
//    float64 and then multiplies by 1/size: the kernel keeps exactly that order (one lane owns one gene, the cells are walked
//    sequentially, accumulators [cluster][lane] in shared memory with bank == lane), so the scores and hence the `>`
//    decisions are bit-identical.
// ------------------------------------------------------------------------------------------------
template <typename LT>
__global__ void __launch_bounds__(128) ligrec_group_means_kernel(const LT* __restrict__ lab, int64_t stride,
                                                                 const double* __restrict__ data, int64_t n_cells, int n_genes,
                                                                 int n_cls, const double* __restrict__ inv_counts,
                                                                 double* __restrict__ G) {
    extern __shared__ double lg_acc[];  // [4 warps][n_cls][32]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p = blockIdx.y;
    const int g = (blockIdx.x * 4 + warp) * 32 + lane;
    double* __restrict__ acc = lg_acc + (size_t)warp * n_cls * 32 + lane;
    for (int k = 0; k < n_cls; ++k) acc[k * 32] = 0.0;
    const LT* __restrict__ row = lab + p * stride;
    const bool ok = g < n_genes;
    const double* __restrict__ col = data + (ok ? g : 0);
    int64_t c = 0;
    for (; c + 4 <= n_cells; c += 4) {
        const int l0 = (int)row[c], l1 = (int)row[c + 1], l2 = (int)row[c + 2], l3 = (int)row[c + 3];
        const double v0 = col[c * n_genes], v1 = col[(c + 1) * n_genes], v2 = col[(c + 2) * n_genes], v3 = col[(c + 3) * n_genes];
        acc[l0 * 32] = __dadd_rn(acc[l0 * 32], v0);
        acc[l1 * 32] = __dadd_rn(acc[l1 * 32], v1);
        acc[l2 * 32] = __dadd_rn(acc[l2 * 32], v2);
        acc[l3 * 32] = __dadd_rn(acc[l3 * 32], v3);
    }
    for (; c < n_cells; ++c) {
        const int l0 = (int)row[c];
        acc[l0 * 32] = __dadd_rn(acc[l0 * 32], col[c * n_genes]);
    }
    if (ok)
        for (int k = 0; k < n_cls; ++k) G[((size_t)p * n_cls + k) * n_genes + g] = __dmul_rn(acc[k * 32], inv_counts[k]);
}

__global__ void ligrec_compare_kernel(const double* __restrict__ G, int64_t np, int n_cls, int n_genes,
                                      const double* __restrict__ mean_obs, const int32_t* __restrict__ inter, int64_t n_inter,
                                      const int32_t* __restrict__ cpairs, int64_t n_cpairs, const uint8_t* __restrict__ valid,
                                      long long* __restrict__ counts) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_inter * n_cpairs || !valid[t]) return;
    const int64_t i = t / n_cpairs, j = t % n_cpairs;
    const int rec = inter[2 * i], lig = inter[2 * i + 1], a = cpairs[2 * j], b = cpairs[2 * j + 1];
    const double obs = __dadd_rn(mean_obs[(size_t)a * n_genes + rec], mean_obs[(size_t)b * n_genes + lig]);
    const size_t oa = (size_t)a * n_genes + rec, ob = (size_t)b * n_genes + lig, per = (size_t)n_cls * n_genes;
    long long cnt = 0;
    for (int64_t p = 0; p < np; ++p) cnt += __dadd_rn(G[p * per + oa], G[p * per + ob]) > obs ? 1 : 0;
    counts[t] += cnt;
}

extern "C" {

int sqb_ligrec_counts(sqb_nhood* h, const double* data, int64_t n_genes, const double* inv_counts, const double* mean_obs,
                      const int32_t* interactions, int64_t n_inter, const int32_t* inter_clusters, int64_t n_cpairs,
                      const uint8_t* valid, int64_t* out_counts) {
    SQB_CHECK(h && data && inv_counts && mean_obs && interactions && inter_clusters && valid && out_counts, SQB_ERR_INVALID,
              "sqb_ligrec_counts: null argument");
    SQB_CHECK(h->uploaded && h->rng_mode == 0, SQB_ERR_STATE, "sqb_ligrec_counts: upload numpy generator states first (sqb_nhood_permute_upload)");
    SQB_CHECK(!h->has_order, SQB_ERR_UNSUPPORTED, "sqb_ligrec_counts: library partitions are not part of the ligrec test");
    SQB_CHECK(n_genes >= 1 && n_genes < 2147483647LL && n_inter >= 1 && n_cpairs >= 1, SQB_ERR_INVALID, "sqb_ligrec_counts: bad sizes");
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    const int C = h->n_cls;
    const size_t smem = (size_t)4 * C * 32 * sizeof(double);
    SQB_CHECK(smem <= c->smem_optin, SQB_ERR_UNSUPPORTED, "sqb_ligrec_counts: %d clusters exceed the shared-memory accumulators", C);
    for (int64_t i = 0; i < n_inter * 2; ++i)
        SQB_CHECK(interactions[i] >= 0 && interactions[i] < n_genes, SQB_ERR_INVALID, "sqb_ligrec_counts: gene index %d out of range", interactions[i]);
    for (int64_t i = 0; i < n_cpairs * 2; ++i)
        SQB_CHECK(inter_clusters[i] >= 0 && inter_clusters[i] < C, SQB_ERR_INVALID, "sqb_ligrec_counts: cluster index %d out of range", inter_clusters[i]);
    const int64_t n = h->n, NT = n_inter * n_cpairs;
    // permutations per pass: the shuffled label rows (upload chunk) and the [perm][cluster][gene] means (<= 1 GB)
    int64_t chunk = h->chunk;
    const int64_t gcap = ((int64_t)1 << 30) / ((int64_t)C * n_genes * 8);
    if (chunk > gcap) chunk = gcap < 1 ? 1 : gcap;
    DevBuf<double> d_data, d_inv, d_obs, d_G;
    DevBuf<int32_t> d_inter, d_cp;
    DevBuf<uint8_t> d_valid;
    DevBuf<long long> d_cnt;
    auto cleanup = [&]() {
        d_data.release(), d_inv.release(), d_obs.release(), d_G.release(), d_inter.release(), d_cp.release(), d_valid.release(), d_cnt.release();
    };
    int rc;
    if ((rc = d_data.alloc((size_t)n * n_genes)) || (rc = d_inv.alloc(C)) || (rc = d_obs.alloc((size_t)C * n_genes)) ||
        (rc = d_G.alloc((size_t)chunk * C * n_genes)) || (rc = d_inter.alloc(2 * n_inter)) || (rc = d_cp.alloc(2 * n_cpairs)) ||
        (rc = d_valid.alloc(NT)) || (rc = d_cnt.alloc(NT)) || (rc = ensure_buffers(h, h->chunk))) {
        cleanup();
        return rc;
    }
    cudaError_t e = cudaMemsetAsync(d_cnt.p, 0, NT * sizeof(long long), c->stream);
    if (e == cudaSuccess && sqb_h2d(c, d_data.p, data, (size_t)n * n_genes * sizeof(double)) != SQB_OK) e = cudaErrorUnknown;
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_inv.p, inv_counts, C * sizeof(double), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_obs.p, mean_obs, (size_t)C * n_genes * sizeof(double), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_inter.p, interactions, 2 * n_inter * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_cp.p, inter_clusters, 2 * n_cpairs * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_valid.p, valid, NT, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess && smem > 48 * 1024) {
        e = cudaFuncSetAttribute(ligrec_group_means_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ligrec_group_means_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    for (int64_t p0 = 0; p0 < h->n_perms && e == cudaSuccess; p0 += chunk) {
        const int64_t np = h->n_perms - p0 < chunk ? h->n_perms - p0 : chunk;
        rc = h->lt_bytes == 1 ? run_chunk<uint8_t>(h, p0, np, false) : run_chunk<uint16_t>(h, p0, np, false);
        if (rc != SQB_OK) {
            cudaStreamSynchronize(c->stream);
            cleanup();
            return rc;
        }
        {
            SqbLaunchScope scope(c, SQB_K_MISC);
            dim3 grid((unsigned)ceil_div64(n_genes, 128), (unsigned)np);
            if (h->lt_bytes == 1)
                ligrec_group_means_kernel<uint8_t><<<grid, 128, smem, c->stream>>>(c->scratch[0].p, h->stride, d_data.p, n, (int)n_genes, C, d_inv.p, d_G.p);
            else
                ligrec_group_means_kernel<uint16_t><<<grid, 128, smem, c->stream>>>(reinterpret_cast<const uint16_t*>(c->scratch[0].p), h->stride,
                                                                                     d_data.p, n, (int)n_genes, C, d_inv.p, d_G.p);
        }
        {
            SqbLaunchScope scope(c, SQB_K_MISC);
            ligrec_compare_kernel<<<(unsigned)ceil_div64(NT, 256), 256, 0, c->stream>>>(d_G.p, np, C, (int)n_genes, d_obs.p, d_inter.p, n_inter, d_cp.p,
                                                                                        n_cpairs, d_valid.p, d_cnt.p);
        }
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_counts, d_cnt.p, NT * sizeof(long long), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    else cudaStreamSynchronize(c->stream);
    cleanup();
    if (e != cudaSuccess) {
        sqb_set_error("sqb_ligrec_counts: %s", cudaGetErrorString(e));
        return SQB_ERR_CUDA;
    }
    return SQB_OK;
}

int sqb_nhood_permute(sqb_nhood* h, const uint64_t* states, int64_t n_perms, uint32_t* out_counts) {
    SQB_TRY(sqb_nhood_permute_upload(h, states, n_perms));
    SQB_TRY(sqb_nhood_permute_run_async(h));
    return sqb_nhood_permute_download(h, out_counts);
}

int sqb_nhood_shuffled_labels(sqb_nhood* h, int64_t p0, int64_t p1, uint32_t* out) {
    SQB_CHECK(h && out, SQB_ERR_INVALID, "sqb_nhood_shuffled_labels: null argument");
    SQB_CHECK(h->uploaded, SQB_ERR_STATE, "sqb_nhood_shuffled_labels: call sqb_nhood_permute_upload first");
    SQB_CHECK(p0 >= 0 && p0 < p1 && p1 <= h->n_perms, SQB_ERR_INVALID, "sqb_nhood_shuffled_labels: bad range [%lld,%lld)",
              (long long)p0, (long long)p1);
    sqb_ctx* c = h->ctx;
    SQB_CUDA(cudaSetDevice(c->device));
    if (h->rng_mode == 1) {  // fast mode: 32 permutations at a time through labT[n][32]
        SQB_TRY(c->scratch[1].alloc((size_t)(h->n + 1) * h->chunk * h->lt_bytes));
        std::vector<uint8_t> host((size_t)h->n * 32 * h->lt_bytes);  // group 0 rows [0, n); row n is the spare row
        for (int64_t q0 = p0; q0 < p1; q0 += 32) {
            const int64_t np = p1 - q0 < 32 ? p1 - q0 : 32;
            if (h->lt_bytes == 1)
                SQB_TRY(philox_labels<uint8_t>(h, q0, np, c->scratch[1].p, 32));
            else
                SQB_TRY(philox_labels<uint16_t>(h, q0, np, reinterpret_cast<uint16_t*>(c->scratch[1].p), 32));
            SQB_CUDA(cudaMemcpyAsync(host.data(), c->scratch[1].p, host.size(), cudaMemcpyDeviceToHost, c->stream));
            SQB_CUDA(cudaStreamSynchronize(c->stream));
            for (int64_t p = 0; p < np; ++p) {
                uint32_t* row = out + (size_t)(q0 - p0 + p) * h->n;
                for (int64_t k = 0; k < h->n; ++k)
                    row[k] = h->lt_bytes == 1 ? host[(size_t)k * 32 + p] : reinterpret_cast<uint16_t*>(host.data())[(size_t)k * 32 + p];
            }
        }
        return SQB_OK;
    }
    SQB_TRY(ensure_buffers(h, h->chunk));
    const size_t row_bytes = (size_t)h->stride * h->lt_bytes;
    int64_t step = h->chunk;
    const int64_t cap = (int64_t)(c->scratch[0].n / row_bytes);
    if (step > cap) step = cap;
    SQB_CHECK(step >= 1, SQB_ERR_STATE, "sqb_nhood_shuffled_labels: label buffer not allocated");
    std::vector<uint8_t> host(row_bytes);
    for (int64_t q0 = p0; q0 < p1; q0 += step) {
        const int64_t np = p1 - q0 < step ? p1 - q0 : step;
        if (h->lt_bytes == 1)
            SQB_TRY(run_chunk<uint8_t>(h, q0, np, false));
        else
            SQB_TRY(run_chunk<uint16_t>(h, q0, np, false));
        for (int64_t p = 0; p < np; ++p) {
            SQB_CUDA(cudaMemcpyAsync(host.data(), c->scratch[0].p + (size_t)p * row_bytes, row_bytes, cudaMemcpyDeviceToHost,
                                     c->stream));
            SQB_CUDA(cudaStreamSynchronize(c->stream));
            uint32_t* row = out + (size_t)(q0 - p0 + p) * h->n;
            for (int64_t k = 0; k < h->n; ++k) {
                uint32_t v = h->lt_bytes == 1 ? host[k] : reinterpret_cast<uint16_t*>(host.data())[k];
                row[h->has_order ? h->h_order[k] : k] = v;
            }
        }
    }
    return SQB_OK;
}

}  // extern "C"
