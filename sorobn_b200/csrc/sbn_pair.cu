// sorobn_b200 -- paired steps: two eliminations per launch, the intermediate in registers (sbn_pair.h).
#include "sbn_pair.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "sbn_internal.h"
#include "sbn_kernels.cuh"
#include "sbn_launch.h"

namespace {

constexpr int kV = 2;  // evidence rows per thread (one 64-bit load / store per entry)

// eight consecutive coefficients (two 128-bit shared-memory loads)
__device__ __forceinline__ void pair_coef8(float (&c)[SBN_PAIR_PW], const float *s) {
    const float4 lo = *reinterpret_cast<const float4 *>(s);
    const float4 hi = *reinterpret_cast<const float4 *>(s + 4);
    c[0] = lo.x, c[1] = lo.y, c[2] = lo.z, c[3] = lo.w;
    c[4] = hi.x, c[5] = hi.y, c[6] = hi.z, c[7] = hi.w;
}

// this row's float offset into a canonical array
template <int V>
__device__ __forceinline__ void pair_ev_offsets(const SbnPairParams &p, const SbnPairEv &d, int b, int (&e)[V]) {
#pragma unroll
    for (int l = 0; l < V; ++l) e[l] = 0;
    for (int k = 0; k < d.n; ++k) {
        const uint8_t *col = p.ev + static_cast<int64_t>(d.col[k]) * p.ld_ev + b;
#pragma unroll
        for (int l = 0; l < V; ++l) e[l] += ((b + l < p.n_rows) ? min(static_cast<int>(col[l]), d.card[k] - 1) : 0) * d.stride[k];
    }
}

// One step on a register tile: acc[d0][d1] = sum_x in[x][d0] * coef[x][d0][d1]   (mode B: coef[x][d1]).
// `k` points at the main array of this tile, `e` holds the per-row offsets into it.
struct PairG {  // a batched coefficient operand (modes GB / GC): row pointer, tile base and pre-scaled strides
    const float *p;
    uint32_t base;
    uint32_t x[SBN_PAIR_T], d0[SBN_PAIR_T], d1[SBN_PAIR_T];
};

template <int MODE, int V>
__device__ __forceinline__ void pair_step(const float (&in)[SBN_PAIR_T][SBN_PAIR_T][V], float (&acc)[SBN_PAIR_T][SBN_PAIR_T][V],
                                          const float *k, const int (&e)[V], const PairG &G) {
    constexpr int T = SBN_PAIR_T, PW = SBN_PAIR_PW;
    // per-row coefficients that arrive one value (CE) or one row pair (GB / GC) at a time are kept as (row 0, row 1)
    // register pairs and go through the packed FFMA2; float4 loads (B, CU) fill four registers of ONE row, pairing
    // them up would cost more moves than the packed FMA saves
    constexpr bool PACKED = V == 2 && (MODE == SBN_PAIR_CE || MODE == SBN_PAIR_GB || MODE == SBN_PAIR_GC);
#pragma unroll
    for (int d0 = 0; d0 < T; ++d0)
#pragma unroll
        for (int d1 = 0; d1 < T; ++d1)
#pragma unroll
            for (int l = 0; l < V; ++l) acc[d0][d1][l] = 0.f;
#pragma unroll
    for (int x = 0; x < T; ++x) {
        float c[V][PW];   // [row][d1]   (B, CU)
        float cp[T][V];   // [d1][row]   (PACKED)
        if constexpr (MODE == SBN_PAIR_B) {
#pragma unroll
            for (int l = 0; l < V; ++l) pair_coef8(c[l], k + e[l] + x * PW);
        } else if constexpr (MODE == SBN_PAIR_GB) {
#pragma unroll
            for (int d1 = 0; d1 < T; ++d1) sbn_ldv<V>(cp[d1], G.p + (G.base + G.x[x] + G.d1[d1]));
        }
#pragma unroll
        for (int d0 = 0; d0 < T; ++d0) {
            if constexpr (MODE == SBN_PAIR_CU) {
                pair_coef8(c[0], k + (x * T + d0) * PW);  // no evidence axis: one broadcast serves every row
            } else if constexpr (MODE == SBN_PAIR_CE) {
#pragma unroll
                for (int d1 = 0; d1 < T; ++d1)
#pragma unroll
                    for (int l = 0; l < V; ++l) cp[d1][l] = k[e[l] + (x * T + d0) * T + d1];
            } else if constexpr (MODE == SBN_PAIR_GC) {
#pragma unroll
                for (int d1 = 0; d1 < T; ++d1) sbn_ldv<V>(cp[d1], G.p + (G.base + G.x[x] + G.d0[d0] + G.d1[d1]));
            }
#pragma unroll
            for (int d1 = 0; d1 < T; ++d1) {
                if constexpr (PACKED) {
                    sbn_fma2(acc[d0][d1], in[x][d0], cp[d1]);
                } else {
#pragma unroll
                    for (int l = 0; l < V; ++l)
                        acc[d0][d1][l] = fmaf(in[x][d0][l], c[MODE == SBN_PAIR_CU ? 0 : l][d1], acc[d0][d1][l]);
                }
            }
        }
    }
}

// Thread = V consecutive evidence rows x one combination r of the axes neither step touches.
//   step 1: mid[y][w] = sum_x c1[x][y][w] * pre1[x][y] * F[x][y]
//   step 2: out[w][z] = sum_y c2[y][w][z] * pre2[y][w] * mid[y][w]
// Coefficients past a real cardinality are zero, F indices past one are clamped: the loop nest is
// always T x T x T and only the stores are predicated.
// Five CTAs per SM (96 registers, a handful of spilled bytes): measured on B200, grid 100k rows, 2 / 3 / 4 / 5 / 6 / 8
// resident CTAs -> 2.65 / 2.65 / 2.57 / 2.52 / 2.60 / 2.92 ms per step.  (Four with a batched coefficient operand: its
// fifteen pre-scaled offsets would spill at 96 registers.)
template <int M1, int M2>
__global__ void __launch_bounds__(SBN_PAIR_ROWS / kV, (M1 >= SBN_PAIR_GB ? 4 : 5)) sbn_pair_kernel(const __grid_constant__ SbnPairParams p) {
    constexpr int T = SBN_PAIR_T, V = kV;
    extern __shared__ __align__(16) float s_canon[];
    __shared__ __align__(8) uint64_t s_bar;
    sbn_pdl_launch_dependents();

    const int rblock = blockIdx.x / p.n_chunks;
    const int chunk = blockIdx.x % p.n_chunks;
    if (threadIdx.x == 0) {
        sbn_mbar_init(&s_bar, 1);
        sbn_fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        sbn_mbar_expect_tx(&s_bar, static_cast<uint32_t>(p.canon_floats) * 4u);
        sbn_tma_bulk_g2s(s_canon, p.canon, static_cast<uint32_t>(p.canon_floats) * 4u, &s_bar);
    }

    const int b = (rblock * static_cast<int>(blockDim.x) + threadIdx.x) * V;
    const bool live = b < p.n_rows;
    int e1[V], e2[V], g1[V], g2[V];  // float offsets of this row's evidence combination: main 1 / 2, pre 1 / 2
    if (live) {
        pair_ev_offsets<V>(p, p.ev_main1, b, e1);
        pair_ev_offsets<V>(p, p.ev_main2, b, e2);
        pair_ev_offsets<V>(p, p.ev_pre1, b, g1);
        pair_ev_offsets<V>(p, p.ev_pre2, b, g2);
    }
    sbn_mbar_wait(&s_bar, 0);
    if (!live) return;
    sbn_pdl_wait();  // coefficients and evidence codes are not written by any launch of the run; F (and G) below are

    // element offsets fit 32 bits (sbn_pair_fits): strides are scaled by the row pitch once, an access then costs
    // one IADD3 and one IMAD.WIDE.U32
    const uint32_t ld = static_cast<uint32_t>(p.ld);
    const float *const fp = p.f + b;
    float *const op = p.out + b;
    uint32_t xs[T], ys[T], ow[T], oz[T];
#pragma unroll
    for (int d = 0; d < T; ++d) {
        xs[d] = static_cast<uint32_t>(min(d, p.cx - 1) * p.f_sx) * ld;
        ys[d] = static_cast<uint32_t>(min(d, p.cy - 1) * p.f_sy) * ld;
        ow[d] = static_cast<uint32_t>(d * p.o_sw) * ld;
        oz[d] = static_cast<uint32_t>(d * p.o_sz) * ld;
    }
    PairG G;
    G.p = p.g + b;
    G.base = 0;
    if constexpr (M1 == SBN_PAIR_GB || M1 == SBN_PAIR_GC) {
#pragma unroll
        for (int d = 0; d < T; ++d) {
            G.x[d] = static_cast<uint32_t>(d * p.g_x) * ld;
            G.d0[d] = static_cast<uint32_t>(d * p.g_y) * ld;
            G.d1[d] = static_cast<uint32_t>(d * p.g_w) * ld;
        }
    }
    const int t_begin = chunk * p.tiles_per_cta;
    const int t_end = min(p.n_tiles, t_begin + p.tiles_per_cta);

    for (int t = t_begin; t < t_end; ++t) {
        const int4 r0 = __ldg(reinterpret_cast<const int4 *>(p.tile_off) + 2 * t);
        const int4 r1 = __ldg(reinterpret_cast<const int4 *>(p.tile_off) + 2 * t + 1);
        const uint32_t ob = static_cast<uint32_t>(r0.x) * ld, fb = static_cast<uint32_t>(r0.y) * ld;

        // every entry of F this tile needs, in flight together
        float f[T][T][V];
#pragma unroll
        for (int x = 0; x < T; ++x)
#pragma unroll
            for (int y = 0; y < T; ++y) sbn_ldv<V>(f[x][y], fp + (fb + xs[x] + ys[y]));
        if (p.has_pre1) {
            const float *const k = s_canon + r1.x;
#pragma unroll
            for (int x = 0; x < T; ++x)
#pragma unroll
                for (int y = 0; y < T; ++y)
#pragma unroll
                    for (int l = 0; l < V; ++l) f[x][y][l] *= k[g1[l] + x * T + y];
        }
        float mid[T][T][V];
        if constexpr (M1 == SBN_PAIR_GB || M1 == SBN_PAIR_GC) G.base = static_cast<uint32_t>(r1.z) * ld;
        pair_step<M1, V>(f, mid, s_canon + r0.z, e1, G);
        if (p.has_pre2) {
            const float *const k = s_canon + r1.y;
#pragma unroll
            for (int y = 0; y < T; ++y)
#pragma unroll
                for (int w = 0; w < T; ++w)
#pragma unroll
                    for (int l = 0; l < V; ++l) mid[y][w][l] *= k[g2[l] + y * T + w];
        }
        float acc[T][T][V];
        pair_step<M2, V>(mid, acc, s_canon + r0.w, e2, G);

#pragma unroll
        for (int z = 0; z < T; ++z)
#pragma unroll
            for (int w = 0; w < T; ++w)
                if (w < p.cw && z < p.cz) sbn_stv<V>(op + (ob + ow[w] + oz[z]), acc[w][z]);
    }
}

// Expanding product + contraction (SbnTripleParams), the body kept for A/B comparisons and for the triples the staged
// body does not cover: thread = one evidence row x one combination of the untouched axes.
// threadIdx.y walks the digits of a tile axis only A carries (when there is one): the warps of a CTA then work on the
// same rows and the same entries of B and C at about the same time, and all but the first of them hit L1.
template <int MINB>
__global__ void __launch_bounds__(SBN_TRIPLE_THREADS, MINB) sbn_triple_kernel_l1(const __grid_constant__ SbnTripleParams p) {
    constexpr int T = SBN_PAIR_T;
    sbn_pdl_entry();
    const int rblock = blockIdx.x / p.n_chunks;
    const int chunk = blockIdx.x % p.n_chunks;
    const int b = rblock * static_cast<int>(blockDim.x) + threadIdx.x;
    if (b >= p.n_rows) return;
    // element offsets fit 32 bits (sbn_pair_fits): strides are scaled by the row pitch once
    const uint32_t ld = static_cast<uint32_t>(p.ld);
    const int g = threadIdx.y;
    const float *const ap = p.a + b + static_cast<uint32_t>(g * p.a_g) * ld;
    const float *const bp = p.b + b;
    const float *const cp = p.c + b;
    float *const op = p.out + b + static_cast<uint32_t>(g * p.o_g) * ld;
    uint32_t ak[T], aj[T], bj[T], bs[T], ck[T], cz[T];
#pragma unroll
    for (int d = 0; d < T; ++d) {
        ak[d] = static_cast<uint32_t>(d * p.a_k) * ld, aj[d] = static_cast<uint32_t>(d * p.a_j) * ld;
        bj[d] = static_cast<uint32_t>(d * p.b_j) * ld, bs[d] = static_cast<uint32_t>(d * p.b_s) * ld;
        ck[d] = static_cast<uint32_t>(d * p.c_k) * ld, cz[d] = static_cast<uint32_t>(d * p.c_z) * ld;
    }
    const uint32_t oz = static_cast<uint32_t>(p.o_z) * ld, os = static_cast<uint32_t>(p.o_s) * ld;
    const int t_begin = chunk * p.tiles_per_cta;
    const int t_end = min(p.n_tiles, t_begin + p.tiles_per_cta);
    for (int t = t_begin; t < t_end; ++t) {
        const int4 row = __ldg(reinterpret_cast<const int4 *>(p.tile_off) + t);
        float acc[T][T];  // [z][s]
#pragma unroll
        for (int z = 0; z < T; ++z)
#pragma unroll
            for (int s = 0; s < T; ++s) acc[z][s] = 0.f;
#pragma unroll 1
        for (int pp = 0; pp < T; ++pp) {
            // the 75 entries of this p, in flight together
            float A[T][T], B[T][T], C[T][T];  // A[k][j]  B[j][s]  C[k][z]
            const uint32_t a0 = static_cast<uint32_t>(row.y + pp * p.a_p) * ld, b0 = static_cast<uint32_t>(row.z + pp * p.b_p) * ld,
                           c0 = static_cast<uint32_t>(row.w + pp * p.c_p) * ld;
#pragma unroll
            for (int j = 0; j < T; ++j)
#pragma unroll
                for (int s = 0; s < T; ++s) B[j][s] = bp[b0 + bj[j] + bs[s]];
#pragma unroll
            for (int k = 0; k < T; ++k)
#pragma unroll
                for (int j = 0; j < T; ++j) A[k][j] = ap[a0 + ak[k] + aj[j]];
#pragma unroll
            for (int k = 0; k < T; ++k)
#pragma unroll
                for (int z = 0; z < T; ++z) C[k][z] = cp[c0 + ck[k] + cz[z]];
#pragma unroll
            for (int k = 0; k < T; ++k) {
                float n[T];  // N[k][s] = sum_j A[k][j] B[j][s]
#pragma unroll
                for (int s = 0; s < T; ++s) {
                    float v = A[k][0] * B[0][s];
#pragma unroll
                    for (int j = 1; j < T; ++j) v = fmaf(A[k][j], B[j][s], v);
                    n[s] = v;
                }
#pragma unroll
                for (int z = 0; z < T; ++z)
#pragma unroll
                    for (int s = 0; s < T; ++s) acc[z][s] = fmaf(C[k][z], n[s], acc[z][s]);
            }
        }
#pragma unroll
        for (int z = 0; z < T; ++z)
#pragma unroll
            for (int s = 0; s < T; ++s) __stcs(op + (static_cast<uint32_t>(row.x) * ld + z * oz + s * os), acc[z][s]);
    }
}

// packed fp32 product (mul.rn.f32x2 -> FMUL2): the first term of an inner product, as the scalar body's `a * b`
__device__ __forceinline__ void triple_mul2(float (&r)[2], const float (&a)[2], const float (&b)[2]) {
    unsigned long long ra, rb, rr;
    memcpy(&ra, a, 8);
    memcpy(&rb, b, 8);
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rr) : "l"(ra), "l"(rb));
    memcpy(r, &rr, 8);
}

__device__ __forceinline__ void triple_cp_async16(float *dst, const float *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sbn_smem_u32(dst)), "l"(src) : "memory");
}

// wait until at most `n` of this thread's cp.async groups are still in flight (the count must be an immediate)
__device__ __forceinline__ void triple_cp_async_wait(int n) {
    if (n <= 0) asm volatile("cp.async.wait_group 0;" ::: "memory");
    else if (n == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
    else asm volatile("cp.async.wait_group 2;" ::: "memory");
}

// Expanding product + contraction, staged (SbnTripleParams, sbn_pair.h).  A CTA walks row blocks of R = 32 rows
// (blockIdx.x, then every gridDim.x-th) and, per row block, p = 0 .. T-1: one "item" per (row block, p).  An item's
// operand entries -- A[g][k][j], B[t][j][s], C[t][k][z] for this p -- are staged as 128-byte runs (32 rows, rows
// innermost as in global memory) by cp.async into a ring of n_stages items, n_stages - 1 of them in flight while the
// CTA computes on the oldest.
// Thread = row pair rp (lane & 15) x slot (2 x warp + lane / 16) = (group digit g, tile t): the two half-warps read
// the same B and C entries (one wavefront each) and two entries of A (two wavefronts).  Per item it loads its 25 B
// entries into registers once, then per k: N[s] = sum_j A[k][j] B[j][s], acc[z][s] += C[k][z] N[s] -- the order of
// the scalar body, on (row b, row b + 1) register pairs (FMUL2 / FFMA2): the results are the same bits.
// Loads are whole 128-byte runs: the row pitch is a multiple of 32, so the last, ragged row block reads rows past
// n_rows inside the pitch and never stores them.
__global__ void __launch_bounds__(SBN_TRIPLE_MAX_THREADS, 1) sbn_triple_kernel(const __grid_constant__ SbnTripleParams p) {
    constexpr int T = SBN_PAIR_T, R = SBN_TRIPLE_ROWS;
    extern __shared__ __align__(128) float s_ring[];
    sbn_pdl_entry();
    const int G = p.group, NT = p.n_tiles, S = p.n_stages;
    const int nA = G * T * T, nB = NT * T * T, nE = nA + 2 * nB;
    const uint32_t ld = static_cast<uint32_t>(p.ld);
    const int4 *const tiles = reinterpret_cast<const int4 *>(p.tile_off);
    // element offset (scaled by the row pitch; fits 32 bits: sbn_pair_fits) of every staged entry, per p
    uint32_t *const s_off = reinterpret_cast<uint32_t *>(s_ring + S * nE * R);
    for (int i = threadIdx.x; i < T * nE; i += blockDim.x) {
        const int pp = i / nE, e = i % nE;
        int off;
        if (e < nA) {
            off = __ldg(tiles).y + pp * p.a_p + (e / (T * T)) * p.a_g + (e / T % T) * p.a_k + (e % T) * p.a_j;
        } else if (e < nA + nB) {
            const int f = e - nA;
            off = __ldg(tiles + f / (T * T)).z + pp * p.b_p + (f / T % T) * p.b_j + (f % T) * p.b_s;
        } else {
            const int f = e - nA - nB;
            off = __ldg(tiles + f / (T * T)).w + pp * p.c_p + (f / T % T) * p.c_k + (f % T) * p.c_z;
        }
        s_off[i] = static_cast<uint32_t>(off) * ld;
    }
    __syncthreads();

    const int n_rb = (p.n_rows + R - 1) / R;
    const int n_items = (n_rb - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x) * T;
    auto issue = [&](int it) {
        if (it < n_items) {
            const uint32_t row0 = (blockIdx.x + static_cast<uint32_t>(it / T) * gridDim.x) * R;
            const uint32_t *const off = s_off + (it % T) * nE;
            float *const dst = s_ring + (it % S) * nE * R;
#pragma unroll 4
            for (int c = threadIdx.x; c < nE * 8; c += blockDim.x) {
                const int e = c >> 3, q = (c & 7) * 4;
                const float *const src = e < nA ? p.a : (e < nA + nB ? p.b : p.c);
                triple_cp_async16(dst + e * R + q, src + (off[e] + row0 + q));
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");  // empty past the last item: the group count stays uniform
    };

    const int lane = threadIdx.x & 31, rp = lane & 15;
    const int slot = 2 * (threadIdx.x >> 5) + (lane >> 4);
    const bool active = slot < G * NT;
    const int g = active ? slot % G : 0, t = active ? slot / G : 0;
    const int sa = g * T * T * R + 2 * rp, sb = (nA + t * T * T) * R + 2 * rp, sc = (nA + nB + t * T * T) * R + 2 * rp;
    float *const op = p.out + static_cast<uint32_t>(__ldg(tiles + t).x + g * p.o_g) * ld;
    const uint32_t oz = static_cast<uint32_t>(p.o_z) * ld, os = static_cast<uint32_t>(p.o_s) * ld;

    float acc[T][T][2];  // [z][s][row]
#pragma unroll
    for (int z = 0; z < T; ++z)
#pragma unroll
        for (int s = 0; s < T; ++s) acc[z][s][0] = acc[z][s][1] = 0.f;
    for (int i = 0; i < S - 1; ++i) issue(i);
#pragma unroll 1
    for (int it = 0; it < n_items; ++it) {
        triple_cp_async_wait(S - 2);  // this thread's copies of item `it` have landed ...
        __syncthreads();              // ... everyone's, and every thread is done with item it - 1, whose stage is refilled now
        issue(it + S - 1);
        if (active) {
            const float *const st = s_ring + (it % S) * nE * R;
            float bv[T][T][2];  // B[j][s]
#pragma unroll
            for (int j = 0; j < T; ++j)
#pragma unroll
                for (int s = 0; s < T; ++s) sbn_ldv<2>(bv[j][s], st + sb + (j * T + s) * R);
#pragma unroll
            for (int k = 0; k < T; ++k) {
                float n[T][2], a[2];  // N[k][s] = sum_j A[k][j] B[j][s]
                sbn_ldv<2>(a, st + sa + k * T * R);
#pragma unroll
                for (int s = 0; s < T; ++s) triple_mul2(n[s], a, bv[0][s]);
#pragma unroll
                for (int j = 1; j < T; ++j) {
                    sbn_ldv<2>(a, st + sa + (k * T + j) * R);
#pragma unroll
                    for (int s = 0; s < T; ++s) sbn_fma2(n[s], a, bv[j][s]);
                }
#pragma unroll
                for (int z = 0; z < T; ++z) {
                    float c[2];
                    sbn_ldv<2>(c, st + sc + (k * T + z) * R);
#pragma unroll
                    for (int s = 0; s < T; ++s) sbn_fma2(acc[z][s], c, n[s]);
                }
            }
        }
        if (it % T == T - 1) {
            const int b = (blockIdx.x + (it / T) * gridDim.x) * R + 2 * rp;
            if (active && b < p.n_rows) {
                float *const o = op + b;
#pragma unroll
                for (int z = 0; z < T; ++z)
#pragma unroll
                    for (int s = 0; s < T; ++s) {
                        if (b + 1 < p.n_rows) sbn_stv<2>(o + (z * oz + s * os), acc[z][s]);
                        else __stcs(o + (z * oz + s * os), acc[z][s][0]);
                    }
            }
#pragma unroll
            for (int z = 0; z < T; ++z)
#pragma unroll
                for (int s = 0; s < T; ++s) acc[z][s][0] = acc[z][s][1] = 0.f;
        }
    }
}

// staged body: p-slices in the shared-memory ring, CTA size (16 row pairs x the (group digit, tile) slots, two per
// warp) and dynamic shared memory (the ring + the per-p entry offsets)
int triple_stages() {
    static const int v = [] {
        const char *e = getenv("SOROBN_B200_TRIPLE_STAGES");
        const int s = e ? atoi(e) : 3;
        return std::min(std::max(s, 2), SBN_TRIPLE_MAX_STAGES);
    }();
    return v;
}
int triple_threads(const SbnTripleParams &q) { return 32 * ((q.group * q.n_tiles + 1) / 2); }
int triple_entries(const SbnTripleParams &q) { return (q.group + 2 * q.n_tiles) * SBN_PAIR_T * SBN_PAIR_T; }
int triple_smem(const SbnTripleParams &q) {
    return triple_entries(q) * (q.n_stages * SBN_TRIPLE_ROWS + SBN_PAIR_T) * 4;
}
constexpr int kTripleSmemMax = SBN_TRIPLE_MAX_ENTRIES * (SBN_TRIPLE_MAX_STAGES * SBN_TRIPLE_ROWS + SBN_PAIR_T) * 4;

void launch_modes(const SbnPair &pr, const SbnPairParams &q, unsigned grid, size_t smem, cudaStream_t stream) {
    const dim3 g(grid), b(SBN_PAIR_ROWS / kV);
#define SBN_PAIR_CASE(A, B)                                          \
    case A * 3 + B:                                                  \
        sbn_launch(sbn_pair_kernel<A, B>, g, b, smem, stream, q);    \
        break;
    switch (pr.m1 * 3 + pr.m2) {
        SBN_PAIR_CASE(0, 0)
        SBN_PAIR_CASE(0, 1)
        SBN_PAIR_CASE(0, 2)
        SBN_PAIR_CASE(1, 0)
        SBN_PAIR_CASE(1, 1)
        SBN_PAIR_CASE(1, 2)
        SBN_PAIR_CASE(2, 0)
        SBN_PAIR_CASE(2, 1)
        SBN_PAIR_CASE(2, 2)
        SBN_PAIR_CASE(3, 0)
        SBN_PAIR_CASE(3, 1)
        SBN_PAIR_CASE(3, 2)
        SBN_PAIR_CASE(4, 0)
        SBN_PAIR_CASE(4, 1)
        SBN_PAIR_CASE(4, 2)
    }
#undef SBN_PAIR_CASE
}

// axis of a factor with cardinalities `cards` (axis 0 fastest, dense) whose entry stride is `stride`
int axis_of_stride(const std::vector<int> &cards, int stride) {
    int64_t acc = 1;
    for (size_t j = 0; j < cards.size(); ++j) {
        if (acc == stride && cards[j] > 1) return static_cast<int>(j);
        acc *= cards[j];
    }
    return -1;
}

struct HostTables {
    std::vector<float> cpt;                  // copy of sbn_program::d_tables
    std::vector<std::vector<float>> slot;    // copies of the unbatched slots, fetched on demand
};

const float *host_table(sbn_program *P, HostTables &H, const InDesc &in, cudaError_t *err) {
    if (!in.is_slot) return H.cpt.data() + P->tables[in.id].first;
    if (H.slot.size() < P->slots.size()) H.slot.resize(P->slots.size());
    std::vector<float> &v = H.slot[in.id];
    if (v.empty()) {
        v.resize(static_cast<size_t>(P->slots[in.id].size));
        *err = cudaMemcpy(v.data(), P->slots[in.id].ptr, v.size() * 4, cudaMemcpyDeviceToHost);
    }
    return v.data();
}

// Some of one step's tables multiplied into one canonical array.
enum Layout { kLayoutB, kLayoutCU, kLayoutCE, kLayoutPre };
struct CanonSpec {
    std::vector<const InDesc *> tabs;
    std::vector<const float *> data;
    Layout layout = kLayoutB;
    int x_card = 1, d0_card = 1, d1_card = 1;
    int d0_axis = -1, d1_axis = -1;          // axes of the step's own output
    std::vector<int> r_axes;                 // axes (of the step's own output) of the untouched variables the tables carry
    std::vector<int> r_cards;
    std::vector<EvAxis> cols;                // distinct evidence columns (stride = canonical float stride)
    int64_t slab = 0, n_r = 1, n_e = 1;
    int64_t floats() const { return tabs.empty() ? 0 : round_up(slab * n_r * n_e, 4); }
};

void fill_canon(const CanonSpec &cs, float *dst) {
    constexpr int T = SBN_PAIR_T, PW = SBN_PAIR_PW;
    if (cs.tabs.empty()) return;
    const bool has_d0 = cs.layout != kLayoutB, has_d1 = cs.layout != kLayoutPre;
    const int n_d1 = !has_d1 ? 1 : (cs.layout == kLayoutCE ? T : PW);
    std::vector<int> ecode(cs.cols.size(), 0), rd(cs.r_axes.size(), 0);
    for (int64_t e = 0; e < cs.n_e; ++e) {
        int64_t rem = e;
        for (size_t k = 0; k < cs.cols.size(); ++k) ecode[k] = static_cast<int>(rem % cs.cols[k].card), rem /= cs.cols[k].card;
        for (int64_t r = 0; r < cs.n_r; ++r) {
            rem = r;
            for (size_t k = 0; k < cs.r_axes.size(); ++k) rd[k] = static_cast<int>(rem % cs.r_cards[k]), rem /= cs.r_cards[k];
            float *slab = dst + (e * cs.n_r + r) * cs.slab;
            for (int x = 0; x < T; ++x)
                for (int d0 = 0; d0 < (has_d0 ? T : 1); ++d0)
                    for (int d1 = 0; d1 < n_d1; ++d1) {
                        double v = 0.0;
                        if (x < cs.x_card && (!has_d0 || d0 < cs.d0_card) && (!has_d1 || d1 < cs.d1_card)) {
                            v = 1.0;
                            for (size_t j = 0; j < cs.tabs.size(); ++j) {
                                const InDesc &in = *cs.tabs[j];
                                int64_t off = static_cast<int64_t>(x) * in.estrides[0];
                                if (has_d0) off += static_cast<int64_t>(d0) * in.strides[cs.d0_axis];
                                if (has_d1) off += static_cast<int64_t>(d1) * in.strides[cs.d1_axis];
                                for (size_t k = 0; k < cs.r_axes.size(); ++k) off += static_cast<int64_t>(rd[k]) * in.strides[cs.r_axes[k]];
                                for (const EvAxis &a : in.ev)
                                    for (size_t k = 0; k < cs.cols.size(); ++k)
                                        if (cs.cols[k].col == a.col) off += static_cast<int64_t>(std::min(ecode[k], a.card - 1)) * a.stride;
                                v *= static_cast<double>(cs.data[j][off]);
                            }
                        }
                        slab[((has_d0 ? x * T + d0 : x) * n_d1) + d1] = static_cast<float>(v);
                    }
        }
    }
}

// Sizes the canonical array of `cs->tabs` (already chosen) for the given layout.
bool size_canon(const StepDesc &st, const std::vector<int> &r_axes, CanonSpec *cs) {
    constexpr int T = SBN_PAIR_T, PW = SBN_PAIR_PW;
    if (cs->tabs.empty()) return true;
    for (const InDesc *in : cs->tabs)
        for (const EvAxis &a : in->ev) {
            bool seen = false;
            for (EvAxis &c : cs->cols)
                if (c.col == a.col) c.card = std::max(c.card, a.card), seen = true;
            if (!seen) cs->cols.push_back({a.col, 0, a.card});
        }
    if (cs->cols.size() > SBN_PAIR_MAX_EV) return false;
    for (int ax : r_axes)
        for (const InDesc *in : cs->tabs)
            if (in->strides[ax] != 0) {
                cs->r_axes.push_back(ax);
                cs->r_cards.push_back(st.cards[ax]);
                break;
            }
    switch (cs->layout) {
        // float4 layouts: rows of a warp gather from the slabs of their own evidence combinations; an odd number
        // of 16-byte chunks per slab spreads neighbouring combinations over different shared-memory banks
        case kLayoutB: cs->slab = T * PW + 4; break;
        case kLayoutCU: cs->slab = T * T * PW; break;
        // scalar layouts: odd slabs, so combinations e and e + 1 start in different banks
        case kLayoutCE: cs->slab = T * T * T; break;
        case kLayoutPre: cs->slab = T * T; break;
    }
    for (int c : cs->r_cards) cs->n_r *= c;
    for (EvAxis &c : cs->cols) {
        c.stride = static_cast<int>(cs->n_e * cs->n_r * cs->slab);
        cs->n_e *= c.card;
        if (cs->n_e * cs->n_r * cs->slab > SBN_PAIR_SMEM_MAX / 4) return false;
    }
    return true;
}

// Splits the tables of one step (every input but `skip`) into the main coefficient array and the
// optional per-row pre factor, and sizes both.
bool spec_step(const StepDesc &st, int skip, int d0_axis, int d1_axis, const std::vector<int> &r_axes, CanonSpec *main,
               CanonSpec *pre) {
    for (CanonSpec *cs : {main, pre}) {
        cs->d0_axis = d0_axis;
        cs->d1_axis = d1_axis;
        cs->x_card = st.ecards[0];
        cs->d0_card = st.cards[d0_axis];
        cs->d1_card = st.cards[d1_axis];
    }
    std::vector<const InDesc *> all;
    for (int i = 0; i < static_cast<int>(st.in.size()); ++i) {
        if (i == skip) continue;
        if (st.in[i].batched) return false;
        all.push_back(&st.in[i]);
    }
    if (all.empty()) return false;
    // evidence tables without the second tile axis can leave the main array ...
    for (const InDesc *in : all) (in->ev.empty() || in->strides[d1_axis] != 0 ? main->tabs : pre->tabs).push_back(in);
    bool main_ev = false;
    for (const InDesc *in : main->tabs) main_ev = main_ev || !in->ev.empty();
    // ... which pays when what stays is evidence-free (a broadcast) or lacks the first tile axis (10 loads, not 125)
    bool main_d0 = false;
    for (const InDesc *in : main->tabs) main_d0 = main_d0 || in->strides[d0_axis] != 0;
    if (main->tabs.empty() || (main_ev && main_d0)) {
        main->tabs = all;
        pre->tabs.clear();
        main_ev = main_d0 = false;
        for (const InDesc *in : all) main_ev = main_ev || !in->ev.empty(), main_d0 = main_d0 || in->strides[d0_axis] != 0;
    }
    main->layout = !main_d0 ? kLayoutB : (main_ev ? kLayoutCE : kLayoutCU);
    pre->layout = kLayoutPre;
    return size_canon(st, r_axes, main) && size_canon(st, r_axes, pre);
}

int mode_of(Layout l) { return l == kLayoutB ? SBN_PAIR_B : (l == kLayoutCU ? SBN_PAIR_CU : SBN_PAIR_CE); }

void set_ev(SbnPairEv *d, const CanonSpec &cs) {
    d->n = static_cast<int32_t>(cs.tabs.empty() ? 0 : cs.cols.size());
    for (int k = 0; k < d->n; ++k) d->col[k] = cs.cols[k].col, d->stride[k] = cs.cols[k].stride, d->card[k] = cs.cols[k].card;
}

// float offset of tile `dig` (digits of the untouched axes `r`, as axes of the step's own output) inside a canonical array
int64_t tile_slab(const CanonSpec &cs, const std::vector<int> &r, const std::vector<int> &dig) {
    int64_t o = 0, m = 1;
    for (size_t k = 0; k < cs.r_axes.size(); ++k)
        for (size_t j = 0; j < r.size(); ++j)
            if (r[j] == cs.r_axes[k]) o += dig[j] * m, m *= cs.r_cards[k];
    return o * cs.slab;
}

// The expanding-product pattern (sbn_pair.h, SbnTripleParams) for two consecutive launched steps; appends the tile table.
SbnPair *plan_triple(sbn_program *P, int i1, int i2, std::vector<int32_t> *tiles) {
    constexpr int T = SBN_PAIR_T;
    const StepDesc &s1 = P->steps[i1], &s2 = P->steps[i2];
    if (s1.kind != 1 || s2.kind != 1 || s1.ecards.size() != 1 || s2.ecards.size() != 2) return nullptr;
    if (s1.in.size() != 2 || s2.in.size() != 2 || s1.ecards[0] != T || s2.ecards[0] != T || s2.ecards[1] != T) return nullptr;
    for (const InDesc &in : s1.in)
        if (!in.batched || !in.is_slot || !in.ev.empty()) return nullptr;
    for (const InDesc &in : s2.in)
        if (!in.batched || !in.is_slot || !in.ev.empty()) return nullptr;
    int mi = -1;
    for (int i = 0; i < 2; ++i)
        if (s2.in[i].id == s1.out_slot) mi = i;
    if (mi < 0 || s2.in[1 - mi].id == s1.out_slot || s1.out_slot == P->post_slot) return nullptr;
    const InDesc &M = s2.in[mi], &C = s2.in[1 - mi];
    // the two variables step 2 sums out, as axes of the intermediate
    const int je[2] = {axis_of_stride(s1.cards, M.estrides[0]), axis_of_stride(s1.cards, M.estrides[1])};
    if (je[0] < 0 || je[1] < 0 || je[0] == je[1]) return nullptr;
    // k: summed out by step 2, carried by exactly one operand of step 1 (that operand is "A"); p: the other one
    int ai = -1, kk = -1;
    for (int e = 0; e < 2 && ai < 0; ++e)
        for (int i = 0; i < 2; ++i)
            if (s1.in[i].strides[je[e]] != 0 && s1.in[1 - i].strides[je[e]] == 0) ai = i, kk = e;
    if (ai < 0) return nullptr;
    const InDesc &A = s1.in[ai], &B = s1.in[1 - ai];
    const int jk = je[kk], jp = je[1 - kk];
    if (A.estrides[0] == 0 || B.estrides[0] == 0) return nullptr;
    // output axes: s = carried by B only, z = new in step 2 (C only); everything else is a tile axis
    const int n2 = static_cast<int>(s2.cards.size());
    std::vector<int> to1(n2, -1);
    int ks = -1, kz = -1;
    for (int k = 0; k < n2; ++k) {
        if (M.strides[k] == 0) {
            if (kz < 0 && s2.cards[k] == T && C.strides[k] != 0) kz = k;
            continue;
        }
        to1[k] = axis_of_stride(s1.cards, M.strides[k]);
        if (to1[k] < 0 || to1[k] == jk || to1[k] == jp || s1.cards[to1[k]] != s2.cards[k]) return nullptr;
        if (ks < 0 && s2.cards[k] == T && A.strides[to1[k]] == 0 && B.strides[to1[k]] != 0 && C.strides[k] == 0) ks = k;
    }
    if (ks < 0 || kz < 0) return nullptr;
    const int out_slot = s2.out_slot;
    if (out_slot == A.id || out_slot == B.id || out_slot == C.id) return nullptr;
    // a tile axis only A carries (T states) is walked inside the thread: B and C are loaded once for its T tiles
    static const bool grouped = [] {
        const char *e = getenv("SOROBN_B200_TRIPLE_GROUP");
        return e ? atoi(e) != 0 : true;
    }();
    int kg = -1;
    for (int k = 0; k < n2 && grouped && kg < 0; ++k)
        if (k != ks && k != kz && to1[k] >= 0 && s2.cards[k] == T && A.strides[to1[k]] != 0 && B.strides[to1[k]] == 0 &&
            C.strides[k] == 0)
            kg = k;
    int64_t n_tiles = 1;
    std::vector<int> r2;
    for (int k = 0; k < n2; ++k)
        if (k != ks && k != kz && k != kg) r2.push_back(k), n_tiles *= s2.cards[k];
    if (n_tiles >= (1LL << 27)) return nullptr;

    SbnPair *pr = new SbnPair();
    memset(&pr->q, 0, sizeof pr->q);
    memset(&pr->t, 0, sizeof pr->t);
    pr->kind = 1;
    pr->step1 = i1, pr->step2 = i2;
    pr->g_in = -1;
    pr->a_in = ai, pr->b_in = 1 - ai, pr->c_in = 1 - mi;
    pr->tile_off_pos = static_cast<int64_t>(tiles->size());
    SbnTripleParams &q = pr->t;
    q.n_tiles = static_cast<int32_t>(n_tiles);
    q.a_j = A.estrides[0], q.a_k = A.strides[jk], q.a_p = A.strides[jp];
    q.b_j = B.estrides[0], q.b_s = B.strides[to1[ks]], q.b_p = B.strides[jp];
    q.c_k = C.estrides[kk], q.c_p = C.estrides[1 - kk], q.c_z = C.strides[kz];
    int64_t os = 1;
    std::vector<int64_t> os2(n2);
    for (int k = 0; k < n2; ++k) os2[k] = os, os *= s2.cards[k];
    q.o_z = static_cast<int32_t>(os2[kz]);
    q.o_s = static_cast<int32_t>(os2[ks]);
    q.group = kg >= 0 ? T : 1;
    q.o_g = kg >= 0 ? static_cast<int32_t>(os2[kg]) : 0;
    q.a_g = kg >= 0 ? A.strides[to1[kg]] : 0;
    std::vector<int> dig(r2.size(), 0);
    for (int64_t t = 0; t < n_tiles; ++t) {
        int64_t ob = 0, ab = 0, bb = 0, cb = 0;
        for (size_t k = 0; k < r2.size(); ++k) {
            const int ax = r2[k];
            ob += dig[k] * os2[ax];
            cb += static_cast<int64_t>(dig[k]) * C.strides[ax];
            if (to1[ax] >= 0) {
                ab += static_cast<int64_t>(dig[k]) * A.strides[to1[ax]];
                bb += static_cast<int64_t>(dig[k]) * B.strides[to1[ax]];
            }
        }
        tiles->push_back(static_cast<int32_t>(ob));
        tiles->push_back(static_cast<int32_t>(ab));
        tiles->push_back(static_cast<int32_t>(bb));
        tiles->push_back(static_cast<int32_t>(cb));
        for (size_t k = 0; k < dig.size(); ++k) {
            if (++dig[k] < s2.cards[r2[k]]) break;
            dig[k] = 0;
        }
    }
    // the staged body: A's entries must not depend on the tile (they are staged once for all tiles), and one p-slice
    // of A, B and C must fit SBN_TRIPLE_MAX_ENTRIES
    bool staged = (q.group + 2 * n_tiles) * T * T <= SBN_TRIPLE_MAX_ENTRIES;
    for (int64_t t = 1; t < n_tiles && staged; ++t) staged = (*tiles)[pr->tile_off_pos + 4 * t + 1] == (*tiles)[pr->tile_off_pos + 1];
    pr->staged_ctas = staged ? 1 : 0;  // the real count: triple_capacity
    q.n_stages = triple_stages();
    return pr;
}

// CTAs of the staged body that are resident at once on P's device (its launches are one wave of them)
cudaError_t triple_capacity(sbn_program *P, SbnPair *pr) {
    int per_sm = 0, n_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sbn_triple_kernel, triple_threads(pr->t),
                                                                  triple_smem(pr->t));
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, P->device);
    if (e == cudaSuccess && per_sm < 1) e = cudaErrorInvalidConfiguration;
    pr->staged_ctas = per_sm * n_sm;
    return e;
}

}  // namespace

cudaError_t sbn_pair_set_attrs() {
    // the pair kernel takes 40 KB of dynamic shared memory at most: below the 48 KB every kernel may use without
    // opting in; the staged triple body's ring takes up to 195 KB
    return cudaFuncSetAttribute(sbn_triple_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTripleSmemMax);
}

void sbn_pair_free(sbn_program *P) {
    for (SbnPair *pr : P->pairs) delete pr;
    P->pairs.clear();
    P->pair_first.clear();
    cudaFree(P->d_pair_canon);
    cudaFree(P->d_pair_tiles);
    P->d_pair_canon = nullptr;
    P->d_pair_tiles = nullptr;
}

cudaError_t sbn_pair_plan(sbn_program *P) {
    constexpr int T = SBN_PAIR_T;
    P->pair_first.assign(P->steps.size(), -1);
    if (P->mode != 1 || P->f64) return cudaSuccess;
    static const int min_card = [] {
        const char *e = getenv("SOROBN_B200_PAIR_MIN_CARD");
        return e ? atoi(e) : 4;
    }();

    static const bool triples_on = [] {
        const char *e = getenv("SOROBN_B200_TRIPLE");
        return e ? atoi(e) != 0 : true;
    }();

    HostTables H;
    std::vector<float> canon;
    std::vector<int32_t> tiles;
    cudaError_t err = cudaSuccess;
    bool fetched = false;

    const int n_steps = static_cast<int>(P->steps.size());
    auto launched = [&](int i) { return P->steps[i].kind != 0; };  // table steps ran when the program was created
    P->pairs_avoid_segments = P->use_chain && !P->segments.empty();
    auto in_segment = [&](int i) { return P->pairs_avoid_segments && P->seg_first[i] != -1; };
    for (int i1 = 0; i1 < n_steps; ++i1) {
        if (!launched(i1) || P->pair_first[i1] != -1) continue;
        int i2 = i1 + 1;
        while (i2 < n_steps && !launched(i2)) ++i2;
        if (i2 >= n_steps) break;
        if (in_segment(i1) || in_segment(i2)) continue;
        const StepDesc &s1 = P->steps[i1], &s2 = P->steps[i2];
        if (triples_on) {
            if (SbnPair *tr = plan_triple(P, i1, i2, &tiles)) {
                P->pair_first[i1] = static_cast<int>(P->pairs.size());
                P->pair_first[i2] = -2;
                P->pairs.push_back(tr);
                if (tr->staged_ctas && (err = triple_capacity(P, tr)) != cudaSuccess) return err;
                continue;
            }
        }
        if (s1.kind != 1 || s2.kind != 1 || s1.ecards.size() != 1 || s2.ecards.size() != 1) continue;
        if (s1.tile == 0 || s2.tile == 0) continue;  // keep to the steps the tiled kernel covers
        // the frontier F of step 1, the intermediate as an operand of step 2
        int fi = -1, gi = -1, mi = -1, n_b1 = 0, n_b2 = 0;
        for (int i = 0; i < static_cast<int>(s1.in.size()); ++i)
            if (s1.in[i].batched) gi = fi, fi = i, ++n_b1;
        for (int i = 0; i < static_cast<int>(s2.in.size()); ++i)
            if (s2.in[i].batched) mi = i, ++n_b2;
        if (n_b1 < 1 || n_b1 > 2 || n_b2 != 1) continue;
        const InDesc &M = s2.in[mi];
        if (!M.is_slot || M.id != s1.out_slot || !M.ev.empty()) continue;
        if (n_b1 == 2) {
            // a second batched operand G supplies step 1's coefficients (modes GB / GC): no tables beside it, and F is
            // the operand that carries the variable step 2 sums out
            if (s1.in.size() != 2) continue;
            const int jy0 = axis_of_stride(s1.cards, M.estrides[0]);
            if (jy0 < 0) continue;
            if (s1.in[fi].strides[jy0] == 0 || (s1.in[gi].strides[jy0] != 0 && P->slots[s1.in[gi].id].size > P->slots[s1.in[fi].id].size))
                std::swap(fi, gi);
            if (!s1.in[gi].is_slot || !s1.in[gi].ev.empty() || s1.in[gi].id == s2.out_slot) continue;
        }
        const InDesc &F = s1.in[fi];
        if (!F.ev.empty()) continue;
        // the launch reads F while it writes the second step's output: never the same buffer
        // (planner.py `_assign_slots` releases a step's operands one step late for this)
        if (!F.is_slot || F.id == s2.out_slot || s1.out_slot == P->post_slot) continue;
        const int cx = s1.ecards[0], cy = s2.ecards[0];
        if (cx > T || cy > T) continue;
        const int jy = axis_of_stride(s1.cards, M.estrides[0]);
        if (jy < 0 || s1.cards[jy] != cy || F.strides[jy] == 0) continue;
        // out2 axes -> out1 axes; exactly one new variable z
        const int n2 = static_cast<int>(s2.cards.size()), n1 = static_cast<int>(s1.cards.size());
        std::vector<int> to1(n2, -1);
        int kz = -1, n_new = 0;
        bool ok = true;
        for (int k = 0; k < n2 && ok; ++k) {
            if (M.strides[k] == 0) {
                kz = k, ++n_new;
                continue;
            }
            to1[k] = axis_of_stride(s1.cards, M.strides[k]);
            if (to1[k] < 0 || to1[k] == jy || s1.cards[to1[k]] != s2.cards[k]) ok = false;
        }
        if (!ok || n_new != 1 || n2 != n1 || s2.cards[kz] > T) continue;
        // small cardinalities: the T^3 loop nest would be mostly padding
        if (std::min(std::min(cx, cy), s2.cards[kz]) < min_card) continue;

        for (int kw = 0; kw < n2; ++kw) {
            // w: a variable step 1 introduces (F lacks it)
            if (kw == kz) continue;
            const int jw = to1[kw];
            if (F.strides[jw] != 0 || s1.cards[jw] > T || s1.cards[jw] < min_card) continue;
            if (gi >= 0 && (s1.in[gi].strides[jw] == 0 || s1.in[gi].estrides[0] == 0 || cx != T || cy != T || s1.cards[jw] != T))
                continue;  // G must carry w and x, and is not padded: exact cardinalities
            std::vector<int> r2, r1;  // untouched axes, as axes of out2 / of out1
            int64_t n_tiles = 1;
            for (int k = 0; k < n2; ++k)
                if (k != kw && k != kz) r2.push_back(k), r1.push_back(to1[k]), n_tiles *= s2.cards[k];
            if (n_tiles >= (1LL << 27)) continue;
            CanonSpec c1, g1, c2, g2;
            if (gi < 0 && !spec_step(s1, fi, jy, jw, r1, &c1, &g1)) continue;
            if (!spec_step(s2, mi, kw, kz, r2, &c2, &g2)) continue;
            const int64_t total = c1.floats() + c2.floats() + g1.floats() + g2.floats();
            if (total * 4 > SBN_PAIR_SMEM_MAX) continue;
            if (!fetched) {
                int64_t n = 0;
                for (size_t t = 0; t < P->tables.size(); ++t) n = std::max(n, P->tables[t].first + P->table_padded[t]);
                H.cpt.resize(static_cast<size_t>(n));
                if (n > 0) err = cudaMemcpy(H.cpt.data(), P->d_tables, static_cast<size_t>(n) * 4, cudaMemcpyDeviceToHost);
                if (err != cudaSuccess) return err;
                fetched = true;
            }
            for (CanonSpec *cs : {&c1, &g1, &c2, &g2})
                for (const InDesc *in : cs->tabs) cs->data.push_back(host_table(P, H, *in, &err));
            if (err != cudaSuccess) return err;

            SbnPair *pr = new SbnPair();
            memset(&pr->q, 0, sizeof pr->q);
            memset(&pr->t, 0, sizeof pr->t);
            pr->kind = 0;
            pr->step1 = i1, pr->step2 = i2, pr->f_in = fi, pr->g_in = gi;
            pr->m1 = mode_of(c1.layout), pr->m2 = mode_of(c2.layout);
            if (gi >= 0) pr->m1 = s1.in[gi].strides[jy] == 0 ? SBN_PAIR_GB : SBN_PAIR_GC;
            pr->canon_pos = static_cast<int64_t>(canon.size());
            pr->tile_off_pos = static_cast<int64_t>(tiles.size());
            SbnPairParams &q = pr->q;
            q.canon_floats = static_cast<int32_t>(total);
            const int64_t at_c1 = 0, at_c2 = c1.floats(), at_g1 = at_c2 + c2.floats(), at_g2 = at_g1 + g1.floats();
            canon.resize(canon.size() + static_cast<size_t>(total), 0.f);
            fill_canon(c1, canon.data() + pr->canon_pos + at_c1);
            fill_canon(c2, canon.data() + pr->canon_pos + at_c2);
            fill_canon(g1, canon.data() + pr->canon_pos + at_g1);
            fill_canon(g2, canon.data() + pr->canon_pos + at_g2);
            q.n_tiles = static_cast<int32_t>(n_tiles);
            q.f_sx = F.estrides[0];
            q.f_sy = F.strides[jy];
            q.cx = cx, q.cy = cy, q.cw = s2.cards[kw], q.cz = s2.cards[kz];
            int64_t os = 1;
            std::vector<int64_t> os2(n2);
            for (int k = 0; k < n2; ++k) os2[k] = os, os *= s2.cards[k];
            q.o_sw = static_cast<int32_t>(os2[kw]);
            q.o_sz = static_cast<int32_t>(os2[kz]);
            if (gi >= 0) q.g_x = s1.in[gi].estrides[0], q.g_y = s1.in[gi].strides[jy], q.g_w = s1.in[gi].strides[jw];
            q.has_pre1 = g1.tabs.empty() ? 0 : 1;
            q.has_pre2 = g2.tabs.empty() ? 0 : 1;
            set_ev(&q.ev_main1, c1);
            set_ev(&q.ev_main2, c2);
            set_ev(&q.ev_pre1, g1);
            set_ev(&q.ev_pre2, g2);
            // tile table: one row per combination of the untouched axes (first axis fastest)
            std::vector<int> dig(r2.size(), 0);
            for (int64_t t = 0; t < n_tiles; ++t) {
                int64_t ob = 0, fb = 0;
                for (size_t k = 0; k < r2.size(); ++k) {
                    ob += dig[k] * os2[r2[k]];
                    fb += static_cast<int64_t>(dig[k]) * F.strides[r1[k]];
                }
                tiles.push_back(static_cast<int32_t>(ob));
                tiles.push_back(static_cast<int32_t>(fb));
                tiles.push_back(static_cast<int32_t>(at_c1 + tile_slab(c1, r1, dig)));
                tiles.push_back(static_cast<int32_t>(at_c2 + tile_slab(c2, r2, dig)));
                tiles.push_back(static_cast<int32_t>(at_g1 + tile_slab(g1, r1, dig)));
                tiles.push_back(static_cast<int32_t>(at_g2 + tile_slab(g2, r2, dig)));
                int64_t gb = 0;
                if (gi >= 0)
                    for (size_t k = 0; k < r1.size(); ++k) gb += static_cast<int64_t>(dig[k]) * s1.in[gi].strides[r1[k]];
                tiles.push_back(static_cast<int32_t>(gb));
                tiles.push_back(0);
                for (size_t k = 0; k < dig.size(); ++k) {
                    if (++dig[k] < s2.cards[r2[k]]) break;
                    dig[k] = 0;
                }
            }
            P->pair_first[i1] = static_cast<int>(P->pairs.size());
            P->pair_first[i2] = -2;
            P->pairs.push_back(pr);
            break;
        }
    }
    if (P->pairs.empty()) return cudaSuccess;
    err = cudaMalloc(&P->d_pair_canon, std::max<size_t>(canon.size(), 4) * 4);
    if (err != cudaSuccess) return err;
    err = cudaMalloc(&P->d_pair_tiles, tiles.size() * 4);
    if (err != cudaSuccess) return err;
    if (!canon.empty()) err = cudaMemcpy(P->d_pair_canon, canon.data(), canon.size() * 4, cudaMemcpyHostToDevice);
    if (err != cudaSuccess) return err;
    return cudaMemcpy(P->d_pair_tiles, tiles.data(), tiles.size() * 4, cudaMemcpyHostToDevice);
}

static cudaError_t triple_launch(sbn_program *P, const SbnPair &pr, int64_t n_rows, cudaStream_t stream) {
    SbnTripleParams q = pr.t;
    const StepDesc &s1 = P->steps[pr.step1], &s2 = P->steps[pr.step2];
    q.a = P->slots[s1.in[pr.a_in].id].ptr;
    q.b = P->slots[s1.in[pr.b_in].id].ptr;
    q.c = P->slots[s2.in[pr.c_in].id].ptr;
    q.out = P->slots[s2.out_slot].ptr;
    q.ld = P->ld;
    q.n_rows = static_cast<int32_t>(n_rows);
    q.tile_off = P->d_pair_tiles + pr.tile_off_pos;
    // SOROBN_B200_TRIPLE_KERNEL=0 selects the L1 body; read at every launch, so that one process can time both
    const char *body = getenv("SOROBN_B200_TRIPLE_KERNEL");
    if (pr.staged_ctas > 0 && !(body && atoi(body) == 0)) {
        // one wave of CTAs, each walking row blocks: the ring stays full across row blocks
        const int64_t n_rblocks = (n_rows + SBN_TRIPLE_ROWS - 1) / SBN_TRIPLE_ROWS;
        const int64_t grid = std::min<int64_t>(n_rblocks, pr.staged_ctas);
        sbn_launch(sbn_triple_kernel, dim3(static_cast<unsigned>(grid)), dim3(triple_threads(q)),
                   static_cast<size_t>(triple_smem(q)), stream, q);
        return cudaGetLastError();
    }
    // with a group axis: 32 rows x T group digits per CTA; without: 128 rows
    const int rows_per_cta = q.group > 1 ? 32 : 128;
    const int64_t n_rblocks = (n_rows + rows_per_cta - 1) / rows_per_cta;
    // few tiles per CTA: the CTAs resident together then cover few row blocks, whose operands stay in L2 for the
    // re-reads by the other tiles
    static const int64_t tpc_env = [] {
        const char *e = getenv("SOROBN_B200_TRIPLE_TPC");
        return e ? atoll(e) : 1LL;
    }();
    // measured on B200 (grid, 100k rows): 3 CTAs / SM (128 registers) 440-453 us, 2 CTAs (152 registers) 464-515 us
    static const int minb = [] {
        const char *e = getenv("SOROBN_B200_TRIPLE_MINB");
        return e ? atoi(e) : 3;
    }();
    const int64_t tpc = std::max<int64_t>(1, std::min<int64_t>(q.n_tiles, tpc_env));
    q.tiles_per_cta = static_cast<int32_t>(tpc);
    q.n_chunks = static_cast<int32_t>((q.n_tiles + tpc - 1) / tpc);
    const int64_t grid = q.n_chunks * n_rblocks;
    if (grid >= (1LL << 31)) return cudaErrorInvalidConfiguration;
    const dim3 g(static_cast<unsigned>(grid)), b(rows_per_cta, q.group);
    if (minb == 3) sbn_launch(sbn_triple_kernel_l1<3>, g, b, 0, stream, q);
    else if (minb == 1) sbn_launch(sbn_triple_kernel_l1<1>, g, b, 0, stream, q);
    else sbn_launch(sbn_triple_kernel_l1<2>, g, b, 0, stream, q);
    return cudaGetLastError();
}

bool sbn_pair_fits(const sbn_program *P, const SbnPair &pr) {
    // the kernels index their operands with 32-bit element offsets: entries x row pitch must stay below 2^31
    const StepDesc &s1 = P->steps[pr.step1], &s2 = P->steps[pr.step2];
    int64_t entries = P->slots[s2.out_slot].size;
    for (const InDesc &in : s1.in)
        if (in.batched) entries = std::max(entries, P->slots[in.id].size);
    for (const InDesc &in : s2.in)
        if (in.batched && in.id != s1.out_slot) entries = std::max(entries, P->slots[in.id].size);
    // (SOROBN_B200_PAIR_IDX_LIMIT lowers the limit: the tests use it to walk the fallback path with small programs)
    const char *e = getenv("SOROBN_B200_PAIR_IDX_LIMIT");
    const int64_t limit = e ? atoll(e) : (1LL << 31);
    return entries * P->ld < limit;
}

cudaError_t sbn_pair_launch(sbn_program *P, const SbnPair &pr, const uint8_t *d_ev, int64_t ld_ev, int64_t n_rows,
                            cudaStream_t stream) {
    if (pr.kind == 1) return triple_launch(P, pr, n_rows, stream);
    SbnPairParams q = pr.q;
    const StepDesc &s1 = P->steps[pr.step1], &s2 = P->steps[pr.step2];
    q.f = P->slots[s1.in[pr.f_in].id].ptr;
    q.g = pr.g_in >= 0 ? P->slots[s1.in[pr.g_in].id].ptr : q.f;
    q.out = P->slots[s2.out_slot].ptr;
    q.ev = d_ev;
    q.ld_ev = ld_ev;
    q.ld = P->ld;
    q.n_rows = static_cast<int32_t>(n_rows);
    q.canon = P->d_pair_canon + pr.canon_pos;
    q.tile_off = P->d_pair_tiles + pr.tile_off_pos;
    const int64_t n_rblocks = (n_rows + SBN_PAIR_ROWS - 1) / SBN_PAIR_ROWS;
    static const int64_t target = [] {
        const char *e = getenv("SOROBN_B200_PAIR_CTAS");
        return e ? atoll(e) : 8LL * 148 * 6;
    }();
    const int64_t chunks = std::max<int64_t>(1, std::min<int64_t>(q.n_tiles, target / std::max<int64_t>(1, n_rblocks)));
    const int64_t tpc = (q.n_tiles + chunks - 1) / chunks;
    q.tiles_per_cta = static_cast<int32_t>(tpc);
    q.n_chunks = static_cast<int32_t>((q.n_tiles + tpc - 1) / tpc);
    const int64_t grid = q.n_chunks * n_rblocks;
    if (grid >= (1LL << 31)) return cudaErrorInvalidConfiguration;
    launch_modes(pr, q, static_cast<unsigned>(grid), static_cast<size_t>(q.canon_floats) * 4, stream);
    return cudaGetLastError();
}
