// sorobn_b200 -- two eliminations in one launch ("paired steps").
//
// A run of `frontier <- sum_x table x frontier` steps (the benchmark grid's hot loop) writes every
// 625-entry intermediate to HBM and reads it straight back: 5000 B per row and step.  When step k + 1
// sums out a variable Y that the frontier F of step k already carries,
//
//     out[w, z, r] = sum_y c2[y, w, z, r] * ( sum_x c1[x, y, w, r] * F[x, y, r] )
//
// a thread that owns one row and one combination r of the untouched axes can keep the whole
// intermediate mid[y, w] (T x T values) in registers: it loads the T x T entries F[., ., r], applies
// step k, applies step k + 1 to the accumulators and stores the T x T entries out[., ., r].  The
// intermediate never exists in memory: 5000 B per row for the pair instead of 10000.
//
//   x = the variable step k eliminates          y = the variable step k + 1 eliminates (an axis of F)
//   w = a variable step k introduces            z = the variable step k + 1 introduces
//
// c1 / c2 are the products of the steps' tables (CPTs, hoisted table products).  They do not depend on
// the batch, so they are multiplied together ONCE, when the program is created, into "canonical"
// coefficient arrays laid out for the kernel (SbnPairMode below), zero-padded past the real
// cardinalities: the kernel is one fixed T x T x T loop nest of FFMAs fed by shared-memory loads with
// immediate offsets.  The arrays are staged in shared memory by one bulk-TMA copy per CTA.
//
// Reference operators fused by one launch: two rounds of `pointwise_mul` (bayes_net.py:253-256) +
// `sum_out` (bayes_net.py:54-103), and the evidence filter of bayes_net.py:772-774.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "../../include/sorobn_b200.h"

#define SBN_PAIR_T 5              // tile edge: every cardinality involved is <= 5
#define SBN_PAIR_PW 8             // coefficients per innermost row (T padded to two float4)
#define SBN_PAIR_MAX_EV 4         // evidence columns the tables of one step may gather
#define SBN_PAIR_ROWS 256         // evidence rows per CTA
#define SBN_TRIPLE_THREADS 160    // CTA of the expanding-product pattern: 32 rows x 5 group digits, or 128 rows x 1
#define SBN_PAIR_SMEM_MAX (40 * 1024)

// evidence columns one canonical array is indexed by: float offset = sum_k min(code_k, card_k - 1) * stride_k
struct SbnPairEv {
    int32_t n;
    int32_t col[SBN_PAIR_MAX_EV], stride[SBN_PAIR_MAX_EV], card[SBN_PAIR_MAX_EV];
};

struct SbnPairParams {
    const float *f;               // the batched operand of the first step  [entries][ld]
    float *out;                   // output of the second step               [entries][ld]
    const uint8_t *ev;
    const float *canon;           // canonical arrays of both steps (global; staged whole)
    const int32_t *tile_off;      // [n_tiles][8] = out entry, F entry, float offsets of main 1, main 2, pre 1, pre 2, G entry, 0
    int64_t ld_ev, ld;
    int32_t n_rows;
    int32_t canon_floats;         // multiple of 4
    int32_t n_tiles, tiles_per_cta, n_chunks;
    int32_t f_sx, f_sy;           // entry strides of x and y in F
    int32_t cx, cy, cw, cz;       // real cardinalities (<= T)
    int32_t o_sw, o_sz;           // entry strides of w and z in the output
    int32_t has_pre1, has_pre2;   // per-row factors applied to F[x][y] / mid[y][w] before the step's sum
    SbnPairEv ev_main1, ev_main2, ev_pre1, ev_pre2;
    const float *g;               // modes GB / GC: the second batched operand of step 1, its coefficients [entries][ld]
    int32_t g_x, g_y, g_w;        // ... and its entry strides (g_y = 0 in mode GB)
};

// Layout of a step's main coefficient array (chosen per step when the program is created):
//   B  -- no table carries the step's first tile axis: [evidence][r][x][8]        two float4 per x
//   CU -- [x][d0][d1] coefficients, no evidence axis:  [r][x][d0][8]              two float4 per (x, d0), the same
//                                                                                 address in every lane (broadcast)
//   CE -- [x][d0][d1] coefficients per evidence row:   [evidence][r][x][d0][d1]   scalar loads; a slab is 125 floats,
//                                                                                 odd, so the rows of a warp hit distinct banks
// A table that has evidence axes but not the second tile axis is kept out of the main array when that
// leaves the main array evidence-free: it becomes the "pre" factor [evidence][r][x][d0] applied to the
// step's operand first (25 scalar loads) and the main coefficients stay a broadcast.
// Step 1 only: when its coefficients are a second BATCHED factor G (`625 <- sum_x B125 x B625`, no tables), they are
// read from global memory, two rows per 64-bit load: GB = G lacks the first tile axis (25 loads per tile), GC = it
// carries it (125 loads per tile).  G has 5 x fewer entries than F and is re-read once per tile, out of L2.
enum SbnPairMode { SBN_PAIR_B = 0, SBN_PAIR_CU = 1, SBN_PAIR_CE = 2, SBN_PAIR_GB = 3, SBN_PAIR_GC = 4 };

// Second pattern: an expanding product and the contraction that consumes it,
//
//     mid[a.., p, k, s, q..] = sum_j A[a.., p, k, j] B[p, q.., j, s]        (e.g. 3125 <- B625 x B625)
//     out[a.., z, s, q..]    = sum_{p, k} C[k, q.., z, p] mid[a.., p, k, s, q..]   (625 <- sum_25 B625 x B3125)
//
// all operands batched, no tables.  The 3125-entry intermediate costs 25,000 B per row to write and read back;
// a thread that owns one row and one combination of the untouched axes (a.., q..) walks p, and per p computes
// N[k][s] = sum_j A[k][j] B[j][s] and out[z][s] += sum_k C[k][z] N[k][s] from 75 loaded entries -- the
// intermediate never exists.
//
// Two kernel bodies.  `sbn_triple_kernel` (the default) gives a CTA a block of 32 rows and every combination of the
// untouched axes: per p it stages the 32-row runs of all A, B and C entries of that p in shared memory (cp.async, a
// ring of `n_stages` p-slices), so each operand entry crosses HBM once per row; a thread then takes 2 rows (one
// register pair, packed FFMA2) and one (group digit, tile), keeps its 25 entries of B in registers and walks k.  It
// needs A to be the same for every tile and at most 15 x 25 entries per p (`SbnPair::staged_ctas`).
// `sbn_triple_kernel_l1` (SOROBN_B200_TRIPLE_KERNEL=0, and every triple the staged body does not cover) is one row per
// thread with the operands re-read once per combination of the axes they lack (from L1 / L2).
#define SBN_TRIPLE_ROWS 32            // rows per block of the staged body: the row pitch is a multiple of it
#define SBN_TRIPLE_MAX_ENTRIES 375    // operand entries staged per p: A (group x 25) + B and C (25 per tile each)
#define SBN_TRIPLE_MAX_STAGES 4
#define SBN_TRIPLE_MAX_THREADS 416    // 16 row pairs x 26 (group digit, tile) slots
struct SbnTripleParams {
    const float *a, *b, *c;
    float *out;
    const int32_t *tile_off;      // [n_tiles][4] = out entry, A entry, B entry, C entry
    int64_t ld;
    int32_t n_rows;
    int32_t n_tiles, tiles_per_cta, n_chunks;
    int32_t a_p, a_k, a_j;        // entry strides
    int32_t b_p, b_j, b_s;
    int32_t c_p, c_k, c_z;
    int32_t o_z, o_s;
    int32_t group;                // 1, or T: threadIdx.y walks the T digits of a tile axis only A carries ...
    int32_t a_g, o_g;             // ... with these entry strides in A and in the output
    int32_t n_stages;             // staged body: p-slices in the shared-memory ring (2 .. SBN_TRIPLE_MAX_STAGES)
};

// One planned pair (host side).
struct SbnPair {
    int kind;                     // 0: two table x frontier steps (SbnPairParams); 1: expanding product + contraction (SbnTripleParams)
    int step1, step2;             // indices into sbn_program::steps
    int f_in;                     // index of the batched operand among step1's inputs
    int g_in;                     // modes GB / GC: index of the second batched operand of step1, else -1
    int m1, m2;                   // SbnPairMode of the two steps
    SbnPairParams q;              // everything but the run-time pointers
    SbnTripleParams t;
    int a_in, b_in, c_in;         // kind 1: operand indices (A, B among step1's inputs, C among step2's)
    int staged_ctas;              // kind 1: CTAs of the staged body that fit the device at once, 0 when it does not apply
    int64_t tile_off_pos;         // int32 offset into the pair tile table
    int64_t canon_pos;            // float offset into the canonical coefficient buffer
};

struct sbn_program;
// Called once, after the evidence-independent steps ran (their outputs are operands here).
cudaError_t sbn_pair_plan(sbn_program *P);
cudaError_t sbn_pair_launch(sbn_program *P, const SbnPair &pr, const uint8_t *d_ev, int64_t ld_ev, int64_t n_rows,
                            cudaStream_t stream);
// false when the reserved row pitch is too large for the kernels' 32-bit element offsets: the two steps then run
// as separate launches
bool sbn_pair_fits(const sbn_program *P, const SbnPair &pr);
cudaError_t sbn_pair_set_attrs();
void sbn_pair_free(sbn_program *P);
