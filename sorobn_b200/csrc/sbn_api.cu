// sorobn_b200 -- C-ABI engine: program parsing, scratch management, launches.
//
// Host-side counterpart of `BayesNet._variable_elimination`
// (/root/reference/sorobn/bayes_net.py:739-794): the reference walks the hidden
// variables in Python and calls pandas for every product / sum-out; here the walk was
// frozen by sorobn_b200/planner.py into a list of steps and this file replays it as
// kernel launches (optionally captured in a CUDA graph) for a batch of evidence rows.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "sbn_chain.h"
#include "sbn_gibbs.cuh"
#include "sbn_internal.h"
#include "sbn_kernels.cuh"
#include "sbn_launch.h"
#include "sbn_pair.h"
#include "sbn_tma.h"

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define SBN_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail(SBN_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                        __LINE__);                                                                  \
    } while (0)

constexpr int32_t kMagic = 0x53424E31;
constexpr int kVersion = 4;
constexpr int kMaxElim = 3;
constexpr int kMaxZ = 256;
constexpr int kHeaderWords = 12;

}  // namespace

namespace {

int parse(sbn_program *P, const int32_t *w, int64_t n) {
    if (n < kHeaderWords) return fail(SBN_E_INVALID, "program shorter than its header");
    if (w[0] != kMagic) return fail(SBN_E_INVALID, "bad program magic 0x%x", w[0]);
    if (w[1] != kVersion) return fail(SBN_E_INVALID, "program version %d, engine expects %d", w[1], kVersion);
    P->mode = w[2];
    P->n_ev = w[3];
    const int n_tables = w[4], n_slots = w[5], n_steps = w[6];
    P->Q = w[7];
    P->post_slot = w[8];
    P->post_batched = w[9];
    if (P->mode != 0 && P->mode != 1) return fail(SBN_E_INVALID, "bad mode %d", P->mode);
    if (P->n_ev < 0 || n_tables < 0 || n_slots <= 0 || n_steps <= 0 || P->Q <= 0)
        return fail(SBN_E_INVALID, "bad header counts");
    if (P->post_slot < 0 || P->post_slot >= n_slots) return fail(SBN_E_INVALID, "post slot out of range");
    int64_t p = kHeaderWords;
    auto need = [&](int64_t k) { return p + k <= n; };
    if (!need(2LL * n_tables + 2LL * n_slots)) return fail(SBN_E_INVALID, "truncated table/slot section");
    for (int t = 0; t < n_tables; ++t) {
        const int64_t off = w[p], size = w[p + 1];
        p += 2;
        if (off < 0 || size <= 0 || (off % 4) != 0) return fail(SBN_E_INVALID, "bad table %d", t);
        P->tables.push_back({off, size});
        P->table_padded.push_back(round_up(size, 4));
    }
    for (int s = 0; s < n_slots; ++s) {
        const int batched = w[p];
        const int64_t size = w[p + 1];
        p += 2;
        if ((batched != 0 && batched != 1) || size <= 0) return fail(SBN_E_INVALID, "bad slot %d", s);
        if (batched && P->mode == 0) return fail(SBN_E_INVALID, "batched slot in a flat program");
        P->slots.push_back({batched != 0, size, round_up(size, 4), nullptr});
    }
    if ((P->slots[P->post_slot].batched ? 1 : 0) != P->post_batched || P->slots[P->post_slot].size < P->Q)
        return fail(SBN_E_INVALID, "posterior slot mismatch");
    for (int s = 0; s < n_steps; ++s) {
        if (!need(5)) return fail(SBN_E_INVALID, "truncated step %d", s);
        StepDesc st;
        st.kind = w[p];
        const int n_in = w[p + 1];
        st.out_slot = w[p + 2];
        const int n_axes = w[p + 3];
        const int n_elim = w[p + 4];
        st.cx = 1;
        p += 5;
        if (st.kind != 0 && st.kind != 1) return fail(SBN_E_INVALID, "step %d: bad kind", s);
        if (st.kind == 1 && P->mode == 0) return fail(SBN_E_INVALID, "step %d: batched step in a flat program", s);
        if (n_in < 1 || n_in > SBN_MAX_IN) return fail(SBN_E_INVALID, "step %d: %d inputs", s, n_in);
        if (n_axes < 0 || n_axes > SBN_MAX_AXES) return fail(SBN_E_INVALID, "step %d: %d axes", s, n_axes);
        if (n_elim < 0 || n_elim > kMaxElim) return fail(SBN_E_INVALID, "step %d: %d eliminated axes", s, n_elim);
        if (st.out_slot < 0 || st.out_slot >= n_slots) return fail(SBN_E_INVALID, "step %d: out slot", s);
        if (!need(n_axes + n_elim)) return fail(SBN_E_INVALID, "truncated step %d", s);
        st.n_out = 1;
        for (int j = 0; j < n_axes; ++j) {
            const int c = w[p + j];
            if (c < 1) return fail(SBN_E_INVALID, "step %d: axis card %d", s, c);
            st.n_out *= c;
            if (st.n_out >= (1LL << 31)) return fail(SBN_E_INVALID, "step %d: output too large", s);
            st.cards.push_back(c);
        }
        p += n_axes;
        for (int k = 0; k < n_elim; ++k) {
            const int c = w[p + k];
            if (c < 1) return fail(SBN_E_INVALID, "step %d: eliminated card %d", s, c);
            if (static_cast<int64_t>(st.cx) * c > kMaxZ) return fail(SBN_E_INVALID, "step %d: too many eliminated states", s);
            st.cx *= c;
            st.ecards.push_back(c);
        }
        p += n_elim;
        const Slot &os = P->slots[st.out_slot];
        if (os.batched != (st.kind == 1)) return fail(SBN_E_INVALID, "step %d: out slot kind mismatch", s);
        if (os.size < st.n_out) return fail(SBN_E_INVALID, "step %d: out slot too small", s);
        for (int i = 0; i < n_in; ++i) {
            if (!need(4)) return fail(SBN_E_INVALID, "truncated step %d input %d", s, i);
            InDesc in;
            in.is_slot = w[p] != 0;
            in.id = w[p + 1];
            in.batched = w[p + 2] != 0;
            in.sx = 0;
            const int n_ev = w[p + 3];
            p += 4;
            if (n_ev < 0 || n_ev > SBN_MAX_EV) return fail(SBN_E_INVALID, "step %d input %d: %d ev axes", s, i, n_ev);
            if (!need(3LL * n_ev + n_elim + n_axes)) return fail(SBN_E_INVALID, "truncated step %d input %d", s, i);
            int64_t size;
            if (in.is_slot) {
                if (in.id < 0 || in.id >= n_slots) return fail(SBN_E_INVALID, "step %d input %d: slot id", s, i);
                if (in.id == st.out_slot) return fail(SBN_E_INVALID, "step %d: output aliases input %d", s, i);
                if (P->slots[in.id].batched != in.batched)
                    return fail(SBN_E_INVALID, "step %d input %d: batched flag mismatch", s, i);
                size = P->slots[in.id].size;
            } else {
                if (in.id < 0 || in.id >= n_tables) return fail(SBN_E_INVALID, "step %d input %d: table id", s, i);
                if (in.batched) return fail(SBN_E_INVALID, "step %d input %d: batched table", s, i);
                size = P->tables[in.id].second;
            }
            if (in.batched && st.kind != 1) return fail(SBN_E_INVALID, "step %d: batched input in flat step", s);
            if (in.batched && n_ev) return fail(SBN_E_INVALID, "step %d input %d: batched input with ev axes", s, i);
            if (n_ev && st.kind != 1 && P->mode != 0)
                return fail(SBN_E_INVALID, "step %d input %d: evidence axes in an unbatched step", s, i);
            int64_t max_off = 0;
            for (int k = 0; k < n_ev; ++k) {
                EvAxis a{w[p], w[p + 1], w[p + 2]};
                p += 3;
                if (a.col < 0 || a.col >= P->n_ev || a.stride < 0 || a.card < 1 || a.card > 256)
                    return fail(SBN_E_INVALID, "step %d input %d: bad ev axis", s, i);
                max_off += static_cast<int64_t>(a.card - 1) * a.stride;
                in.ev.push_back(a);
            }
            for (int k = 0; k < n_elim; ++k) {
                const int sk = w[p + k];
                if (sk < 0) return fail(SBN_E_INVALID, "step %d input %d: negative stride", s, i);
                max_off += static_cast<int64_t>(st.ecards[k] - 1) * sk;
                in.estrides.push_back(sk);
            }
            p += n_elim;
            if (n_elim >= 1) in.sx = in.estrides[0];  // zoff enumerates joint states with this variable fastest
            for (int j = 0; j < n_axes; ++j) {
                const int sj = w[p + j];
                if (sj < 0) return fail(SBN_E_INVALID, "step %d input %d: negative stride", s, i);
                max_off += static_cast<int64_t>(st.cards[j] - 1) * sj;
                in.strides.push_back(sj);
            }
            p += n_axes;
            if (max_off >= size) return fail(SBN_E_INVALID, "step %d input %d: reads past its buffer", s, i);
            st.in.push_back(std::move(in));
        }
        P->steps.push_back(std::move(st));
    }
    if (p != n) return fail(SBN_E_INVALID, "trailing words in program");
    if (P->mode == 1) {
        // evidence-independent tables are computed once per program (run_table_steps): their slots
        // must not be recycled (planner: _assign_slots keep_unbatched)
        std::vector<int> writes(P->slots.size(), 0);
        for (const StepDesc &st : P->steps)
            if (st.kind == 0 && ++writes[st.out_slot] > 1)
                return fail(SBN_E_INVALID, "unbatched slot %d is written twice in a batched program", st.out_slot);
    }
    if (P->steps.back().out_slot != P->post_slot) return fail(SBN_E_INVALID, "last step does not write the posterior");
    return SBN_OK;
}

constexpr int kTiledMaxIn = 4;
constexpr int64_t kTileTableMax = 1 << 23;  // int32 words per step

// Tables staged per CTA: SBN_SMEM_BUDGET keeps several CTAs per SM.  Opt-in experiment
// (SOROBN_B200_SMEM_BIG=<KB>, up to 200): a launch around a larger CPT (8^5 entries = 128 KB) stages
// it with ONE CTA per SM walking every tile of its rows.  Measured on dag50: no gain (4 warps per
// SM are latency-bound on the shared-memory gathers: 2.65 vs 2.13 ms and 2.03 vs 2.21 ms on the two
// launches it applies to), so the default leaves such tables to the L1/L2 gathers of the plain kernel.
int64_t smem_big() {
    static const int64_t v = [] {
        const char *e = getenv("SOROBN_B200_SMEM_BIG");
        const int64_t kb = e ? atoll(e) : SBN_SMEM_BUDGET / 1024;
        return std::max<int64_t>(SBN_SMEM_BUDGET, std::min<int64_t>(kb * 1024, SBN_SMEM_BIG));
    }();
    return v;
}

// Slab variant of the tiled kernel: eligible when the launch multiplies one batched factor on
// the A side with one on the B side (plus at most one table without tile axes), both with
// private axes beyond the tile.  Emits the tile table in slab order (shared digits, then the
// B-private digits and B blocks, then the A-private digits and A blocks) and the slab's entry
// offsets.  Returns false when the step does not qualify (the caller then emits the plain
// tile table).
// Sliced staging.  The planner ships a CPT that is too big for shared memory with the output
// axes >= 2 outermost (planner.py `_relayout_big_tables`), so the tiles of one chunk touch a
// contiguous part of it.  Find the largest chunk whose parts fit SBN_SMEM_BUDGET and record, per
// chunk and input, which floats to stage and where.
int64_t slice_budget() {
    static const int64_t v = [] {
        const char *e = getenv("SOROBN_B200_SLICE_KB");
        // swept on B200 (dag50, 1M rows): 64 KB -> 8.46 ms, 32 KB -> 8.14 ms (more CTAs per SM),
        // 16 KB -> 10.8 ms (the launch with two 128 KB CPTs no longer fits and leaves the tiled kernel)
        const int64_t kb = e ? atoll(e) : 32;
        return std::max<int64_t>(1024, std::min<int64_t>(kb * 1024, SBN_SMEM_BUDGET));
    }();
    return v;
}
bool plan_slices(sbn_program *P, StepDesc &st, int T, std::vector<int32_t> *words) {
    const int n_in = static_cast<int>(st.in.size());
    const int n_axes = static_cast<int>(st.cards.size());
    const int row_words = n_in + 2;
    std::vector<int64_t> span(n_in, 0), size(n_in, 0);
    for (int i = 0; i < n_in; ++i) {
        const InDesc &in = st.in[st.order[i]];
        if (in.batched) continue;
        size[i] = in.is_slot ? P->slots[in.id].padded : P->table_padded[in.id];
        int64_t sp = 0;
        for (size_t k = 0; k < st.ecards.size(); ++k) sp += static_cast<int64_t>(st.ecards[k] - 1) * in.estrides[k];
        if (n_axes > 0) sp += static_cast<int64_t>(std::min(T, st.cards[0]) - 1) * in.strides[0];
        if (n_axes > 1) sp += static_cast<int64_t>(std::min(T, st.cards[1]) - 1) * in.strides[1];
        for (const EvAxis &a : in.ev) sp += static_cast<int64_t>(a.card - 1) * a.stride;
        span[i] = sp;
    }
    for (int64_t tpc = st.n_tiles; tpc >= 1; tpc = (tpc == 1 ? 0 : (tpc + 1) / 2)) {
        const int64_t chunks = (st.n_tiles + tpc - 1) / tpc;
        std::vector<int32_t> rec;
        rec.reserve(static_cast<size_t>(chunks) * n_in * 3);
        int64_t worst = 0;
        for (int64_t c = 0; c < chunks; ++c) {
            int64_t smem = 0;
            for (int i = 0; i < n_in; ++i) {
                if (st.in[st.order[i]].batched) {
                    rec.insert(rec.end(), {0, 0, -1});
                    continue;
                }
                int64_t lo = INT64_MAX, hi = 0;
                for (int64_t t = c * tpc; t < std::min(st.n_tiles, (c + 1) * tpc); ++t) {
                    const int64_t base = (*words)[static_cast<size_t>(st.tile_off_pos + t * row_words + 2 + i)];
                    lo = std::min(lo, base);
                    hi = std::max(hi, base + span[i] + 1);
                }
                lo = lo / 4 * 4;
                const int64_t len = std::min(round_up(hi - lo, 4), size[i] - lo);
                rec.insert(rec.end(), {static_cast<int32_t>(lo), static_cast<int32_t>(len), static_cast<int32_t>(smem)});
                smem += len;
            }
            worst = std::max(worst, smem);
        }
        if (worst * 4 <= slice_budget()) {
            st.slice_pos = static_cast<int64_t>(words->size());
            words->insert(words->end(), rec.begin(), rec.end());
            st.slice_tpc = tpc;
            st.slice_smem = worst;
            return true;
        }
    }
    return false;
}

bool plan_slab(sbn_program *P, StepDesc &st, int T, std::vector<int32_t> *words) {
    (void)P;
    const int n_axes = static_cast<int>(st.cards.size());
    const int n_in = static_cast<int>(st.in.size());
    if (st.nc != 0 || st.na != 1 || st.nb != 1 || st.nu > 1 || n_in > 3 || n_axes < 3) return false;
    if (st.ecards.size() != 1) return false;
    if (!(st.cx == T || (T == 4 && st.cx == 8))) return false;  // needs the preload schedule
    const InDesc &A = st.in[st.order[st.nu]], &B = st.in[st.order[st.nu + 1]];
    if (!A.batched || !B.batched) return false;
    const int c0 = st.cards[0], c1 = st.cards[1];
    std::vector<int> pa, pb, sh;  // axes >= 2: private to A, private to B, shared
    int64_t n_pa = 1, n_pb = 1, n_sh = 1;
    for (int j = 2; j < n_axes; ++j) {
        const bool ha = A.strides[j] != 0, hb = B.strides[j] != 0;
        if (ha && !hb) { pa.push_back(j); n_pa *= st.cards[j]; }
        else if (hb && !ha) { pb.push_back(j); n_pb *= st.cards[j]; }
        else { sh.push_back(j); n_sh *= st.cards[j]; }
    }
    if (n_pa == 1 || n_pb == 1) return false;  // nothing is re-read: the plain tile walk is optimal
    // small operands are re-read from L2 anyway (measured: B125 x B125 is faster without the slab)
    if (static_cast<int64_t>(c0) * n_pa * st.cx < 512 || static_cast<int64_t>(c1) * n_pb * st.cx < 512) return false;
    const int64_t ma = static_cast<int64_t>(c0) * n_pa;
    const int64_t n_slab = ma * st.cx;
    if (n_slab * kSlabThreads * kRowsPerThread * 4 > kSlabSmemMax) return false;
    const int n_ta = (c0 + T - 1) / T, n_tb = (c1 + T - 1) / T;
    const int64_t tiles_per_super = n_pb * n_tb * n_pa * n_ta;
    if (n_sh * tiles_per_super * (n_in + 5) > kTileTableMax) return false;

    st.slab = true;
    st.slab_ma = static_cast<int>(ma);
    st.n_slab = static_cast<int>(n_slab);
    st.n_super = n_sh;
    st.tiles_per_super = tiles_per_super;
    // slab entry k = x * ma + (d0 + c0 * pa_index)  ->  element offset inside A (shared digits 0)
    st.slab_off_pos = static_cast<int64_t>(words->size());
    for (int x = 0; x < st.cx; ++x)
        for (int64_t ia = 0; ia < n_pa; ++ia)
            for (int d0 = 0; d0 < c0; ++d0) {
                int64_t off = static_cast<int64_t>(x) * A.sx + static_cast<int64_t>(d0) * A.strides[0];
                int64_t r = ia;
                for (int j : pa) {
                    off += (r % st.cards[j]) * A.strides[j];
                    r /= st.cards[j];
                }
                words->push_back(static_cast<int32_t>(off));
            }
    // NOTE the loop nest above emits (x, ia, d0) with d0 fastest: index = x*ma + ia*c0 + d0

    std::vector<int64_t> out_stride(n_axes, 1);
    for (int j = 1; j < n_axes; ++j) out_stride[j] = out_stride[j - 1] * st.cards[j - 1];
    st.slab_tile_off_pos = static_cast<int64_t>(words->size());
    std::vector<int> digit(n_axes, 0);
    for (int64_t is = 0; is < n_sh; ++is) {
        int64_t r = is;
        for (int j : sh) { digit[j] = static_cast<int>(r % st.cards[j]); r /= st.cards[j]; }
        int64_t a_super = 0;
        for (int j : sh) a_super += static_cast<int64_t>(digit[j]) * A.strides[j];
        for (int64_t ib = 0; ib < n_pb; ++ib) {
            r = ib;
            for (int j : pb) { digit[j] = static_cast<int>(r % st.cards[j]); r /= st.cards[j]; }
            for (int tb = 0; tb < n_tb; ++tb) {
                for (int64_t ia = 0; ia < n_pa; ++ia) {
                    r = ia;
                    for (int j : pa) { digit[j] = static_cast<int>(r % st.cards[j]); r /= st.cards[j]; }
                    for (int ta = 0; ta < n_ta; ++ta) {
                        const int na = std::min(T, c0 - ta * T), nb = std::min(T, c1 - tb * T);
                        int64_t o = static_cast<int64_t>(ta) * T + static_cast<int64_t>(tb) * T * c0;
                        for (int j = 2; j < n_axes; ++j) o += static_cast<int64_t>(digit[j]) * out_stride[j];
                        words->push_back(static_cast<int32_t>(o));
                        words->push_back(na | (nb << 8));
                        for (int i = 0; i < n_in; ++i) {
                            const InDesc &in = st.in[st.order[i]];
                            int64_t off = static_cast<int64_t>(ta) * T * in.strides[0] + static_cast<int64_t>(tb) * T * in.strides[1];
                            for (int j = 2; j < n_axes; ++j) off += static_cast<int64_t>(digit[j]) * in.strides[j];
                            words->push_back(static_cast<int32_t>(off));
                        }
                        words->push_back(static_cast<int32_t>(is));
                        words->push_back(static_cast<int32_t>(ta * T + static_cast<int64_t>(c0) * ia));
                        words->push_back(static_cast<int32_t>(a_super));
                    }
                }
            }
        }
    }
    return true;
}

// Host half of the tiled kernel: pick the tile edge and precompute, for every tile, the
// output entry and each input's element offset (the row-invariant mixed-radix
// decomposition, hoisted out of the kernel).
void plan_tiles(sbn_program *P, std::vector<int32_t> *words) {
    // joint-state offset tables of the steps that sum out several variables at once:
    // zoff[i][z] = sum_k digit_k(z) * estride_i[k], first eliminated variable fastest
    for (StepDesc &st : P->steps) {
        st.zoff_pos = -1;
        if (st.ecards.size() < 2) continue;
        st.zoff_pos = static_cast<int64_t>(words->size());
        for (const InDesc &in : st.in) {
            for (int z = 0; z < st.cx; ++z) {
                int r = z;
                int64_t off = 0;
                for (size_t k = 0; k < st.ecards.size(); ++k) {
                    off += static_cast<int64_t>(r % st.ecards[k]) * in.estrides[k];
                    r /= st.ecards[k];
                }
                words->push_back(static_cast<int32_t>(off));
            }
        }
    }
    for (StepDesc &st : P->steps) {
        st.tile = 0;
        if (st.kind != 1 || st.in.size() > static_cast<size_t>(kTiledMaxIn)) continue;

        int64_t smem = 0;
        for (const InDesc &in : st.in)
            if (!in.batched) smem += in.is_slot ? P->slots[in.id].padded : P->table_padded[in.id];
        const bool over = smem * 4 > SBN_SMEM_BUDGET;
        st.big_tables = over && smem * 4 <= smem_big();
        const bool sliced = over && !st.big_tables;  // decided below, once the tiles are known
        const int n_axes = static_cast<int>(st.cards.size());
        const int c0 = n_axes > 0 ? st.cards[0] : 1;
        const int c1 = n_axes > 1 ? st.cards[1] : 1;
        if (c0 > 255 * 5 || c1 > 255 * 5) continue;
        // sort the inputs by the tile axes they carry
        std::vector<int> us, as, bs, cs;
        for (size_t i = 0; i < st.in.size(); ++i) {
            const bool h0 = n_axes > 0 && st.in[i].strides[0] != 0;
            const bool h1 = n_axes > 1 && st.in[i].strides[1] != 0;
            if (h0 && h1) cs.push_back(static_cast<int>(i));
            else if (h0) as.push_back(static_cast<int>(i));
            else if (h1) bs.push_back(static_cast<int>(i));
            else us.push_back(static_cast<int>(i));
        }
        if (cs.size() > 1) continue;  // two inputs span the whole tile: plain kernel
        if (cs.empty()) {
            // a factor without tile axes may ride on either side (stride 0 re-reads one entry)
            while (us.size() > 2 || (as.empty() && !us.empty())) {
                if (as.size() < 2) as.push_back(us.back());
                else if (n_axes > 1 && bs.size() < 2) bs.push_back(us.back());
                else break;
                us.pop_back();
            }
            if (us.size() > 2 || as.empty() || as.size() > 2 || bs.size() > 2) continue;
            if (n_axes > 1 && bs.empty()) continue;
        } else {
            // with a C-side input the instantiated combinations are NU, NA, NB <= 1
            if (us.size() > 1 || as.size() > 1 || bs.size() > 1) continue;
        }
        st.nu = static_cast<int>(us.size());
        st.na = static_cast<int>(as.size());
        st.nb = static_cast<int>(bs.size());
        st.nc = static_cast<int>(cs.size());
        st.order = us;
        st.order.insert(st.order.end(), as.begin(), as.end());
        st.order.insert(st.order.end(), bs.begin(), bs.end());
        st.order.insert(st.order.end(), cs.begin(), cs.end());
        if (st.zoff_pos >= 0) {
            // the tiled kernel sees its inputs in `order`: give it the offset rows in that order
            st.zoff_tiled_pos = static_cast<int64_t>(words->size());
            for (int slot : st.order)
                for (int z = 0; z < st.cx; ++z) {
                    const int32_t v = (*words)[static_cast<size_t>(st.zoff_pos) + static_cast<size_t>(slot) * st.cx + z];
                    words->push_back(v);
                }
        }
        // tile edge: least padding waste, ties to the larger tile
        int best_t = 2;
        double best_w = 1e30;
        for (int t = 2; t <= 5; ++t) {
            auto waste = [&](int c) { return static_cast<double>((c + t - 1) / t * t) / c; };
            // a single-axis output has a T x 1 tile: axis 1 wastes nothing
            const double w = waste(c0) * (n_axes > 1 ? waste(c1) : 1.0);
            if (w < best_w - 1e-9 || (w < best_w + 1e-9 && t > best_t)) {
                best_w = w;
                best_t = t;
            }
        }
        const int T = best_t;
        const int n_ta = (c0 + T - 1) / T, n_tb = (c1 + T - 1) / T;
        const int64_t rest = st.n_out / (static_cast<int64_t>(c0) * c1);
        const int64_t n_tiles = rest * n_ta * n_tb;
        const int n_in = static_cast<int>(st.in.size());
        if (n_tiles * (n_in + 2) > kTileTableMax) continue;
        st.tile = T;
        st.n_tiles = n_tiles;
        st.slab = false;
        if (!over) plan_slab(P, st, T, words);  // optional second tile table in slab order
        st.tile_off_pos = static_cast<int64_t>(words->size());
        std::vector<int64_t> off(n_in);
        for (int64_t r = 0; r < rest; ++r) {
            int64_t q = r;
            std::fill(off.begin(), off.end(), 0);
            for (int j = 2; j < n_axes; ++j) {
                const int d = static_cast<int>(q % st.cards[j]);
                q /= st.cards[j];
                for (int i = 0; i < n_in; ++i) off[i] += static_cast<int64_t>(d) * st.in[st.order[i]].strides[j];
            }
            for (int tb = 0; tb < n_tb; ++tb) {
                for (int ta = 0; ta < n_ta; ++ta) {
                    const int na = std::min(T, c0 - ta * T), nb = std::min(T, c1 - tb * T);
                    words->push_back(static_cast<int32_t>(r * c0 * c1 + static_cast<int64_t>(tb) * T * c0 + ta * T));
                    words->push_back(na | (nb << 8));
                    for (int i = 0; i < n_in; ++i) {
                        int64_t o = off[i];
                        if (n_axes > 0) o += static_cast<int64_t>(ta) * T * st.in[st.order[i]].strides[0];
                        if (n_axes > 1) o += static_cast<int64_t>(tb) * T * st.in[st.order[i]].strides[1];
                        words->push_back(static_cast<int32_t>(o));
                    }
                }
            }
        }
        if (sliced && !plan_slices(P, st, T, words)) st.tile = 0;  // plain kernel, tables from L1/L2
    }
}

void free_scratch(sbn_program *P) {
    if (P->exec) {
        cudaGraphExecDestroy(P->exec);
        P->exec = nullptr;
    }
    if (P->pipe_exec) {
        cudaGraphExecDestroy(P->pipe_exec);
        P->pipe_exec = nullptr;
    }
    cudaFree(P->d_arena);
    cudaFree(P->d_ev);
    cudaFree(P->d_out);
    cudaFree(P->d_total);
    P->d_total = nullptr;
    P->d_arena = nullptr;
    P->d_ev = nullptr;
    P->d_out = nullptr;
    P->reserved_rows = 0;
    P->ld = 0;
}

int64_t batched_floats_per_row(const sbn_program *P) {
    int64_t t = 0;
    for (const Slot &s : P->slots)
        if (s.batched) t += s.size;
    return t;
}

// Fill the kernel parameter block of one step.
void build_params(const sbn_program *P, const StepDesc &st, const uint8_t *ev, int64_t ld_ev, int64_t n_rows,
                  SbnStep *q) {
    memset(q, 0, sizeof *q);
    q->out = P->slots[st.out_slot].ptr;
    q->ev = ev;
    q->ld_ev = ld_ev;
    q->ld = P->ld;
    q->n_rows = static_cast<int32_t>(n_rows);
    q->n_in = static_cast<int32_t>(st.in.size());
    q->n_axes = static_cast<int32_t>(st.cards.size());
    q->cx = st.cx;
    q->cx_inner = st.ecards.empty() ? 1 : st.ecards[0];
    q->zoff = st.zoff_pos >= 0 ? P->d_tile_off + st.zoff_pos : nullptr;
    if (st.kind == 1 && st.tile > 0 && P->use_tiled && !P->f64 && st.zoff_tiled_pos >= 0) q->zoff = P->d_tile_off + st.zoff_tiled_pos;
    q->n_out = static_cast<int32_t>(st.n_out);
    for (size_t j = 0; j < st.cards.size(); ++j) q->card[j] = st.cards[j];
    int smem = 0;
    const bool tiled = st.kind == 1 && st.tile > 0 && P->use_tiled && !P->f64;
    for (size_t i = 0; i < st.in.size(); ++i) {
        const InDesc &in = st.in[tiled ? st.order[i] : i];
        SbnInput &d = q->in[i];
        int64_t padded;
        if (in.is_slot) {
            d.ptr = P->slots[in.id].ptr;
            padded = P->slots[in.id].padded;
        } else {
            d.ptr = reinterpret_cast<const float *>(reinterpret_cast<const char *>(P->d_tables) +
                                                    P->tables[in.id].first * (P->f64 ? 8 : 4));
            padded = P->table_padded[in.id];
        }
        d.batched = in.batched ? 1 : 0;
        d.sx = in.sx;
        d.n_ev = static_cast<int32_t>(in.ev.size());
        for (size_t k = 0; k < in.ev.size(); ++k) {
            d.ev_col[k] = in.ev[k].col;
            d.ev_stride[k] = in.ev[k].stride;
            d.ev_card[k] = in.ev[k].card;
        }
        for (size_t j = 0; j < in.strides.size(); ++j) d.stride[j] = in.strides[j];
        d.smem_off = -1;
        d.stage_floats = 0;
        if (tiled && st.slice_pos >= 0) {
            // sliced staging: the kernel reads (first float, floats, offset) per chunk from q->slices
            if (!in.batched) d.smem_off = 0;
        } else if (st.kind == 1 && !P->f64 && !in.batched && (smem + padded) * 4 <= (tiled ? smem_big() : SBN_SMEM_BUDGET)) {
            d.smem_off = smem;
            d.stage_floats = static_cast<int32_t>(padded);
            smem += static_cast<int>(padded);
        }
    }
    q->smem_floats = smem;
    q->slices = nullptr;
    if (tiled && st.slice_pos >= 0) {
        q->smem_floats = static_cast<int32_t>(st.slice_smem);
        q->slices = P->d_tile_off + st.slice_pos;
    }
    if (tiled) {
        const int64_t rows_per_cta = static_cast<int64_t>(tiled_threads()) * kRowsPerThread;
        const int64_t n_rblocks = (n_rows + rows_per_cta - 1) / rows_per_cta;
        // enough CTAs for ~8 waves (148 SMs x ~6 resident CTAs), otherwise as many
        // consecutive tiles per CTA as possible (neighbouring tiles share operands in L1)
        static const int64_t target_env = [] {
            const char *e = getenv("SOROBN_B200_TARGET_CTAS");
            return e ? atoll(e) : 0LL;
        }();
        // swept on B200 (grid workload): 3552 -> 4.20 ms, 7104 -> 4.10 ms, 14208 -> 4.23 ms
        // big tables: one CTA per SM, so few CTAs that each amortise their 100+ KB of staging
        int64_t target = st.big_tables ? 4 * 148 : (target_env > 0 ? target_env : 8 * 148 * 6);
        static const int64_t small_env = [] {
            const char *e = getenv("SOROBN_B200_SMALL_WAVE");
            return e ? atoll(e) : 2000LL;
        }();
        // A launch with few tiles in total (at one tile per CTA: under ~4.5 waves) runs as ONE wave
        // of CTAs that each walk all their tiles: staging and the first loads are paid once per CTA,
        // not once per tile (grid: 3.305 -> 3.264 ms; the 125-entry table-only launches 22 -> 17 us).
        if (small_env > 0 && !st.big_tables && st.n_tiles * n_rblocks <= small_env) target = 3 * 148;
        int64_t chunks = std::max<int64_t>(1, std::min<int64_t>(st.n_tiles, target / std::max<int64_t>(1, n_rblocks)));
        int64_t tpc = (st.n_tiles + chunks - 1) / chunks;
        if (st.slice_pos >= 0) tpc = st.slice_tpc;  // the slices were cut for this chunk size
        q->tiles_per_cta = static_cast<int32_t>(tpc);
        q->n_tiles = static_cast<int32_t>(st.n_tiles);
        q->n_chunks = static_cast<int32_t>((st.n_tiles + tpc - 1) / tpc);
        q->tile_off = P->d_tile_off + st.tile_off_pos;
        q->n_bblocks = static_cast<int32_t>(n_rblocks);
        q->tile1 = 0;
        q->n_tile1 = 0;
        if (st.slab && !st.big_tables && P->use_preload && P->use_slab) {
            // whole groups per CTA; 64-thread CTAs (128 rows) so that the slab fits shared memory
            const int64_t rows_slab = static_cast<int64_t>(kSlabThreads) * kRowsPerThread;
            const int64_t n_rb = (n_rows + rows_slab - 1) / rows_slab;
            const int64_t groups = std::max<int64_t>(1, std::min<int64_t>(st.n_super, target / std::max<int64_t>(1, n_rb)));
            const int64_t supers_per_cta = (st.n_super + groups - 1) / groups;
            q->tiles_per_cta = static_cast<int32_t>(supers_per_cta * st.tiles_per_super);
            q->n_chunks = static_cast<int32_t>((st.n_super + supers_per_cta - 1) / supers_per_cta);
            q->n_bblocks = static_cast<int32_t>(n_rb);
            q->tile_off = P->d_tile_off + st.slab_tile_off_pos;
            q->slab_off = P->d_tile_off + st.slab_off_pos;
            q->n_slab = st.n_slab;
            q->slab_ma = st.slab_ma;
            q->slab_smem_off = static_cast<int32_t>(round_up(q->smem_floats, 4));
        }
    } else if (st.kind == 1) {
        const int c0 = q->n_axes > 0 ? q->card[0] : 1;
        const int c1 = q->n_axes > 1 ? q->card[1] : 1;
        const int64_t rows_per_cta = P->f64 ? SBN_THREADS * 2 : SBN_ROWS_PER_CTA;  // double2 / float4 per thread
        const int64_t n_bblocks = (n_rows + rows_per_cta - 1) / rows_per_cta;
        const int64_t rest = st.n_out / (static_cast<int64_t>(c0) * c1);
        // Tile = axis 0 x tile1 digits of axis 1.  Start from ~32 outputs per thread and
        // shrink while the grid is below two full waves (148 SMs x 16 CTAs).
        int tile1 = std::max(1, std::min(c1, 32 / std::max(1, c0)));
        auto ctas = [&](int t1) { return n_bblocks * ((c1 + t1 - 1) / t1) * rest; };
        while (tile1 > 1 && ctas(tile1) < 2 * 148 * 16) tile1 = (tile1 + 1) / 2;
        q->tile1 = tile1;
        q->n_tile1 = (c1 + tile1 - 1) / tile1;
        q->n_bblocks = static_cast<int32_t>(n_bblocks);
    }
}

cudaError_t launch_tiled(const StepDesc &st, const SbnStep &q, bool preload, int64_t grid, cudaStream_t stream) {
    // the kernel instantiations live in four translation units (sbn_tiled_*.cu), grouped by the number of
    // inputs without a tile axis / with a both-axes input
    if (q.slab_off != nullptr) return sbn_slab_launch(st.nu, q, st.tile, grid, stream);
    const int key = st.nu * 1000 + st.na * 100 + st.nb * 10 + st.nc;
    // the preload schedule keeps every operand of a tile, for one block of eliminated states, in
    // registers: only for <= 3 inputs, or 4 when two of them carry no tile axis (one value per state)
    preload = preload && (st.in.size() <= 3 || (st.nu == 2 && st.na == 1 && st.nb == 1));
    if (st.nc > 0) return sbn_tiled_c_launch(key, q, st.tile, preload, grid, stream);
    if (st.nu == 0) return sbn_tiled_u0_launch(key, q, st.tile, preload, grid, stream);
    if (st.nu == 1) return sbn_tiled_u1_launch(key, q, st.tile, preload, grid, stream);
    return sbn_tiled_u2_launch(key, q, st.tile, preload, grid, stream);
}

cudaError_t set_tiled_attrs() {
    cudaError_t e = sbn_tiled_u0_set_attrs();
    if (e == cudaSuccess) e = sbn_tiled_u1_set_attrs();
    if (e == cudaSuccess) e = sbn_tiled_u2_set_attrs();
    if (e == cudaSuccess) e = sbn_tiled_c_set_attrs();
    return e;
}

cudaError_t launch_step(sbn_program *P, const StepDesc &st, const SbnStep &q, cudaStream_t stream) {
    P->launches++;
    if (st.kind == 1 && q.tile_off != nullptr && sbn_tma_eligible(P, st))
        return sbn_tma_launch(P, st, q.ev, q.ld_ev, q.n_rows, stream);
    if (st.kind == 1 && q.tile_off != nullptr) {
        const int64_t chunks = (q.n_tiles + q.tiles_per_cta - 1) / q.tiles_per_cta;
        const int64_t grid = chunks * q.n_bblocks;
        if (grid >= (1LL << 31)) return cudaErrorInvalidConfiguration;
        return launch_tiled(st, q, P->use_preload, grid, stream);
    }
    if (st.kind == 0) {
        const int threads = 256;
        const int64_t grid = (st.n_out + threads - 1) / threads;
        if (P->f64) sbn_launch(sbn_step_flat<double>, dim3(static_cast<unsigned>(grid)), dim3(threads), 0, stream, q);
        else sbn_launch(sbn_step_flat<float>, dim3(static_cast<unsigned>(grid)), dim3(threads), 0, stream, q);
        return cudaGetLastError();
    }
    const int64_t rest = st.n_out / (static_cast<int64_t>(q.n_axes > 0 ? q.card[0] : 1) * (q.n_axes > 1 ? q.card[1] : 1));
    const int64_t grid = static_cast<int64_t>(q.n_bblocks) * q.n_tile1 * rest;
    if (grid >= (1LL << 31)) return cudaErrorInvalidConfiguration;
    if (P->f64) {
        const dim3 g(static_cast<unsigned>(grid)), b(SBN_THREADS);
        switch (q.n_in) {
            case 1: sbn_launch(sbn_step_batched_f64<1>, g, b, 0, stream, q); break;
            case 2: sbn_launch(sbn_step_batched_f64<2>, g, b, 0, stream, q); break;
            case 3: sbn_launch(sbn_step_batched_f64<3>, g, b, 0, stream, q); break;
            case 4: sbn_launch(sbn_step_batched_f64<4>, g, b, 0, stream, q); break;
            case 5: sbn_launch(sbn_step_batched_f64<5>, g, b, 0, stream, q); break;
            case 6: sbn_launch(sbn_step_batched_f64<6>, g, b, 0, stream, q); break;
            case 7: sbn_launch(sbn_step_batched_f64<7>, g, b, 0, stream, q); break;
            case 8: sbn_launch(sbn_step_batched_f64<8>, g, b, 0, stream, q); break;
            default: return cudaErrorInvalidValue;
        }
        return cudaGetLastError();
    }
    return sbn_batched_launch(q, grid, stream);
}

cudaError_t launch_normalise(sbn_program *P, float *d_out, int64_t ld_out, int64_t n_rows, cudaStream_t stream) {
    P->launches++;
    const int threads = 256;
    const int64_t grid = (n_rows + threads - 1) / threads;
    if (P->f64)
        sbn_normalise<double><<<static_cast<unsigned>(grid), threads, 0, stream>>>(
            reinterpret_cast<const double *>(P->slots[P->post_slot].ptr), P->ld, P->post_batched, P->Q,
            reinterpret_cast<double *>(d_out), ld_out, static_cast<int>(n_rows), 1e-290,
            reinterpret_cast<double *>(P->d_total));
    else
        sbn_normalise<float><<<static_cast<unsigned>(grid), threads, 0, stream>>>(
            P->slots[P->post_slot].ptr, P->ld, P->post_batched, P->Q, d_out, ld_out, static_cast<int>(n_rows),
            SBN_MIN_TOTAL_F32, P->d_total);
    return cudaGetLastError();
}

// Evidence-independent steps of a batched program (products of CPTs, possibly keeping evidence
// variables as ordinary axes) depend on the tables only: they run once, in create_common, and
// every later run reads their outputs (19 of the 67 launches of the benchmark grid's step).
inline bool hoisted(const sbn_program *P, const StepDesc &st) { return P->mode == 1 && st.kind == 0; }

inline bool chain_on(const sbn_program *P) {
    return P->use_chain && P->chain_fits && P->use_tiled && !P->use_branches && !P->segments.empty();
}

inline bool pair_on(const sbn_program *P) {
    // with the on-chip segments running, only pairs that were planned around them (SOROBN_B200_CHAIN=1 at creation)
    return P->use_pair && P->use_tiled && !P->use_branches && (!chain_on(P) || P->pairs_avoid_segments) && !P->pairs.empty();
}

inline bool graph_allowed(const sbn_program *P) { return P->use_graph; }

int run_table_steps(sbn_program *P) {
    if (P->mode != 1) return SBN_OK;
    SbnStep q;
    for (const StepDesc &st : P->steps) {
        if (!hoisted(P, st)) continue;
        build_params(P, st, nullptr, 0, 1, &q);
        SBN_CUDA(launch_step(P, st, q, P->stream));
    }
    SBN_CUDA(cudaStreamSynchronize(P->stream));
    P->setup_launches = P->launches;
    P->launches = 0;
    return SBN_OK;
}

// The normalisation can ride in the posterior step when that step runs on the tiled kernel (not the
// slab / TMA / plain variants) and its whole output is ONE tile (Q <= T x T joint query states).
inline bool fold_normalise(const sbn_program *P, const StepDesc &st, const SbnStep &q) {
#if !SBN_FOLD_NORMALISE
    // Compiled out by default (sbn_kernels.cuh): measured on B200, the extra epilogue in every instantiation of
    // the tiled kernel costs ~10 % on ALL launches (grid 3.14 -> 3.46 ms, dag50 7.26 -> 7.64 ms) to save one
    // 6 us launch (Asia 30 -> 24 us).
    (void)P;
    (void)st;
    (void)q;
    return false;
#endif
    static const bool enabled = [] {
        const char *e = getenv("SOROBN_B200_FOLD_NORMALISE");
        return e ? atoi(e) != 0 : true;
    }();
    return enabled && !P->f64 && P->post_batched && st.kind == 1 && q.tile_off != nullptr && q.slab_off == nullptr && st.n_tiles == 1 &&
           st.n_out == P->Q && !sbn_tma_eligible(P, st);
}

int issue_all(sbn_program *P, const uint8_t *d_ev, int64_t ld_ev, int64_t n_rows, float *d_out, int64_t ld_out,
              cudaStream_t stream, cudaEvent_t *events) {
    SbnStep q;
    int k = 0;
    bool folded = false;
    bool skip_second = false;  // the pair launched last covers the next launched step
    for (const StepDesc &st : P->steps) {
        if (events) SBN_CUDA(cudaEventRecord(events[k], stream));
        ++k;
        if (hoisted(P, st)) continue;  // computed once, when the program was created
        const int seg = chain_on(P) ? P->seg_first[k - 1] : -1;
        if (seg == -2) continue;       // runs inside the segment launched at its first step
        if (seg >= 0) {
            P->launches++;
            SBN_CUDA(sbn_chain_launch(P, *P->segments[seg], d_ev, ld_ev, n_rows, d_out, ld_out, stream));
            continue;
        }
        int pair = pair_on(P) ? P->pair_first[k - 1] : -1;
        if (pair == -2 && !skip_second) pair = -1;  // its first step ran on its own (row pitch beyond 32-bit offsets)
        skip_second = false;
        if (pair == -2) continue;      // computed by the launch of the step that feeds it
        if (pair >= 0 && !sbn_pair_fits(P, *P->pairs[pair])) pair = -1;
        if (pair >= 0) {
            skip_second = true;
            P->launches++;
            SBN_CUDA(sbn_pair_launch(P, *P->pairs[pair], d_ev, ld_ev, n_rows, stream));
            continue;
        }
        build_params(P, st, d_ev, ld_ev, n_rows, &q);
        if (k == static_cast<int>(P->steps.size()) && fold_normalise(P, st, q)) {
            // the posterior step's whole output is one register tile: normalise there, skip the extra launch
            q.norm_out = d_out;
            q.norm_ld = ld_out;
            q.norm_totals = P->d_total;
            q.norm_min = SBN_MIN_TOTAL_F32;
            folded = true;
        }
        SBN_CUDA(launch_step(P, st, q, stream));
    }
    if (events) SBN_CUDA(cudaEventRecord(events[k], stream));
    if (!folded && !(chain_on(P) && !P->segments.empty() && P->segments.back()->ends_in_posterior))
        SBN_CUDA(launch_normalise(P, d_out, ld_out, n_rows, stream));
    if (events) SBN_CUDA(cudaEventRecord(events[k + 1], stream));
    return SBN_OK;
}

// Capture-time variant of issue_all: steps are spread over the branch streams and ordered
// by events, so the instantiated graph carries exactly the true dependencies:
//   * read-after-write: a step waits for the producers of its slot inputs;
//   * slot reuse: a step that overwrites a slot waits for the slot's previous writer and
//     for every reader of the previous tenant.
// A step runs on the stream of the producer of its largest slot input (chains stay on one
// stream, no event needed); leaves take the branch streams round-robin.
int issue_branched(sbn_program *P, const uint8_t *d_ev, int64_t ld_ev, int64_t n_rows, float *d_out, int64_t ld_out,
                   cudaStream_t origin) {
    const int n_steps = static_cast<int>(P->steps.size());
    const int n_slots = static_cast<int>(P->slots.size());
    std::vector<int> last_writer(n_slots, -1);
    std::vector<std::vector<int>> readers(n_slots);
    std::vector<int> stream_of(n_steps, 0);
    cudaEvent_t fork = P->step_done[n_steps];  // reused as the fork event before any step
    SBN_CUDA(cudaEventRecord(fork, origin));
    bool joined[sbn_program::kBranches] = {false, false, false, false};
    int rr = 0;
    SbnStep q;
    for (int s = 0; s < n_steps; ++s) {
        const StepDesc &st = P->steps[s];
        if (hoisted(P, st)) continue;
        std::vector<int> deps;
        int home = -1;
        int64_t home_size = -1;
        for (const InDesc &in : st.in) {
            if (!in.is_slot) continue;
            const int w = last_writer[in.id];
            if (w >= 0 && !hoisted(P, P->steps[w])) {
                deps.push_back(w);
                if (P->slots[in.id].size > home_size) {
                    home_size = P->slots[in.id].size;
                    home = stream_of[w];
                }
            }
        }
        if (last_writer[st.out_slot] >= 0) deps.push_back(last_writer[st.out_slot]);
        for (int r : readers[st.out_slot]) deps.push_back(r);
        const int k = home >= 0 ? home : (rr++ % sbn_program::kBranches);
        stream_of[s] = k;
        cudaStream_t stream = P->branch[k];
        if (!joined[k]) {
            SBN_CUDA(cudaStreamWaitEvent(stream, fork, 0));
            joined[k] = true;
        }
        std::sort(deps.begin(), deps.end());
        deps.erase(std::unique(deps.begin(), deps.end()), deps.end());
        for (int d : deps)
            if (stream_of[d] != k) SBN_CUDA(cudaStreamWaitEvent(stream, P->step_done[d], 0));
        build_params(P, st, d_ev, ld_ev, n_rows, &q);
        SBN_CUDA(launch_step(P, st, q, stream));
        SBN_CUDA(cudaEventRecord(P->step_done[s], stream));
        for (const InDesc &in : st.in)
            if (in.is_slot) readers[in.id].push_back(s);
        last_writer[st.out_slot] = s;
        readers[st.out_slot].clear();
    }
    // join: the origin stream waits for the tail of every branch that was used, then normalises
    std::vector<int> tail(sbn_program::kBranches, -1);
    for (int s = 0; s < n_steps; ++s)
        if (!hoisted(P, P->steps[s])) tail[stream_of[s]] = s;
    for (int k = 0; k < sbn_program::kBranches; ++k)
        if (tail[k] >= 0) SBN_CUDA(cudaStreamWaitEvent(origin, P->step_done[tail[k]], 0));
    SBN_CUDA(launch_normalise(P, d_out, ld_out, n_rows, origin));
    return SBN_OK;
}

int check_run_args(sbn_program *P, const void *ev, int64_t ld_ev, int64_t n_rows, const void *out, int64_t ld_out) {
    if (!P) return fail(SBN_E_INVALID, "null program");
    if (n_rows <= 0) return fail(SBN_E_INVALID, "n_rows must be positive");
    if (!out) return fail(SBN_E_INVALID, "null output");
    if (P->n_ev > 0 && !ev) return fail(SBN_E_INVALID, "null evidence");
    if (P->n_ev > 1 && ld_ev < n_rows) return fail(SBN_E_INVALID, "ld_ev < n_rows");
    if (P->Q > 1 && ld_out < n_rows) return fail(SBN_E_INVALID, "ld_out < n_rows");
    if (P->mode == 0 && n_rows != 1) return fail(SBN_E_INVALID, "a flat program answers exactly one row");
    return SBN_OK;
}

}  // namespace

// =========================================================================== C ABI
extern "C" {

int sbn_abi_version(void) { return SBN_ABI_VERSION; }
const char *sbn_last_error(void) { return g_err.c_str(); }

int sbn_device_count(int *count) {
    if (!count) return fail(SBN_E_INVALID, "null count");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        *count = 0;
        return fail(SBN_E_NODEVICE, "no CUDA device: %s", cudaGetErrorString(e));
    }
    *count = n;
    return SBN_OK;
}

static int create_common(int device, const int32_t *words, int64_t n_words, const void *tables, int64_t n_table_floats,
                         bool f64, sbn_program **out) {
    if (!words || !out || (n_table_floats > 0 && !tables)) return fail(SBN_E_INVALID, "null argument");
    *out = nullptr;
    sbn_program *P = new sbn_program();
    P->device = device;
    P->f64 = f64;
    {
        const char *e = getenv("SOROBN_B200_CHAIN");
        P->use_chain = e && atoi(e) != 0;  // on-chip segments are opt-in (see sbn_chain.cu)
        e = getenv("SOROBN_B200_TMA");
        P->use_tma = e && atoi(e) != 0;    // so is the tensor-map TMA pipeline kernel (see sbn_tma.cu: no gain measured)
        e = getenv("SOROBN_B200_PAIR");
        P->use_pair = e ? atoi(e) != 0 : true;  // paired steps (sbn_pair.h)
    }
    const size_t elem = f64 ? 8 : 4;
    int rc = parse(P, words, n_words);

    if (rc != SBN_OK) {
        delete P;
        return rc;
    }
    for (size_t t = 0; t < P->tables.size(); ++t) {
        if (P->tables[t].first + P->table_padded[t] > n_table_floats) {
            delete P;
            return fail(SBN_E_INVALID, "table %zu lies outside the table blob", t);
        }
    }
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        delete P;
        return fail(SBN_E_NODEVICE, "no CUDA device available");
    }
    if (device < 0 || device >= n_dev) {
        delete P;
        return fail(SBN_E_NODEVICE, "device %d out of range (%d visible)", device, n_dev);
    }
    auto bail = [&](int code) {
        sbn_program_destroy(P);
        return code;
    };
#define SBN_CUDA_P(call)                                                                                      \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess)                                                                                \
            return bail(fail(SBN_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__)); \
    } while (0)
    SBN_CUDA_P(cudaSetDevice(device));
    cudaDeviceProp prop;
    SBN_CUDA_P(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return bail(fail(SBN_E_NODEVICE, "device %d is sm_%d%d; this library is built for sm_100a only",
                                           device, prop.major, prop.minor));
    SBN_CUDA_P(cudaStreamCreateWithFlags(&P->stream, cudaStreamNonBlocking));
    for (int k = 0; k < sbn_program::kBranches; ++k)
        SBN_CUDA_P(cudaStreamCreateWithFlags(&P->branch[k], cudaStreamNonBlocking));
    P->step_done.resize(P->steps.size() + 1);
    for (auto &e : P->step_done) SBN_CUDA_P(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    if (n_table_floats > 0) {
        // All setup traffic goes through the program's own (non-blocking) stream and is
        // synchronised below: a NULL-stream cudaMemcpy from pageable memory may return before
        // the DMA lands and would not be ordered with later work on P->stream.
        SBN_CUDA_P(cudaMalloc(&P->d_tables, static_cast<size_t>(n_table_floats) * elem));
        SBN_CUDA_P(cudaMemcpyAsync(P->d_tables, tables, static_cast<size_t>(n_table_floats) * elem,
                                   cudaMemcpyHostToDevice, P->stream));
    }
    // evidence-independent scratch: one allocation, 256-byte aligned sub-buffers
    int64_t shared_floats = 0;
    for (Slot &s : P->slots)
        if (!s.batched) shared_floats += round_up(s.padded, 64);
    if (shared_floats > 0) {
        SBN_CUDA_P(cudaMalloc(&P->d_shared, static_cast<size_t>(shared_floats) * elem));
        SBN_CUDA_P(cudaMemsetAsync(P->d_shared, 0, static_cast<size_t>(shared_floats) * elem, P->stream));
        int64_t off = 0;
        for (Slot &s : P->slots)
            if (!s.batched) {
                s.ptr = reinterpret_cast<float *>(reinterpret_cast<char *>(P->d_shared) + off * elem);
                off += round_up(s.padded, 64);
            }
    }
    {
        std::vector<int32_t> &tile_words = P->h_tile_words;  // kept: sbn_chain_bind derives its byte tables from them
        tile_words.clear();
        plan_tiles(P, &tile_words);
        if (!tile_words.empty()) {
            SBN_CUDA_P(cudaMalloc(&P->d_tile_off, tile_words.size() * 4));
            SBN_CUDA_P(cudaMemcpyAsync(P->d_tile_off, tile_words.data(), tile_words.size() * 4,
                                       cudaMemcpyHostToDevice, P->stream));
        }
        SBN_CUDA_P(cudaStreamSynchronize(P->stream));
        sbn_chain_plan(P);
    }
    {
        // opt every step-kernel instantiation into SBN_SMEM_BUDGET of dynamic shared memory
        // (once per device and process)
        static bool done[64] = {false};
        if (device < 64 && !done[device]) {
            SBN_CUDA_P(sbn_batched_set_attrs());
            SBN_CUDA_P(set_tiled_attrs());
            SBN_CUDA_P(sbn_chain_set_attrs());
            SBN_CUDA_P(sbn_tma_set_attrs());
            SBN_CUDA_P(sbn_pair_set_attrs());
            done[device] = true;
        }
    }
#undef SBN_CUDA_P
    rc = run_table_steps(P);
    if (rc != SBN_OK) return bail(rc);
    {
        // pairs multiply the tables of two steps on the host: needs the outputs of the table steps above
        cudaError_t e = sbn_pair_plan(P);
        if (e != cudaSuccess) return bail(fail(SBN_E_CUDA, "planning the paired steps failed: %s", cudaGetErrorString(e)));
    }
    *out = P;
    return SBN_OK;
}

int sbn_program_create(int device, const int32_t *words, int64_t n_words, const float *tables, int64_t n_table_floats,
                       sbn_program **out) {
    return create_common(device, words, n_words, tables, n_table_floats, false, out);
}

int sbn_program_create_f64(int device, const int32_t *words, int64_t n_words, const double *tables,
                           int64_t n_table_doubles, sbn_program **out) {
    return create_common(device, words, n_words, tables, n_table_doubles, true, out);
}

void sbn_program_destroy(sbn_program *P) {
    if (!P) return;
    cudaSetDevice(P->device);
    free_scratch(P);
    sbn_chain_free(P);
    sbn_pair_free(P);
    cudaFree(P->d_shared);
    cudaFree(P->d_tile_off);
    cudaFree(P->d_tables);
    if (P->stream) cudaStreamDestroy(P->stream);
    for (auto &b : P->branch)
        if (b) cudaStreamDestroy(b);
    for (auto &e : P->step_done)
        if (e) cudaEventDestroy(e);
    for (auto &e : P->pipe_events)
        if (e) cudaEventDestroy(e);
    delete P;
}

int sbn_program_reserve(sbn_program *P, int64_t max_rows) {
    if (!P) return fail(SBN_E_INVALID, "null program");
    if (max_rows <= 0) return fail(SBN_E_INVALID, "max_rows must be positive");
    if (P->mode == 0) max_rows = 1;
    if (max_rows <= P->reserved_rows) return SBN_OK;
    SBN_CUDA(cudaSetDevice(P->device));
    SBN_CUDA(cudaStreamSynchronize(P->stream));
    free_scratch(P);
    const int64_t elem = P->f64 ? 8 : 4;
    const int64_t per_row = batched_floats_per_row(P) * elem + P->n_ev + static_cast<int64_t>(P->Q) * elem + elem;
    size_t free_b = 0, total_b = 0;
    SBN_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const int64_t budget = static_cast<int64_t>(free_b * 0.85);
    int64_t rows = max_rows;
    if (per_row > 0 && round_up(rows, 32) * per_row > budget) rows = (budget / per_row) / 32 * 32;
    if (rows <= 0)
        return fail(SBN_E_NOMEM, "one evidence row needs %lld bytes of scratch; %lld free", (long long)per_row,
                    (long long)free_b);
    const int64_t ld = round_up(rows, 32);
    const int64_t arena = batched_floats_per_row(P) * ld;
    if (arena > 0) {
        cudaError_t e = cudaMalloc(&P->d_arena, static_cast<size_t>(arena) * elem);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(SBN_E_NOMEM, "cudaMalloc of %lld scratch bytes failed: %s", (long long)(arena * elem),
                        cudaGetErrorString(e));
        }
        int64_t off = 0;
        for (Slot &s : P->slots)
            if (s.batched) {
                s.ptr = reinterpret_cast<float *>(reinterpret_cast<char *>(P->d_arena) + off * elem);
                off += s.size * ld;
            }
    }
    if (P->n_ev > 0) {
        SBN_CUDA(cudaMalloc(&P->d_ev, static_cast<size_t>(P->n_ev) * ld));
        SBN_CUDA(cudaMemsetAsync(P->d_ev, 0, static_cast<size_t>(P->n_ev) * ld, P->stream));
    }
    SBN_CUDA(cudaMalloc(&P->d_out, static_cast<size_t>(P->Q) * ld * (P->f64 ? 8 : 4)));
    SBN_CUDA(cudaMalloc(&P->d_total, static_cast<size_t>(ld) * (P->f64 ? 8 : 4)));
    SBN_CUDA(cudaStreamSynchronize(P->stream));  // the memset must not race a caller's stream
    P->reserved_rows = rows;
    P->ld = ld;
    SBN_CUDA(sbn_chain_bind(P));  // segment descriptors point into the new arena
    return SBN_OK;
}

static int run_device_impl(sbn_program *P, const uint8_t *d_ev, int64_t ld_ev, int64_t n_rows, float *d_out,
                           int64_t ld_out, void *stream_);

int sbn_program_run_device(sbn_program *P, const uint8_t *d_ev, int64_t ld_ev, int64_t n_rows, float *d_out,
                           int64_t ld_out, void *stream_) {
    if (P && P->f64) return fail(SBN_E_INVALID, "float64 programs only run through sbn_program_run_host_f64");
    return run_device_impl(P, d_ev, ld_ev, n_rows, d_out, ld_out, stream_);
}

static int run_device_impl(sbn_program *P, const uint8_t *d_ev, int64_t ld_ev, int64_t n_rows, float *d_out,
                           int64_t ld_out, void *stream_) {
    int rc = check_run_args(P, d_ev, ld_ev, n_rows, d_out, ld_out);
    if (rc != SBN_OK) return rc;
    SBN_CUDA(cudaSetDevice(P->device));
    if (n_rows > P->reserved_rows) {  // grows (never shrinks); capped by the free device memory
        rc = sbn_program_reserve(P, n_rows);
        if (rc != SBN_OK) return rc;
    }
    if (n_rows > P->reserved_rows)
        return fail(SBN_E_NOMEM, "n_rows %lld exceeds the %lld rows of scratch that fit the device; use the host path "
                    "(it runs in chunks) or smaller batches", (long long)n_rows, (long long)P->reserved_rows);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!P->use_graph) return issue_all(P, d_ev, ld_ev, n_rows, d_out, ld_out, stream, nullptr);

    auto &k = P->graph_key;
    if (!P->exec || k.ev != d_ev || k.ld_ev != ld_ev || k.n_rows != n_rows || k.out != d_out || k.ld_out != ld_out) {
        if (P->exec) {
            cudaGraphExecDestroy(P->exec);
            P->exec = nullptr;
        }
        cudaStream_t cap = P->stream;  // capture on the program's own stream, replay on the caller's
        SBN_CUDA(cudaStreamBeginCapture(cap, cudaStreamCaptureModeRelaxed));
        const int64_t before = P->launches;
        rc = P->use_branches ? issue_branched(P, d_ev, ld_ev, n_rows, d_out, ld_out, cap)
                             : issue_all(P, d_ev, ld_ev, n_rows, d_out, ld_out, cap, nullptr);
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamEndCapture(cap, &graph);
        P->graph_launches = P->launches - before;
        P->launches = before;
        if (rc != SBN_OK) {
            if (graph) cudaGraphDestroy(graph);
            return rc;
        }
        if (e != cudaSuccess) return fail(SBN_E_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
        e = cudaGraphInstantiate(&P->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) return fail(SBN_E_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
        k = {d_ev, ld_ev, n_rows, d_out, ld_out};
    }
    SBN_CUDA(cudaGraphLaunch(P->exec, stream));
    P->launches += P->graph_launches;
    return SBN_OK;
}

static int run_host_common(sbn_program *P, const uint8_t *ev, int64_t ld_ev, int64_t n_rows, void *out_, int64_t ld_out,
                           bool f64, bool want_totals = false) {
    int rc = check_run_args(P, ev, ld_ev, n_rows, out_, want_totals ? n_rows : ld_out);
    if (rc != SBN_OK) return rc;
    if (P->f64 != f64) return fail(SBN_E_INVALID, "program precision does not match the run call");
    const size_t elem = f64 ? 8 : 4;
    char *out = static_cast<char *>(out_);
    SBN_CUDA(cudaSetDevice(P->device));
    if (n_rows > P->reserved_rows) {
        // the chunk capacity follows the largest batch seen so far (a program first used for one
        // row must not answer a later million-row batch one row at a time); the reservation is
        // capped by the free device memory, larger batches run in chunks
        rc = sbn_program_reserve(P, n_rows);
        if (rc != SBN_OK) return rc;
    }
    const int64_t cap = P->reserved_rows;
    // Transfer-bound programs (a handful of launches for megabytes of codes in and posteriors
    // out: Asia is ONE batched launch for 4 MB + 8 MB per million rows) are pipelined: the batch is
    // cut into column ranges of the same staging buffers, H2D / kernels / D2H run on three streams
    // chained by events, so a range's posteriors drain while the next range computes and the one
    // after uploads -- PCIe is full duplex.  Launch-heavy programs (the grid: 48 launches per run,
    // 5 MB of copies against 3 ms of kernels) keep the single CUDA-graph replay.
    int64_t launches_per_run = 1;
    for (size_t k = 0; k < P->steps.size(); ++k)
        if (!hoisted(P, P->steps[k])) ++launches_per_run;
    const int64_t bytes = n_rows * (P->n_ev + static_cast<int64_t>(want_totals ? 1 : P->Q) * static_cast<int64_t>(elem));
    static const int pipe_env = [] {
        const char *e = getenv("SOROBN_B200_PIPELINE");
        return e ? atoi(e) : 1;
    }();
    if (pipe_env && !want_totals && n_rows <= cap && launches_per_run <= 8 && bytes >= (int64_t(2) << 20) && n_rows >= 4 * 32768) {
        constexpr int kMaxRanges = 8;
        static const int kRanges = [] {
            const char *e = getenv("SOROBN_B200_PIPE_RANGES");
            // swept on B200 (Asia, 1M rows, 4 MB in + 8 MB out): 2 / 3 / 4 / 6 / 8 ranges -> 0.240 / 0.235 / 0.245 /
            // 0.251 / 0.253 ms, unpipelined 0.268 ms: the copies (51 GB/s for both directions together) are the bound
            const int v = e ? atoi(e) : 3;
            return v >= 2 && v <= kMaxRanges ? v : 3;
        }();
        if (P->pipe_events.empty()) {
            P->pipe_events.resize(3 + 2 * kMaxRanges);
            for (auto &e : P->pipe_events) SBN_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        cudaStream_t s_in = P->branch[0], s_run = P->stream, s_out = P->branch[1];
        const int64_t range = round_up((n_rows + kRanges - 1) / kRanges, 32);
        // the whole fan-out is issued into a stream capture and replayed as ONE graph launch when the
        // host buffers are pinned (a dozen copies, launches and event edges cost more CPU time than
        // the 0.2 ms they overlap); the graph is kept for the (buffers, rows) it was built for
        auto pinned = [](const void *ptr) {
            cudaPointerAttributes a;
            if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
                cudaGetLastError();
                return false;
            }
            return a.type == cudaMemoryTypeHost;
        };
        const bool as_graph = graph_allowed(P) && pinned(out) && (P->n_ev == 0 || pinned(ev));
        auto &key = P->pipe_key;
        const bool hit = as_graph && P->pipe_exec && key.ev == ev && key.ld_ev == ld_ev && key.n_rows == n_rows && key.out == out &&
                         key.ld_out == ld_out;
        if (!hit) {
            if (P->pipe_exec) {
                cudaGraphExecDestroy(P->pipe_exec);
                P->pipe_exec = nullptr;
            }
            const bool graph_was = P->use_graph;
            P->use_graph = false;  // a few plain launches per range: nothing to amortise inside
            cudaError_t e = cudaSuccess;
            if (as_graph) {
                e = cudaStreamBeginCapture(s_run, cudaStreamCaptureModeRelaxed);
                if (e == cudaSuccess) e = cudaEventRecord(P->pipe_events[0], s_run);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(s_in, P->pipe_events[0], 0);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(s_out, P->pipe_events[0], 0);
            }
            const int64_t before = P->launches;
            int k = 0;
            for (int64_t r0 = 0; r0 < n_rows && rc == SBN_OK && e == cudaSuccess; r0 += range, ++k) {
                const int64_t rows = std::min(range, n_rows - r0);
                cudaEvent_t up = P->pipe_events[1 + 2 * k], done = P->pipe_events[2 + 2 * k];
                if (P->n_ev > 0) {
                    e = cudaMemcpy2DAsync(P->d_ev + r0, static_cast<size_t>(P->ld), ev + r0, static_cast<size_t>(ld_ev),
                                          static_cast<size_t>(rows), static_cast<size_t>(P->n_ev), cudaMemcpyHostToDevice, s_in);
                    if (e == cudaSuccess) e = cudaEventRecord(up, s_in);
                    if (e == cudaSuccess) e = cudaStreamWaitEvent(s_run, up, 0);
                    if (e != cudaSuccess) break;
                }
                rc = run_device_impl(P, P->d_ev + r0, P->ld, rows, reinterpret_cast<float *>(reinterpret_cast<char *>(P->d_out) + r0 * elem),
                                     P->ld, s_run);
                if (rc != SBN_OK) break;
                e = cudaEventRecord(done, s_run);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(s_out, done, 0);
                // (P(event) runs are not pipelined: d_total is indexed by the row inside the launch)
                if (e == cudaSuccess)
                    e = cudaMemcpy2DAsync(out + r0 * elem, static_cast<size_t>(ld_out) * elem, reinterpret_cast<char *>(P->d_out) + r0 * elem,
                                          static_cast<size_t>(P->ld) * elem, static_cast<size_t>(rows) * elem, static_cast<size_t>(P->Q),
                                          cudaMemcpyDeviceToHost, s_out);
            }
            P->use_graph = graph_was;
            if (as_graph) {
                // join the side streams back into the origin, end the capture
                cudaEvent_t j_in = P->pipe_events[1 + 2 * kMaxRanges], j_out = P->pipe_events[2 + 2 * kMaxRanges];
                if (e == cudaSuccess) e = cudaEventRecord(j_in, s_in);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(s_run, j_in, 0);
                if (e == cudaSuccess) e = cudaEventRecord(j_out, s_out);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(s_run, j_out, 0);
                cudaGraph_t graph = nullptr;
                const cudaError_t e_end = cudaStreamEndCapture(s_run, &graph);
                P->pipe_launches = P->launches - before;
                P->launches = before;
                if (e == cudaSuccess) e = e_end;
                if (e == cudaSuccess && rc == SBN_OK) e = cudaGraphInstantiate(&P->pipe_exec, graph, 0);
                if (graph) cudaGraphDestroy(graph);
                if (rc != SBN_OK) return rc;
                if (e != cudaSuccess) {
                    cudaGetLastError();
                    return fail(SBN_E_CUDA, "pipelined graph capture failed: %s", cudaGetErrorString(e));
                }
                key = {ev, ld_ev, n_rows, out, ld_out};
            } else {
                cudaError_t e1 = cudaStreamSynchronize(s_in), e2 = cudaStreamSynchronize(s_run), e3 = cudaStreamSynchronize(s_out);
                if (rc != SBN_OK) return rc;
                if (e != cudaSuccess || e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)
                    return fail(SBN_E_CUDA, "pipelined run failed: %s",
                                cudaGetErrorString(e != cudaSuccess ? e : e1 != cudaSuccess ? e1 : e2 != cudaSuccess ? e2 : e3));
                return SBN_OK;
            }
        }
        SBN_CUDA(cudaGraphLaunch(P->pipe_exec, s_run));
        P->launches += P->pipe_launches;
        SBN_CUDA(cudaStreamSynchronize(s_run));
        return SBN_OK;
    }
    for (int64_t r0 = 0; r0 < n_rows; r0 += cap) {
        const int64_t rows = std::min(cap, n_rows - r0);
        if (P->n_ev > 0)
            SBN_CUDA(cudaMemcpy2DAsync(P->d_ev, static_cast<size_t>(P->ld), ev + r0, static_cast<size_t>(ld_ev),
                                       static_cast<size_t>(rows), static_cast<size_t>(P->n_ev), cudaMemcpyHostToDevice,
                                       P->stream));
        rc = run_device_impl(P, P->d_ev, P->ld, rows, P->d_out, P->ld, P->stream);
        if (rc != SBN_OK) return rc;
        if (want_totals)
            SBN_CUDA(cudaMemcpyAsync(out + r0 * elem, P->d_total, static_cast<size_t>(rows) * elem,
                                     cudaMemcpyDeviceToHost, P->stream));
        else
            SBN_CUDA(cudaMemcpy2DAsync(out + r0 * elem, static_cast<size_t>(ld_out) * elem, P->d_out,
                                       static_cast<size_t>(P->ld) * elem, static_cast<size_t>(rows) * elem,
                                       static_cast<size_t>(P->Q), cudaMemcpyDeviceToHost, P->stream));
    }
    SBN_CUDA(cudaStreamSynchronize(P->stream));
    return SBN_OK;
}

int sbn_program_run_host(sbn_program *P, const uint8_t *ev, int64_t ld_ev, int64_t n_rows, float *out, int64_t ld_out) {
    return run_host_common(P, ev, ld_ev, n_rows, out, ld_out, false);
}

int sbn_program_run_host_f64(sbn_program *P, const uint8_t *ev, int64_t ld_ev, int64_t n_rows, double *out,
                             int64_t ld_out) {
    return run_host_common(P, ev, ld_ev, n_rows, out, ld_out, true);
}

int sbn_program_evidence_host(sbn_program *P, const uint8_t *ev, int64_t ld_ev, int64_t n_rows, float *prob) {
    return run_host_common(P, ev, ld_ev, n_rows, prob, n_rows, false, true);
}

int sbn_program_evidence_host_f64(sbn_program *P, const uint8_t *ev, int64_t ld_ev, int64_t n_rows, double *prob) {
    return run_host_common(P, ev, ld_ev, n_rows, prob, n_rows, true, true);
}

int sbn_program_profile(sbn_program *P, const uint8_t *d_ev, int64_t ld_ev, int64_t n_rows, float *d_out,
                        int64_t ld_out, void *stream_, float *step_ms, int64_t n_step_ms) {
    int rc = check_run_args(P, d_ev, ld_ev, n_rows, d_out, ld_out);
    if (rc != SBN_OK) return rc;
    if (P->f64) return fail(SBN_E_INVALID, "profiling is for float32 programs");
    const int64_t n = static_cast<int64_t>(P->steps.size()) + 1;
    if (!step_ms || n_step_ms < n) return fail(SBN_E_INVALID, "step_ms needs %lld entries", (long long)n);
    SBN_CUDA(cudaSetDevice(P->device));
    if (n_rows > P->reserved_rows) {
        rc = sbn_program_reserve(P, n_rows);
        if (rc != SBN_OK) return rc;
    }
    if (n_rows > P->reserved_rows) return fail(SBN_E_NOMEM, "n_rows exceeds the scratch that fits the device");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto &e : ev) SBN_CUDA(cudaEventCreate(&e));
    rc = issue_all(P, d_ev, ld_ev, n_rows, d_out, ld_out, stream, ev.data());
    if (rc == SBN_OK) {
        cudaError_t e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) rc = fail(SBN_E_CUDA, "profile run failed: %s", cudaGetErrorString(e));
    }
    if (rc == SBN_OK)
        for (int64_t i = 0; i < n; ++i) cudaEventElapsedTime(&step_ms[i], ev[i], ev[i + 1]);
    for (auto &e : ev) cudaEventDestroy(e);
    return rc;
}

int sbn_program_info(const sbn_program *P, int64_t *info, int64_t n_info) {
    if (!P || !info || n_info < 8) return fail(SBN_E_INVALID, "info needs at least 8 entries");
    if (n_info >= 12) {
        int64_t covered = 0, hbm = 0, scratch = 0;
        for (const SbnSegment *seg : P->segments) {
            covered += static_cast<int64_t>(seg->steps.size());
            hbm += seg->hbm_bytes_per_row;
            scratch = std::max(scratch, seg->scratch_floats);
        }
        info[8] = chain_on(P) ? static_cast<int64_t>(P->segments.size()) : 0;
        info[9] = chain_on(P) ? covered : 0;
        info[10] = chain_on(P) ? hbm : 0;
        info[11] = scratch;
    }
    if (n_info >= 14) {
        int64_t saved = 0;
        for (const SbnPair *pr : P->pairs) saved += 8 * P->steps[pr->step1].n_out;  // one fp32 write + one read per entry
        info[12] = pair_on(P) ? static_cast<int64_t>(P->pairs.size()) : 0;
        info[13] = pair_on(P) ? saved : 0;
    }
    info[0] = P->Q;
    info[1] = P->n_ev;
    info[2] = static_cast<int64_t>(P->steps.size());
    info[3] = batched_floats_per_row(P);
    info[4] = P->reserved_rows;
    info[5] = P->launches;
    info[6] = P->mode;
    int64_t shared = 0;
    for (const Slot &s : P->slots)
        if (!s.batched) shared += s.size;
    info[7] = shared;
    return SBN_OK;
}

int sbn_program_step_roles(const sbn_program *P, int32_t *roles, int64_t n_roles) {
    if (!P || !roles || n_roles < static_cast<int64_t>(P->steps.size())) return fail(SBN_E_INVALID, "roles needs n_steps entries");
    int first_kind = 0;
    bool second_follows = false;
    for (size_t i = 0; i < P->steps.size(); ++i) {
        const StepDesc &st = P->steps[i];
        if (P->mode != 1 || hoisted(P, st)) {
            roles[i] = 0;
            continue;
        }
        roles[i] = 1;
        if (chain_on(P) && P->seg_first[i] != -1) {
            roles[i] = 6;
            continue;
        }
        int pair = pair_on(P) ? P->pair_first[i] : -1;
        if (pair == -2 && !second_follows) pair = -1;
        second_follows = false;
        if (pair == -2) roles[i] = first_kind == 1 ? 5 : 3;
        if (pair >= 0 && sbn_pair_fits(P, *P->pairs[pair])) {
            first_kind = P->pairs[pair]->kind;
            roles[i] = first_kind == 1 ? 4 : 2;
            second_follows = true;
        }
    }
    return SBN_OK;
}

static void drop_graphs(sbn_program *P) {
    // captured launches embed the kernel variants and pointers of the moment they were captured
    if (P->exec) {
        cudaGraphExecDestroy(P->exec);
        P->exec = nullptr;
    }
    if (P->pipe_exec) {
        cudaGraphExecDestroy(P->pipe_exec);
        P->pipe_exec = nullptr;
    }
}

int sbn_program_set_graph(sbn_program *P, int enabled) {
    if (!P) return fail(SBN_E_INVALID, "null program");
    P->use_graph = enabled != 0;
    P->use_branches = enabled == 3;
    drop_graphs(P);
    return SBN_OK;
}

int sbn_program_set_tiled(sbn_program *P, int enabled) {
    if (!P) return fail(SBN_E_INVALID, "null program");
    drop_graphs(P);
    P->use_tiled = enabled != 0;
    P->use_preload = enabled != 4;
    P->use_slab = enabled != 5;
    if (enabled == 8) P->use_tma = false;
    if (enabled == 9) P->use_tma = true;
    if (enabled == 6) P->use_chain = false;
    if (enabled == 7) P->use_chain = true;
    if (enabled == 10) P->use_pair = false;
    if (enabled == 11) P->use_pair = true;
    return SBN_OK;
}

int sbn_host_alloc(void **ptr, int64_t bytes) {
    if (!ptr || bytes <= 0) return fail(SBN_E_INVALID, "bad host allocation request");
    SBN_CUDA(cudaHostAlloc(ptr, static_cast<size_t>(bytes), cudaHostAllocDefault));
    return SBN_OK;
}

int sbn_host_free(void *ptr) {
    if (ptr) SBN_CUDA(cudaFreeHost(ptr));
    return SBN_OK;
}

}  // extern "C"

// ================================================================== Gibbs sampling
struct sbn_sampler {
    int device = 0;
    int n_vars = 0, n_query = 0, n_ev = 0, n_cycle = 0, Q = 0;
    int32_t *d_ints = nullptr;  // one allocation for every int array
    float *d_tables = nullptr;
    const int32_t *card = nullptr, *cpt_off = nullptr, *par_ptr = nullptr, *par_idx = nullptr, *par_stride = nullptr,
                  *chi_ptr = nullptr, *chi_idx = nullptr, *chi_stride = nullptr, *cycle = nullptr, *query = nullptr,
                  *ev_var = nullptr, *prog = nullptr, *flat = nullptr;
    int prog_words = 0, flat_words = 0;
    int64_t table_floats = 0;
    int max_card = 1;
    std::vector<int32_t> h_cycle;   // host copies for sbn_gibbs_conditional
    std::vector<int32_t> h_card;
    uint8_t *d_ev = nullptr;
    float *d_out = nullptr;
    int64_t cap = 0;
    cudaStream_t stream = nullptr;
    int64_t launches = 0;
};

extern "C" {

int sbn_gibbs_create(int device, int32_t n_vars, const int32_t *card, const int32_t *par_ptr, const int32_t *par_idx,
                     const int32_t *cpt_off, const float *tables, int64_t n_table_floats, int32_t n_query,
                     const int32_t *query, int32_t n_ev, const int32_t *ev_vars, int32_t n_cycle, const int32_t *cycle,
                     sbn_sampler **out) {
    if (!card || !par_ptr || !cpt_off || !tables || !query || !cycle || !out || (n_ev > 0 && !ev_vars))
        return fail(SBN_E_INVALID, "null argument");
    *out = nullptr;
    if (n_vars <= 0 || n_query <= 0 || n_cycle <= 0 || n_ev < 0) return fail(SBN_E_INVALID, "bad counts");
    const int n_par = par_ptr[n_vars];
    if (n_par > 0 && !par_idx) return fail(SBN_E_INVALID, "null parent list");
    // parents precede children (ids are topological) and every CPT lies inside the blob
    std::vector<int32_t> par_stride(n_par), chi_ptr(n_vars + 1, 0), chi_idx(n_par), chi_stride(n_par);
    for (int v = 0; v < n_vars; ++v) {
        if (card[v] < 1 || card[v] > SBN_GIBBS_MAX_CARD) return fail(SBN_E_INVALID, "variable %d has %d states (max %d)", v, card[v], SBN_GIBBS_MAX_CARD);
        if (par_ptr[v] > par_ptr[v + 1]) return fail(SBN_E_INVALID, "bad parent CSR");
        int64_t stride = card[v];
        for (int k = par_ptr[v + 1] - 1; k >= par_ptr[v]; --k) {
            const int pv = par_idx[k];
            if (pv < 0 || pv >= v) return fail(SBN_E_INVALID, "variable ids must be topological (parent %d of %d)", pv, v);
            par_stride[k] = static_cast<int32_t>(stride);
            stride *= card[pv];
            if (stride >= (1LL << 31)) return fail(SBN_E_INVALID, "CPT of variable %d is too large", v);
            chi_ptr[pv + 1]++;
        }
        if (cpt_off[v] < 0 || cpt_off[v] + stride > n_table_floats) return fail(SBN_E_INVALID, "CPT %d outside the table blob", v);
    }
    for (int v = 0; v < n_vars; ++v) chi_ptr[v + 1] += chi_ptr[v];
    {
        std::vector<int32_t> fill(chi_ptr.begin(), chi_ptr.end() - 1);
        for (int v = 0; v < n_vars; ++v)
            for (int k = par_ptr[v]; k < par_ptr[v + 1]; ++k) {
                const int pv = par_idx[k];
                chi_idx[fill[pv]] = v;
                chi_stride[fill[pv]] = par_stride[k];
                fill[pv]++;
            }
    }
    int64_t Q = 1;
    for (int k = 0; k < n_query; ++k) {
        if (query[k] < 0 || query[k] >= n_vars) return fail(SBN_E_INVALID, "query id out of range");
        Q *= card[query[k]];
        if (Q > 4096) return fail(SBN_E_INVALID, "more than 4096 joint query states");
    }
    for (int k = 0; k < n_ev; ++k)
        if (ev_vars[k] < 0 || ev_vars[k] >= n_vars) return fail(SBN_E_INVALID, "evidence id out of range");
    for (int k = 0; k < n_cycle; ++k)
        if (cycle[k] < 0 || cycle[k] >= n_vars) return fail(SBN_E_INVALID, "cycle id out of range");
    // the resampling cycle compiled into one record per position (layout: sbn_gibbs.cuh)
    std::vector<int32_t> prog(n_cycle, 0);
    int max_card = 1;
    for (int i = 0; i < n_cycle; ++i) {
        const int v = cycle[i];
        prog[i] = static_cast<int32_t>(prog.size());
        max_card = std::max(max_card, card[v]);
        const int np = par_ptr[v + 1] - par_ptr[v], nc = chi_ptr[v + 1] - chi_ptr[v];
        if (np > 255 || nc > 255 || v > 0xffff) return fail(SBN_E_INVALID, "variable %d has too many parents / children for the sampler", v);
        prog.push_back(v | card[v] << 16);
        prog.push_back(cpt_off[v]);
        prog.push_back(np | nc << 8);
        for (int k = par_ptr[v]; k < par_ptr[v + 1]; ++k) {
            prog.push_back(par_idx[k]);
            prog.push_back(par_stride[k]);
        }
        for (int k = chi_ptr[v]; k < chi_ptr[v + 1]; ++k) {
            const int ch = chi_idx[k];
            prog.push_back(cpt_off[ch]);
            prog.push_back(ch);
            prog.push_back(chi_stride[k]);
            int others = 0;
            for (int j = par_ptr[ch]; j < par_ptr[ch + 1]; ++j) others += par_idx[j] != v;
            prog.push_back(others);
            for (int j = par_ptr[ch]; j < par_ptr[ch + 1]; ++j)
                if (par_idx[j] != v) {
                    prog.push_back(par_idx[j]);
                    prog.push_back(par_stride[j]);
                }
        }
    }
    // the straight-line variant (sbn_gibbs_flat_kernel): fixed-size records, when the network is small enough
    std::vector<int32_t> flat;
    bool flat_ok = max_card <= 8 && n_query <= 4 && n_vars < 0xffff;
    const int32_t ones_off = static_cast<int32_t>(n_table_floats);  // a 1.0f appended to the table blob
    for (int i = 0; i < n_cycle && flat_ok; ++i) {
        const int v = cycle[i];
        const int np = par_ptr[v + 1] - par_ptr[v], nc = chi_ptr[v + 1] - chi_ptr[v];
        if (np > SBN_GF_TERMS || nc > SBN_GF_GROUPS - 1) { flat_ok = false; break; }
        std::vector<int32_t> rec(SBN_GF_WORDS, 0);
        rec[0] = v | card[v] << 16;
        auto group = [&](int g) { return rec.data() + 2 + g * (2 + 2 * SBN_GF_TERMS); };
        for (int g = 0; g < SBN_GF_GROUPS; ++g) {  // padding: the constant 1.0, terms on the dummy state
            int32_t *gw = group(g);
            gw[0] = ones_off;
            gw[1] = 0;
            for (int k = 0; k < SBN_GF_TERMS; ++k) { gw[2 + 2 * k] = n_vars; gw[3 + 2 * k] = 0; }
        }
        int32_t *g0 = group(0);
        g0[0] = cpt_off[v];
        g0[1] = 1;
        for (int k = par_ptr[v], t = 0; k < par_ptr[v + 1]; ++k, ++t) { g0[2 + 2 * t] = par_idx[k]; g0[3 + 2 * t] = par_stride[k]; }
        for (int k = chi_ptr[v], g = 1; k < chi_ptr[v + 1] && flat_ok; ++k, ++g) {
            const int ch = chi_idx[k];
            int32_t *gw = group(g);
            gw[0] = cpt_off[ch];
            gw[1] = chi_stride[k];
            int t = 0;
            gw[2] = ch;  // the child's own state, stride 1
            gw[3] = 1;
            ++t;
            for (int j = par_ptr[ch]; j < par_ptr[ch + 1]; ++j)
                if (par_idx[j] != v) {
                    if (t >= SBN_GF_TERMS) { flat_ok = false; break; }
                    gw[2 + 2 * t] = par_idx[j];
                    gw[3 + 2 * t] = par_stride[j];
                    ++t;
                }
        }
        flat.insert(flat.end(), rec.begin(), rec.end());
    }
    if (flat_ok) {
        const size_t need = flat.size() * 4 + ((static_cast<size_t>(n_table_floats) + 1 + 3) / 4) * 16 +
                            ((static_cast<size_t>(n_vars + 1) * SBN_GIBBS_CHAINS + 15) / 16) * 16 + static_cast<size_t>(Q) * SBN_GIBBS_CHAINS * 4;
        if (need > 100 * 1024) flat_ok = false;  // two CTAs per SM
    }
    const size_t smem_min = ((prog.size() + 3) / 4) * 16 + ((static_cast<size_t>(n_vars) * SBN_GIBBS_CHAINS + 15) / 16) * 16 +
                            static_cast<size_t>(Q) * SBN_GIBBS_CHAINS * 4;
    if (smem_min > 200 * 1024) return fail(SBN_E_INVALID, "chain state needs %zu bytes of shared memory per CTA", smem_min);

    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(SBN_E_NODEVICE, "no CUDA device available");
    if (device < 0 || device >= n_dev) return fail(SBN_E_NODEVICE, "device %d out of range", device);
    sbn_sampler *S = new sbn_sampler();
    S->device = device;
    S->n_vars = n_vars;
    S->n_query = n_query;
    S->n_ev = n_ev;
    S->n_cycle = n_cycle;
    S->Q = static_cast<int>(Q);
    auto bail = [&](int code) {
        sbn_gibbs_destroy(S);
        return code;
    };
#define SBN_CUDA_S(call)                                                                                   \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess) return bail(fail(SBN_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_))); \
    } while (0)
    SBN_CUDA_S(cudaSetDevice(device));
    SBN_CUDA_S(cudaStreamCreateWithFlags(&S->stream, cudaStreamNonBlocking));
    std::vector<int32_t> ints;
    auto put = [&](const int32_t *src, size_t n) {
        const size_t at = ints.size();
        ints.insert(ints.end(), src, src + n);
        return at;
    };
    const size_t o_card = put(card, n_vars), o_off = put(cpt_off, n_vars), o_pp = put(par_ptr, n_vars + 1),
                 o_pi = put(par_idx ? par_idx : card, n_par), o_ps = put(par_stride.data(), n_par),
                 o_cp = put(chi_ptr.data(), n_vars + 1), o_ci = put(chi_idx.data(), n_par),
                 o_cs = put(chi_stride.data(), n_par), o_cy = put(cycle, n_cycle), o_q = put(query, n_query),
                 o_ev = put(ev_vars ? ev_vars : card, n_ev), o_prog = put(prog.data(), prog.size());
    while (ints.size() % 4) ints.push_back(0);  // the flat records are read as int4
    const size_t o_flat = put(flat.data(), flat_ok ? flat.size() : 0);
    SBN_CUDA_S(cudaMalloc(&S->d_ints, ints.size() * 4 + 4));
    SBN_CUDA_S(cudaMemcpyAsync(S->d_ints, ints.data(), ints.size() * 4, cudaMemcpyHostToDevice, S->stream));
    SBN_CUDA_S(cudaMalloc(&S->d_tables, static_cast<size_t>(n_table_floats + 1) * 4));
    SBN_CUDA_S(cudaMemcpyAsync(S->d_tables, tables, static_cast<size_t>(n_table_floats) * 4, cudaMemcpyHostToDevice, S->stream));
    {
        static const float one = 1.0f;  // the padding entry of the straight-line records
        SBN_CUDA_S(cudaMemcpyAsync(S->d_tables + n_table_floats, &one, 4, cudaMemcpyHostToDevice, S->stream));
    }
    SBN_CUDA_S(cudaStreamSynchronize(S->stream));
    S->card = S->d_ints + o_card;
    S->cpt_off = S->d_ints + o_off;
    S->par_ptr = S->d_ints + o_pp;
    S->par_idx = S->d_ints + o_pi;
    S->par_stride = S->d_ints + o_ps;
    S->chi_ptr = S->d_ints + o_cp;
    S->chi_idx = S->d_ints + o_ci;
    S->chi_stride = S->d_ints + o_cs;
    S->cycle = S->d_ints + o_cy;
    S->query = S->d_ints + o_q;
    S->ev_var = S->d_ints + o_ev;
    S->prog = S->d_ints + o_prog;
    S->prog_words = static_cast<int>(prog.size());
    S->flat = flat_ok ? S->d_ints + o_flat : nullptr;
    S->flat_words = flat_ok ? static_cast<int>(flat.size()) : 0;
    SBN_CUDA_S(cudaFuncSetAttribute(sbn_gibbs_flat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    S->table_floats = n_table_floats;
    S->max_card = max_card;
    S->h_cycle.assign(cycle, cycle + n_cycle);
    S->h_card.assign(card, card + n_vars);
    SBN_CUDA_S(cudaFuncSetAttribute(sbn_gibbs_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    SBN_CUDA_S(cudaFuncSetAttribute(sbn_gibbs_kernel<SBN_GIBBS_MAX_CARD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    SBN_CUDA_S(cudaFuncSetAttribute(sbn_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
#undef SBN_CUDA_S
    *out = S;
    return SBN_OK;
}

void sbn_gibbs_destroy(sbn_sampler *S) {
    if (!S) return;
    cudaSetDevice(S->device);
    cudaFree(S->d_ints);
    cudaFree(S->d_tables);
    cudaFree(S->d_ev);
    cudaFree(S->d_out);
    if (S->stream) cudaStreamDestroy(S->stream);
    delete S;
}

static int sampler_run(sbn_sampler *S, int algo, const uint8_t *ev, int64_t ld_ev, int64_t n_chains, int64_t n_iterations,
                       uint64_t seed, float *out, int64_t ld_out) {
    if (!S || !out) return fail(SBN_E_INVALID, "null argument");
    const bool force_generic = algo == 3;  // Gibbs through the generic kernel (cross-check of the straight-line one)
    if (algo == 3) algo = 0;
    if (algo < 0 || algo > 2) return fail(SBN_E_INVALID, "unknown sampling algorithm %d", algo);
    if (n_chains <= 0 || n_iterations <= 0) return fail(SBN_E_INVALID, "n_chains and n_iterations must be positive");
    if (S->n_ev > 0 && (!ev || (S->n_ev > 1 && ld_ev < n_chains))) return fail(SBN_E_INVALID, "bad evidence");
    if (S->Q > 1 && ld_out < n_chains) return fail(SBN_E_INVALID, "ld_out < n_chains");
    SBN_CUDA(cudaSetDevice(S->device));
    if (n_chains > S->cap) {
        cudaFree(S->d_ev);
        cudaFree(S->d_out);
        S->d_ev = nullptr;
        S->d_out = nullptr;
        if (S->n_ev > 0) SBN_CUDA(cudaMalloc(&S->d_ev, static_cast<size_t>(S->n_ev) * n_chains));
        SBN_CUDA(cudaMalloc(&S->d_out, static_cast<size_t>(S->Q) * n_chains * 4));
        S->cap = n_chains;
    }
    if (S->n_ev > 0)
        SBN_CUDA(cudaMemcpy2DAsync(S->d_ev, static_cast<size_t>(n_chains), ev, static_cast<size_t>(ld_ev),
                                   static_cast<size_t>(n_chains), static_cast<size_t>(S->n_ev), cudaMemcpyHostToDevice, S->stream));
    SbnGibbs g;
    memset(&g, 0, sizeof g);
    g.n_vars = S->n_vars;
    g.n_cycle = S->n_cycle;
    g.n_query = S->n_query;
    g.Q = S->Q;
    g.n_ev = S->n_ev;
    g.card = S->card;
    g.cpt_off = S->cpt_off;
    g.par_ptr = S->par_ptr;
    g.par_idx = S->par_idx;
    g.par_stride = S->par_stride;
    g.chi_ptr = S->chi_ptr;
    g.chi_idx = S->chi_idx;
    g.chi_stride = S->chi_stride;
    g.cycle = S->cycle;
    g.query = S->query;
    g.ev_var = S->ev_var;
    g.tables = S->d_tables;
    g.ev = S->d_ev;
    g.ld_ev = n_chains;
    g.out = S->d_out;
    g.ld_out = n_chains;
    g.n_chains = n_chains;
    g.n_iterations = n_iterations;
    g.seed = seed;
    g.prog = S->prog;
    g.prog_words = S->prog_words;
    g.table_floats = static_cast<int32_t>(S->table_floats);
    static const bool flat_env = [] {
        const char *e = getenv("SOROBN_B200_GIBBS_FLAT");
        return e ? atoi(e) != 0 : true;
    }();
    if (algo == 0 && S->flat && flat_env && !force_generic) {
        g.prog = S->flat;
        g.prog_words = S->flat_words;
        g.table_floats = static_cast<int32_t>(S->table_floats + 1);
        g.tables_in_smem = 1;
        const size_t smem = static_cast<size_t>(S->flat_words) * 4 + ((static_cast<size_t>(g.table_floats) + 3) / 4) * 16 +
                            ((static_cast<size_t>(S->n_vars + 1) * SBN_GIBBS_CHAINS + 15) / 16) * 16 + static_cast<size_t>(S->Q) * SBN_GIBBS_CHAINS * 4;
        const int64_t grid = (n_chains + SBN_GIBBS_CHAINS - 1) / SBN_GIBBS_CHAINS;
        sbn_gibbs_flat_kernel<<<static_cast<unsigned>(grid), SBN_GIBBS_CHAINS, smem, S->stream>>>(g);
    } else if (algo == 0) {
        const size_t base = ((static_cast<size_t>(S->prog_words) + 3) / 4) * 16 + ((static_cast<size_t>(S->n_vars) * SBN_GIBBS_CHAINS + 15) / 16) * 16 +
                            static_cast<size_t>(S->Q) * SBN_GIBBS_CHAINS * 4;
        const size_t tab = ((static_cast<size_t>(S->table_floats) + 3) / 4) * 16;
        // every CPT in shared memory when that still leaves two CTAs per SM
        g.tables_in_smem = base + tab <= 100 * 1024 ? 1 : 0;
        const size_t smem = base + (g.tables_in_smem ? tab : 0);
        const int64_t grid = (n_chains + SBN_GIBBS_CHAINS - 1) / SBN_GIBBS_CHAINS;
        if (S->max_card <= 8) sbn_gibbs_kernel<8><<<static_cast<unsigned>(grid), SBN_GIBBS_CHAINS, smem, S->stream>>>(g);
        else sbn_gibbs_kernel<SBN_GIBBS_MAX_CARD><<<static_cast<unsigned>(grid), SBN_GIBBS_CHAINS, smem, S->stream>>>(g);
    } else {
        // one CTA per evidence row; its threads share the row's n_iterations samples
        const size_t smem = ((static_cast<size_t>(S->n_vars) * (SBN_GIBBS_THREADS + 1) + 15) / 16) * 16 + static_cast<size_t>(S->Q) * 8;
        if (smem > 200 * 1024) return fail(SBN_E_INVALID, "sampler state needs %zu bytes of shared memory", smem);
        sbn_forward_kernel<<<static_cast<unsigned>(n_chains), SBN_GIBBS_THREADS, smem, S->stream>>>(g, algo);
    }
    SBN_CUDA(cudaGetLastError());
    S->launches++;
    SBN_CUDA(cudaMemcpy2DAsync(out, static_cast<size_t>(ld_out) * 4, S->d_out, static_cast<size_t>(n_chains) * 4,
                               static_cast<size_t>(n_chains) * 4, static_cast<size_t>(S->Q), cudaMemcpyDeviceToHost, S->stream));
    SBN_CUDA(cudaStreamSynchronize(S->stream));
    return SBN_OK;
}

int sbn_gibbs_conditional(sbn_sampler *S, int32_t var, const uint8_t *joint, float *out) {
    if (!S || !joint || !out) return fail(SBN_E_INVALID, "null argument");
    int pos = -1;
    for (size_t i = 0; i < S->h_cycle.size(); ++i)
        if (S->h_cycle[i] == var) pos = static_cast<int>(i);
    if (pos < 0) return fail(SBN_E_INVALID, "variable %d is not in the sampler's cycle", var);
    SBN_CUDA(cudaSetDevice(S->device));
    uint8_t *d_joint = nullptr;
    float *d_w = nullptr;
    SBN_CUDA(cudaMalloc(&d_joint, static_cast<size_t>(S->n_vars)));
    SBN_CUDA(cudaMalloc(&d_w, SBN_GIBBS_MAX_CARD * sizeof(float)));
    SBN_CUDA(cudaMemcpyAsync(d_joint, joint, static_cast<size_t>(S->n_vars), cudaMemcpyHostToDevice, S->stream));
    SbnGibbs g;
    memset(&g, 0, sizeof g);
    g.card = S->card;
    g.prog = S->prog;
    g.tables = S->d_tables;
    sbn_gibbs_conditional_kernel<<<1, 32, 0, S->stream>>>(g, pos, d_joint, d_w);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(out, d_w, static_cast<size_t>(S->h_card[var]) * sizeof(float), cudaMemcpyDeviceToHost, S->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(S->stream);
    cudaFree(d_joint);
    cudaFree(d_w);
    if (e != cudaSuccess) return fail(SBN_E_CUDA, "sbn_gibbs_conditional failed: %s", cudaGetErrorString(e));
    return SBN_OK;
}

int sbn_gibbs_run_host(sbn_sampler *S, const uint8_t *ev, int64_t ld_ev, int64_t n_chains, int64_t n_iterations,
                       uint64_t seed, float *out, int64_t ld_out) {
    return sampler_run(S, 0, ev, ld_ev, n_chains, n_iterations, seed, out, ld_out);
}

int sbn_sampler_run_host(sbn_sampler *S, int algo, const uint8_t *ev, int64_t ld_ev, int64_t n_rows, int64_t n_iterations,
                         uint64_t seed, float *out, int64_t ld_out) {
    return sampler_run(S, algo, ev, ld_ev, n_rows, n_iterations, seed, out, ld_out);
}

}  // extern "C"
