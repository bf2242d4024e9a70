// Two-state chain DP as a parallel scan of clamp-add maps, and the batched multiplier search.
//
// Replaces /root/reference/rocco/_chain_dp.c:109-186 (sequential Viterbi with back-pointers) and
// /root/reference/rocco/dp.py:89-164 (bisection driven from Python, 62 DP passes).
//
// With V0/V1 the best values ending unselected/selected, d = V1 - V0 obeys
//     d_0 = s_0 - lambda,     d_i = min(max(d_{i-1}, -c_{i-1}), c_{i-1}) + (s_i - lambda)
// and the back-pointers collapse to: z_{n-1} = [d_{n-1} > 0];  z_i = 1 if d_i > c_i, 0 if d_i < -c_i,
// else z_{i+1}.  Each step is a map x -> min(max(x + p, lo), hi); such maps are closed under
// composition, so the forward sweep is an associative scan (per-thread serial compose, warp-shuffle
// scan, decoupled look-back across tiles) and the backward pointer chase becomes a "nearest decided
// bin to the right" propagation resolved inside the tile, with only the undecided tile suffix
// deferred to a tiny per-chromosome pass.
//
// Tie-break fidelity: the reference compares (value, fewer selected bins) lexicographically.  Values
// here are either plain doubles (VD, fast path) or (double, int) pairs ordered lexicographically (VL).
// The fast path counts every decision that lands exactly on a threshold; if any occurred for a
// multiplier, that multiplier is re-solved with VL, which is the reference's rule restated on d.
#include "common.cuh"

#include <math.h>

#include <algorithm>
#include <cmath>

namespace rb {
namespace chain {

constexpr int THREADS = 256;
constexpr int ITEMS = 16;
constexpr int TILE = THREADS * ITEMS;   // 4096 bins per tile
constexpr int WARPS = THREADS / 32;
constexpr int PAD_STRIDE = ITEMS + 1;   // smem padding: conflict-free blocked reads
constexpr int MAX_LEVELS = 8;
constexpr int MAX_SLOTS = 256;          // multipliers per launch set

// ------------------------------------------------------------------ value types
struct VD { double v; };
struct VL { double v; int k; };          // k = selected-count difference; fewer is better

__device__ __forceinline__ VD v_make(VD *, double v, int) { return VD{v}; }
__device__ __forceinline__ VL v_make(VL *, double v, int k) { return VL{v, k}; }
__device__ __forceinline__ VD v_add(VD a, VD b) { return VD{a.v + b.v}; }
__device__ __forceinline__ VL v_add(VL a, VL b) { return VL{a.v + b.v, a.k + b.k}; }
// strict "a is worse than b"
__device__ __forceinline__ bool v_lt(VD a, VD b) { return a.v < b.v; }
__device__ __forceinline__ bool v_lt(VL a, VL b) { return a.v < b.v || (a.v == b.v && a.k > b.k); }
__device__ __forceinline__ bool v_eq(VD a, VD b) { return a.v == b.v; }
__device__ __forceinline__ bool v_eq(VL a, VL b) { return a.v == b.v && a.k == b.k; }
template <typename V> __device__ __forceinline__ V v_max(V a, V b) { return v_lt(a, b) ? b : a; }
template <typename V> __device__ __forceinline__ V v_min(V a, V b) { return v_lt(b, a) ? b : a; }
// plain doubles: the same selections as one compare + select (rb::dmax / rb::dmin; ties keep a, as above)
template <> __device__ __forceinline__ VD v_max<VD>(VD a, VD b) { return VD{dmax(b.v, a.v)}; }
template <> __device__ __forceinline__ VD v_min<VD>(VD a, VD b) { return VD{dmin(b.v, a.v)}; }
template <typename V> __device__ __forceinline__ V v_clamp(V x, V lo, V hi) { return v_min(v_max(x, lo), hi); }
__device__ __forceinline__ VD v_shfl_up(VD a, int d) { return VD{__shfl_up_sync(0xffffffffu, a.v, d)}; }
__device__ __forceinline__ VL v_shfl_up(VL a, int d) {
    return VL{__shfl_up_sync(0xffffffffu, a.v, d), __shfl_up_sync(0xffffffffu, a.k, d)};
}

template <typename V> struct Map { V p, lo, hi; };   // x -> min(max(x + p, lo), hi)

template <typename V> __device__ __forceinline__ Map<V> map_identity() {
    V *t = nullptr;
    return Map<V>{v_make(t, 0.0, 0), v_make(t, -INFINITY, 0), v_make(t, INFINITY, 0)};
}
template <typename V> __device__ __forceinline__ Map<V> map_const(V a) {
    V *t = nullptr;
    return Map<V>{v_make(t, 0.0, 0), a, a};
}
// apply f first, then g
template <typename V> __device__ __forceinline__ Map<V> map_compose(const Map<V> &f, const Map<V> &g) {
    Map<V> r;
    r.p = v_add(f.p, g.p);
    r.lo = v_clamp(v_add(f.lo, g.p), g.lo, g.hi);
    r.hi = v_clamp(v_add(f.hi, g.p), g.lo, g.hi);
    return r;
}
template <typename V> __device__ __forceinline__ V map_apply(const Map<V> &f, V x) {
    return v_clamp(v_add(x, f.p), f.lo, f.hi);
}
// one DP step appended to f: clamp to [-c, c], then add a
template <typename V> __device__ __forceinline__ Map<V> map_step(const Map<V> &f, V a, V cneg, V cpos) {
    Map<V> r;
    r.p = v_add(f.p, a);
    r.lo = v_add(v_clamp(f.lo, cneg, cpos), a);
    r.hi = v_add(v_clamp(f.hi, cneg, cpos), a);
    return r;
}
template <typename V> __device__ __forceinline__ Map<V> map_shfl_up(const Map<V> &m, int d) {
    return Map<V>{v_shfl_up(m.p, d), v_shfl_up(m.lo, d), v_shfl_up(m.hi, d)};
}
// L2-coherent reads of look-back payloads written by other blocks
__device__ __forceinline__ VD v_ldcg(const VD *p) { return VD{__ldcg(&p->v)}; }
__device__ __forceinline__ VL v_ldcg(const VL *p) { return VL{__ldcg(&p->v), __ldcg(&p->k)}; }
template <typename V> __device__ __forceinline__ Map<V> map_ldcg(const Map<V> *m) {
    return Map<V>{v_ldcg(&m->p), v_ldcg(&m->lo), v_ldcg(&m->hi)};
}

// ------------------------------------------------------------------ device-side descriptors
struct ChromDev {
    long long offset;       // element offset of this chromosome in the concatenated arrays
    long long n;
    double gamma;
    double cost_sum;
    long long target;
    int tile0;              // first tile index
    int ntiles;
    int mode;               // 0 fixed multiplier, 1 budget search
    int max_iter;
    int seq;                // 1: short chromosome solved by the exact sequential kernel (one tile)
    int pad;
};

enum Phase : int { PH_BRACKET = 0, PH_BISECT = 1, PH_DONE = 2, PH_HOST = 3, PH_MANUAL = 4 };

struct SearchDev {
    double lower, upper;
    double smin, smax;
    int phase;
    int iters_left;
    int levels;             // levels (=> 2^levels - 1 slots) of the round in flight
    int nslots;             // active multipliers this round
    int need_lex;
    int passes;
    int rounds;
    int pad;
};

struct TileOut { int cnt; int pend; int head; int ties; };   // head: 0/1 value, 2 = whole tile undecided
// multiplier sweep only: objective pieces of the tile (resolved = bins up to the tile's last decided bin)
struct TileSweep { double ssz; double spend; int sw; int zp; };

struct Params {
    const double *scores;
    const double *costs;        // nullable
    const ChromDev *chroms;
    SearchDev *search;
    const int *tile_chrom;
    double *lam;                // [nchrom][MAX_SLOTS]
    long long *counts;          // [nchrom][MAX_SLOTS]
    long long *tiecnt;          // [nchrom][MAX_SLOTS]
    int *flags;                 // [slot][tile]  (epoch<<2 | state)
    void *agg;                  // [slot][tile] Map<V>
    void *incl;                 // [slot][tile] V
    TileOut *tout;              // [slot][tile]
    int *ticket;
    uint8_t *mask;              // EMIT only
    int *zin;                   // [tile]  EMIT: value flowing into the tile from the right
    long long *near_ties;       // [nchrom] EMIT only
    TileSweep *tsweep;          // [slot][tile]  (nullptr unless sweeping)
    double *sweep_ssz;          // [nchrom][MAX_SLOTS] sum s*z
    long long *sweep_sw;        // [nchrom][MAX_SLOTS] switches
    uint8_t *bt;                // [ntiles * TILE] back-pointers of the sequential kernel (EMIT only)
    double *seq_value;          // [nchrom] DP best value of the sequential kernel (EMIT only)
    int ntiles;
    int nchrom;
    int slots_per_block;        // multipliers handled sequentially by one block
    int ngroups;                // ceil(max nslots / slots_per_block)
    int epoch;
    int lex_pass;               // 1: only chromosomes with need_lex
    int exact_mode;             // 1: multipliers with a decision inside the reference's rounding noise are replayed sequentially
    // tile freezing (search rounds; nullptr: off).  state bit 0: every decision of the tile is stable over the whole current
    // bracket and its last bin is saturated; read buffer = previous round, write buffer = this round
    const int *fz_read;
    int *fz_write;
    TileOut *fz_out;            // [tile] the tile's fixed outputs
    double *fz_incl;            // [tile] +-HUGE: the saturated value it hands to its successor
    // adaptive tree depth (nullptr: off): tiles that did real work in round r are counted in live_cnt[r & 1]; while that
    // stays above live_threshold the rounds are throughput-bound and the controller asks for ONE level per round (a deeper
    // tree evaluates 2^L - 1 multipliers to advance L levels); below it rounds are latency-bound and take levels_base
    int *live_cnt;
    int round_id;
    int levels_base;
    int live_threshold;
    int group;                  // 1: genome mode, the members' search is driven by the group controller (k_genome_control)
};

// ------------------------------------------------------------------ the tile kernel
template <typename V, bool VEC_COST, bool EMIT>
__global__ void __launch_bounds__(THREADS, 4) k_chain_tiles(Params P)
{
    extern __shared__ double smem[];
    double *s_sc = smem;                               // TILE + THREADS (padded)
    double *s_cs = smem + (TILE + THREADS);            // VEC_COST only: TILE + 1 + padding
    __shared__ Map<V> s_wtot[WARPS];
    __shared__ V s_din;
    __shared__ int s_ticket;
    __shared__ int s_whas[WARPS], s_whead[WARPS];
    __shared__ int s_red[WARPS][4];
    __shared__ double s_sw_d[WARPS][2];
    __shared__ int s_sw_i[WARPS][2];
    __shared__ int s_firstz[WARPS];

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) s_ticket = atomicAdd(P.ticket, 1);
    __syncthreads();
    const int ticket = s_ticket;
    const int group = ticket % P.ngroups;
    const int tile = ticket / P.ngroups;
    const int c = P.tile_chrom[tile];
    const ChromDev cd = P.chroms[c];
    const SearchDev sd = P.search[c];
    if (cd.seq) return;
    if (P.lex_pass ? (sd.need_lex == 0) : (sd.phase == PH_DONE && !EMIT) || sd.phase == PH_HOST) return;
    const int slot0 = group * P.slots_per_block;
    if (slot0 >= sd.nslots) return;
    const int slot1 = min(sd.nslots, slot0 + P.slots_per_block);

    const long long s0 = (long long)(tile - cd.tile0) * TILE;     // first bin of this tile
    const int len = (int)min((long long)TILE, cd.n - s0);
    const bool first_tile = (tile == cd.tile0);
    const bool last_tile = (s0 + len == cd.n);
    const double *gsc = P.scores + cd.offset + s0;

    // ---- frozen tiles.  d_i(lambda) moves by at most len_i |dlambda|, len_i = 1 + the number of unsaturated bins
    // right before i, so a bin whose distance to both thresholds exceeds len_i x (bracket width) keeps its decision class
    // for every multiplier the bisection can still visit (the bracket only shrinks).  A tile all of whose bins are that
    // stable, whose last bin is saturated and whose predecessor ends saturated and stable, contributes the same
    // (count, pending, head) to every later round and hands the same clamp value on: it is answered from the values
    // stored when that was established (previous round's buffer) without touching its scores again.
    const bool fz_on = !EMIT && P.fz_read != nullptr && sd.phase == PH_BISECT;
    if (fz_on) {
        const bool frozen = (P.fz_read[tile] & 1) && (first_tile || (P.fz_read[tile - 1] & 1));
        if (frozen) {
            if (tid == 0) {
                V *gincl = reinterpret_cast<V *>(P.incl);
                V *tv0 = nullptr;
                const TileOut o = P.fz_out[tile];
                for (int slot = slot0; slot < slot1; ++slot) {
                    const size_t sidx = (size_t)slot * P.ntiles + tile;
                    P.tout[sidx] = o;
                    gincl[sidx] = v_make(tv0, P.fz_incl[tile], 0);
                    st_release_i32(P.flags + sidx, (P.epoch << 2) | 2);
                }
                if (group == 0 && !P.lex_pass) P.fz_write[tile] = P.fz_read[tile];
            }
            return;
        }
    }
    if (!EMIT && P.live_cnt && !P.lex_pass && group == 0 && tid == 0) atomicAdd(&P.live_cnt[P.round_id & 1], 1);
    const bool fz_eval = fz_on && !P.lex_pass && group == 0;       // this CTA establishes the tile's state for the next round
    const double fz_width = sd.upper - sd.lower;
    __shared__ int s_fzlen[WARPS];
    __shared__ int s_fzlast;

    // stage scores (coalesced) into the padded blocked layout: all of a thread's loads are issued before the first store
    // (eight at a time; sixteen dependent round trips to DRAM per thread otherwise: a third of a search round)
#pragma unroll
    for (int k0 = 0; k0 < ITEMS; k0 += 8) {
        double v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int e = tid + (k0 + k) * THREADS; v[k] = (e < len) ? __ldg(gsc + e) : 0.0; }
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int e = tid + (k0 + k) * THREADS; s_sc[e + e / ITEMS] = v[k]; }
    }
    if (VEC_COST) {
        // s_cs[e] = cost between bins (s0+e-1) and (s0+e);  e in [0, TILE]
        const double *gcs = P.costs + cd.offset + s0 - 1;
        for (int e = tid; e <= TILE; e += THREADS) {
            double v = 0.0;
            if (e <= len && (s0 + e) >= 1 && (s0 + e) < cd.n) v = __ldg(gcs + e);
            s_cs[e + e / ITEMS] = v;
        }
    }
    __syncthreads();

    double sc[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) sc[j] = s_sc[tid * PAD_STRIDE + j];
    const int base = tid * ITEMS;
    const int cnt = max(0, min(ITEMS, len - base));               // valid items of this thread
    const unsigned vm = (cnt >= 32) ? 0xffffffffu : ((1u << cnt) - 1u);
    V *tv = nullptr;

    for (int slot = slot0; slot < slot1; ++slot) {
        const double lam = P.lam[(size_t)c * MAX_SLOTS + slot];
        const size_t sidx = (size_t)slot * P.ntiles + tile;

        // ---- pass 1: compose this thread's maps
        Map<V> m = map_identity<V>();
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            if (j < cnt) {
                const V a = v_make(tv, sc[j] - lam, 1);
                if (first_tile && base + j == 0) {
                    m = map_const<V>(a);
                } else {
                    const double cc = VEC_COST ? s_cs[(base + j) + (base + j) / ITEMS] : cd.gamma;
                    m = map_step<V>(m, a, v_make(tv, -cc, 0), v_make(tv, cc, 0));
                }
            }
        }
        // ---- block scan (inclusive within warp)
        Map<V> inc = m;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            Map<V> o = map_shfl_up<V>(inc, d);
            if (lane >= d) inc = map_compose<V>(o, inc);
        }
        if (lane == 31) s_wtot[wid] = inc;
        Map<V> excl = map_shfl_up<V>(inc, 1);
        if (lane == 0) excl = map_identity<V>();
        __syncthreads();
        Map<V> wpre = map_identity<V>();
        for (int w = 0; w < wid; ++w) wpre = map_compose<V>(wpre, s_wtot[w]);
        excl = map_compose<V>(wpre, excl);

        // ---- publish + decoupled look-back (one thread)
        if (tid == 0) {
            Map<V> A = s_wtot[0];
            for (int w = 1; w < WARPS; ++w) A = map_compose<V>(A, s_wtot[w]);
            Map<V> *gagg = reinterpret_cast<Map<V> *>(P.agg);
            V *gincl = reinterpret_cast<V *>(P.incl);
            V din = v_make(tv, 0.0, 0);
            const bool is_const = v_eq(A.lo, A.hi);
            if (first_tile || is_const) {
                gincl[sidx] = A.lo;
                st_release_i32(P.flags + sidx, (P.epoch << 2) | 2);
            } else {
                gagg[sidx] = A;
                st_release_i32(P.flags + sidx, (P.epoch << 2) | 1);
            }
            if (!first_tile) {
                Map<V> acc = map_identity<V>();
                size_t j = sidx - 1;
                for (;;) {
                    int f = ld_acquire_i32(P.flags + j);
                    if ((f >> 2) != P.epoch || (f & 3) == 0) { __nanosleep(20); continue; }
                    if ((f & 3) == 2) {
                        V x = v_ldcg(gincl + j);
                        din = map_apply<V>(acc, x);
                        break;
                    }
                    Map<V> a = map_ldcg<V>(gagg + j);
                    acc = map_compose<V>(a, acc);
                    --j;
                }
                if (!is_const) {
                    gincl[sidx] = map_apply<V>(A, din);
                    st_release_i32(P.flags + sidx, (P.epoch << 2) | 2);
                }
            }
            s_din = din;
        }
        __syncthreads();

        // ---- pass 2: actual d values, decisions
        V x = map_apply<V>(excl, s_din);
        unsigned dec = 0, val = 0;
        int ties = 0, near = 0;
        const bool fz_track = fz_eval && slot == slot0;
        int fz_run = 0, fz_sat = 0, fz_lastok = 0;       // bins since the last saturated one in this chunk; any saturated bin; last bin of the tile stable
        double fz_a = INFINITY, fz_b = INFINITY;         // min slack of the bins before / after the chunk's first saturated bin
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            if (j < cnt) {
                const V a = v_make(tv, sc[j] - lam, 1);
                const long long gi = s0 + base + j;
                if (gi == 0) {
                    x = a;
                } else {
                    const double cc = VEC_COST ? s_cs[(base + j) + (base + j) / ITEMS] : cd.gamma;
                    x = v_add(v_clamp(x, v_make(tv, -cc, 0), v_make(tv, cc, 0)), a);
                }
                if (fz_track) {
                    const bool term = (gi == cd.n - 1);
                    const double cr_ = term ? 0.0 : (VEC_COST ? s_cs[(base + j + 1) + (base + j + 1) / ITEMS] : cd.gamma);
                    const double margin = term ? fabs(x.v) : dmin(fabs(x.v - cr_), fabs(x.v + cr_));
                    fz_run += 1;
                    const double slack = margin - (double)fz_run * fz_width;
                    if (fz_sat) fz_b = dmin(slack, fz_b); else fz_a = dmin(slack, fz_a);
                    const bool sat = term || x.v > cr_ || x.v < -cr_;
                    if (base + j == len - 1) fz_lastok = sat ? 1 : 0;
                    if (sat) { fz_sat = 1; fz_run = 0; }
                }
                if (gi == cd.n - 1) {                 // terminal choice (_chain_dp.c:167-179)
                    dec |= 1u << j;
                    if (v_lt(v_make(tv, 0.0, 0), x)) val |= 1u << j;
                    ties += (x.v == 0.0);
                    if (P.exact_mode) near += (fabs(x.v) <= 1.0e-7);
                } else {
                    const double cr = VEC_COST ? s_cs[(base + j + 1) + (base + j + 1) / ITEMS] : cd.gamma;
                    if (v_lt(v_make(tv, cr, 0), x)) { dec |= 1u << j; val |= 1u << j; }
                    else if (v_lt(x, v_make(tv, -cr, 0))) { dec |= 1u << j; }
                    ties += (x.v == cr) || (x.v == -cr);
                    if (EMIT || P.exact_mode) {
                        const double tol = (P.exact_mode ? 1.0e-7 : 1.0e-9) * (1.0 + fabs(cr));
                        near += (fabs(x.v - cr) <= tol) || (fabs(x.v + cr) <= tol);
                    }
                }
            }
        }

        // ---- backward: nearest decided bin to the right
        const int has = dec != 0;
        const int headv = has ? ((val >> (__ffs(dec) - 1)) & 1) : 0;
        const unsigned D = __ballot_sync(0xffffffffu, has);
        const unsigned Hv = __ballot_sync(0xffffffffu, headv);
        if (lane == 0) {
            s_whas[wid] = D != 0;
            s_whead[wid] = D ? ((Hv >> (__ffs(D) - 1)) & 1) : 0;
        }
        __syncthreads();
        int known = 0, zin = 0;
        {
            const unsigned above = D & ~((2u << lane) - 1u);
            if (above) { known = 1; zin = (Hv >> (__ffs(above) - 1)) & 1; }
            else {
                for (int w = wid + 1; w < WARPS; ++w)
                    if (s_whas[w]) { known = 1; zin = s_whead[w]; break; }
            }
        }
        unsigned z = 0;
        {
            int cur = known ? zin : 0;
#pragma unroll
            for (int j = ITEMS - 1; j >= 0; --j) {
                if ((dec >> j) & 1u) cur = (val >> j) & 1u;
                z |= (unsigned)cur << j;
            }
        }
        z &= vm;
        unsigned pm = 0;                         // items that copy the (unknown) value from the right
        if (!known) pm = (dec ? ~((2u << (31 - __clz(dec))) - 1u) : 0xffffffffu) & vm;

        int r_cnt = __popc(z), r_pend = __popc(pm), r_ties = ties, r_near = near;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            r_cnt += __shfl_xor_sync(0xffffffffu, r_cnt, d);
            r_pend += __shfl_xor_sync(0xffffffffu, r_pend, d);
            r_ties += __shfl_xor_sync(0xffffffffu, r_ties, d);
            r_near += __shfl_xor_sync(0xffffffffu, r_near, d);
        }
        if (lane == 0) { s_red[wid][0] = r_cnt; s_red[wid][1] = r_pend; s_red[wid][2] = r_ties; s_red[wid][3] = r_near; }

        if (P.tsweep) {
            const unsigned rm = vm & ~pm;                          // resolved items of this thread
            double ssz = 0.0, spend = 0.0;
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                if ((z >> j) & (rm >> j) & 1u) ssz += sc[j];
                if ((pm >> j) & 1u) spend += sc[j];
            }
            int sw = __popc((z ^ (z >> 1)) & rm & (rm >> 1) & ((1u << (ITEMS - 1)) - 1u));
            // pair (last item of this thread, first item of the next thread)
            const unsigned firstinfo = (rm & 1u) | ((z & 1u) << 1);
            unsigned nxt = __shfl_down_sync(0xffffffffu, firstinfo, 1);
            if (lane == 0) s_firstz[wid] = (int)firstinfo;
            __syncthreads();
            if (lane == 31) nxt = (wid + 1 < WARPS) ? (unsigned)s_firstz[wid + 1] : 0u;
            if (cnt == ITEMS && ((rm >> (ITEMS - 1)) & 1u) && (nxt & 1u))
                sw += (int)(((z >> (ITEMS - 1)) & 1u) ^ ((nxt >> 1) & 1u));
            int pkey = has ? (((base + 31 - __clz(dec)) << 1) | (int)((val >> (31 - __clz(dec))) & 1u)) : -1;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                ssz += __shfl_xor_sync(0xffffffffu, ssz, d);
                spend += __shfl_xor_sync(0xffffffffu, spend, d);
                sw += __shfl_xor_sync(0xffffffffu, sw, d);
                pkey = max(pkey, __shfl_xor_sync(0xffffffffu, pkey, d));
            }
            if (lane == 0) { s_sw_d[wid][0] = ssz; s_sw_d[wid][1] = spend; s_sw_i[wid][0] = sw; s_sw_i[wid][1] = pkey; }
        }
        if (EMIT) {
            uint8_t *gm = P.mask + cd.offset + s0 + base;
            if (cnt == ITEMS && ((reinterpret_cast<uintptr_t>(gm) & 15) == 0)) {
                uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
                for (int j = 0; j < ITEMS; ++j) w[j >> 2] |= ((z >> j) & 1u) << (8 * (j & 3));
                *reinterpret_cast<uint4 *>(gm) = make_uint4(w[0], w[1], w[2], w[3]);
            } else {
                for (int j = 0; j < cnt; ++j) gm[j] = (uint8_t)((z >> j) & 1u);
            }
        }
        __syncthreads();
        if (tid == 0) {
            TileOut o{0, 0, 0, 0};
            int nr = 0, any = 0;
            for (int w = 0; w < WARPS; ++w) {
                o.cnt += s_red[w][0]; o.pend += s_red[w][1]; o.ties += s_red[w][2]; nr += s_red[w][3];
                any |= s_whas[w];
            }
            o.head = any ? (int)(z & 1u) : 2;
            if (P.exact_mode) o.ties += nr;          // near ties count like ties: the multiplier is re-evaluated by the exact replay
            P.tout[sidx] = o;
            if (P.tsweep) {
                TileSweep ts{0.0, 0.0, 0, 0};
                int pk = -1;
                for (int w = 0; w < WARPS; ++w) { ts.ssz += s_sw_d[w][0]; ts.spend += s_sw_d[w][1]; ts.sw += s_sw_i[w][0]; pk = max(pk, s_sw_i[w][1]); }
                ts.zp = pk < 0 ? 2 : (pk & 1);
                P.tsweep[sidx] = ts;
            }
            if (EMIT && nr) atomicAdd(reinterpret_cast<unsigned long long *>(P.near_ties + c), (unsigned long long)nr);
        }
        __syncthreads();
        if (fz_track) {
            // bins since the last saturated bin BEFORE this thread's chunk: scan of (saturated seen, run length) over the threads
            const int SATBIT = 1 << 30;
            int st = fz_sat ? (SATBIT | fz_run) : cnt;
            int inc = st;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int o = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d && !(inc & SATBIT)) inc = (o & SATBIT) | ((o & ~SATBIT) + inc);
            }
            int before = __shfl_up_sync(0xffffffffu, inc, 1);
            if (lane == 0) before = 0;
            if (lane == 31) s_fzlen[wid] = inc;
            if (tid == 0) s_fzlast = 0;
            __syncthreads();
            // the tile's first bin follows a saturated bin (checked below) or is bin 0 of the chromosome: run length 0 there
            int wpre = 0;
            for (int w = 0; w < wid; ++w) { const int t = s_fzlen[w]; wpre = (t & SATBIT) ? t : ((wpre & SATBIT) | ((wpre & ~SATBIT) + t)); }
            if (!(before & SATBIT)) before = (wpre & SATBIT) | ((wpre & ~SATBIT) + before);
            const int in_len = before & ~SATBIT;
            const double eps = 1.0e-9 * (1.0 + fabs(cd.gamma));
            int ok = (cnt == 0) || ((fz_a - (double)in_len * fz_width > eps) && (fz_b > eps));
            if (fz_lastok && cnt > 0 && base + cnt == len) s_fzlast = 1;
            ok = __syncthreads_and(ok);
            if (tid == 0) {
                const V din_ = s_din;
                const bool in_sat = first_tile || fabs(din_.v) > (VEC_COST ? s_cs[0] : cd.gamma) + eps;   // the clamp of the first step saturates
                const bool own = ok && s_fzlast && in_sat && P.tout[sidx].ties == 0;
                P.fz_write[tile] = own ? 1 : 0;
                if (own) {
                    P.fz_out[tile] = P.tout[sidx];
                    P.fz_incl[tile] = 0.0;               // set by the owner of the last bin below
                }
            }
            __syncthreads();
            if (cnt > 0 && base + cnt == len) P.fz_incl[tile] = x.v > 0.0 ? 1.0e300 : -1.0e300;
        }
    }
    (void)last_tile;
}


// ------------------------------------------------------------------ short chromosomes: exact sequential emulation
// For n <= TILE the reference's recurrence is replayed operation for operation (_chain_dp.c:109-186):
// same association order, same (value, fewer-count) comparisons, so value/count/mask are the
// reference's bits.  This matters because on short inputs the 60-step bisection converges to
// neighbouring doubles around a breakpoint, where the reference's decisions are rounding-determined.
// One thread per (chromosome, multiplier); the threads of a block read the same scores (broadcast).
template <bool VEC_COST, bool EMIT>
__global__ void __launch_bounds__(256) k_chain_seq(Params P)
{
    const int c = blockIdx.x;
    const ChromDev cd = P.chroms[c];
    if (!cd.seq) return;
    const SearchDev sd = P.search[c];
    if ((sd.phase == PH_DONE && !EMIT) || sd.phase == PH_HOST) return;
    const int slot = threadIdx.x;
    if (slot >= sd.nslots) return;
    const double lam = P.lam[(size_t)c * MAX_SLOTS + slot];
    const double *s = P.scores + cd.offset;
    const double *cs = VEC_COST ? P.costs + cd.offset : nullptr;
    uint8_t *bt = EMIT ? P.bt + (size_t)cd.tile0 * TILE : nullptr;
    const int n = (int)cd.n;
    double v0 = 0.0, v1 = s[0] - lam;
    long long k0 = 0, k1 = 1;
    for (int i = 1; i < n; ++i) {
        const double cc = VEC_COST ? cs[i - 1] : cd.gamma;
        const double si = s[i];
        const double off_leave = v1 - cc;
        const double on_keep = v1 + si - lam;
        const double on_enter = v0 - cc + si - lam;
        const bool leave = (off_leave > v0) || (off_leave == v0 && k1 < k0);
        const bool enter = (on_enter > on_keep) || (on_enter == on_keep && (k0 + 1) < (k1 + 1));
        const double nv0 = leave ? off_leave : v0;
        const long long nk0 = leave ? k1 : k0;
        const double nv1 = enter ? on_enter : on_keep;
        const long long nk1 = (enter ? k0 : k1) + 1;
        if (EMIT) bt[i] = (uint8_t)((leave ? 1 : 0) | (enter ? 0 : 2));   // bit0: pred of state 0, bit1: pred of state 1
        v0 = nv0; k0 = nk0; v1 = nv1; k1 = nk1;
    }
    const bool end_on = (v1 > v0) || (v1 == v0 && k1 < k0);
    const long long cnt = end_on ? k1 : k0;
    P.counts[(size_t)c * MAX_SLOTS + slot] = cnt;
    P.tiecnt[(size_t)c * MAX_SLOTS + slot] = 0;
    if (EMIT && slot == 0) {
        uint8_t *m = P.mask + cd.offset;
        int st = end_on ? 1 : 0;
        m[n - 1] = (uint8_t)st;
        for (int i = n - 1; i > 0; --i) {
            st = st ? ((bt[i] >> 1) & 1) : (bt[i] & 1);
            m[i - 1] = (uint8_t)st;
        }
        P.seq_value[c] = end_on ? v1 : v0;
        P.tout[cd.tile0] = TileOut{(int)cnt, 0, (int)m[0], 0};
        P.zin[cd.tile0] = 0;
    }
}

// ------------------------------------------------------------------ exact replay for long chromosomes (opt-in)
// The reference's decisions compare ABSOLUTE values V0, V1 (|V| up to ~1e5-1e6, ulp ~1e-11..1e-10) and its rounding
// errors accumulate along the whole chromosome; the scan works on d = V1 - V0 with errors of ~1e-15.  Both agree on every
// decision whose margin exceeds that noise, i.e. everywhere except at multipliers within ~1e-9 of a breakpoint of
// count(lambda) -- exactly where the last bisection levels land.  The noise is a function of the full prefix of the
// recurrence, so it cannot be reproduced tile-locally: in exact mode a multiplier that shows any decision within
// 1e-7 (1 + c) of its threshold is re-evaluated by replaying the reference's recurrence (_chain_dp.c:109-186) operation
// for operation, one thread per (chromosome, multiplier), over the whole chromosome (~13 ns per bin).  The searched
// multiplier and the mask are then the reference's bits for any length; the price is why this is not the default.
template <bool VEC_COST, bool EMIT>
__global__ void __launch_bounds__(MAX_SLOTS) k_chain_replay(Params P)
{
    const int c = blockIdx.x;
    const ChromDev cd = P.chroms[c];
    const SearchDev sd = P.search[c];
    if (cd.seq || !sd.need_lex) return;
    const int slot = threadIdx.x;
    if (slot >= sd.nslots) return;
    const double lam = P.lam[(size_t)c * MAX_SLOTS + slot];
    const double *s = P.scores + cd.offset;
    const double *cs = VEC_COST ? P.costs + cd.offset : nullptr;
    const bool emit = EMIT && slot == 0;
    uint8_t *bt = EMIT ? P.bt + (size_t)cd.tile0 * TILE : nullptr;
    const long long n = cd.n;
    double v0 = 0.0, v1 = s[0] - lam;
    long long k0 = 0, k1 = 1;
    constexpr int CH = 8;
    for (long long i0 = 1; i0 < n; i0 += CH) {
        double sv[CH], cv[CH];
#pragma unroll
        for (int k = 0; k < CH; ++k) {                      // the loads of a chunk are issued before its dependent chain
            const long long i = i0 + k;
            sv[k] = i < n ? s[i] : 0.0;
            cv[k] = (VEC_COST && i < n) ? cs[i - 1] : cd.gamma;
        }
#pragma unroll
        for (int k = 0; k < CH; ++k) {
            const long long i = i0 + k;
            if (i >= n) break;
            const double cc = cv[k], si = sv[k];
            const double off_leave = v1 - cc;
            const double on_keep = v1 + si - lam;
            const double on_enter = v0 - cc + si - lam;
            const bool leave = (off_leave > v0) || (off_leave == v0 && k1 < k0);
            const bool enter = (on_enter > on_keep) || (on_enter == on_keep && (k0 + 1) < (k1 + 1));
            const double nv0 = leave ? off_leave : v0;
            const long long nk0 = leave ? k1 : k0;
            const double nv1 = enter ? on_enter : on_keep;
            const long long nk1 = (enter ? k0 : k1) + 1;
            if (emit) bt[i] = (uint8_t)((leave ? 1 : 0) | (enter ? 0 : 2));
            v0 = nv0; k0 = nk0; v1 = nv1; k1 = nk1;
        }
    }
    const bool end_on = (v1 > v0) || (v1 == v0 && k1 < k0);
    P.counts[(size_t)c * MAX_SLOTS + slot] = end_on ? k1 : k0;
    P.tiecnt[(size_t)c * MAX_SLOTS + slot] = 0;
    if (emit) {
        uint8_t *m = P.mask + cd.offset;
        int st = end_on ? 1 : 0;
        m[n - 1] = (uint8_t)st;
        for (long long i = n - 1; i > 0; --i) {
            st = st ? ((bt[i] >> 1) & 1) : (bt[i] & 1);
            m[i - 1] = (uint8_t)st;
        }
        // the mask is final: nothing left pending for k_chain_finalize, which still needs each tile's right neighbour
        for (int t = 0; t < cd.ntiles; ++t) {
            TileOut o = P.tout[cd.tile0 + t];
            o.pend = 0;
            P.tout[cd.tile0 + t] = o;
            const long long nxt = (long long)(t + 1) * TILE;
            P.zin[cd.tile0 + t] = nxt < n ? (int)m[nxt] : 0;
        }
    }
}

// ------------------------------------------------------------------ per-chromosome finish + search controller
// One block per chromosome, one warp per multiplier slot (looping when there are more slots than warps).
// Multipliers whose count needs no DP pass (costs are >= 0):
//   lambda > max(s): every s_i - lambda < 0, so d_i <= 0 throughout and nothing is selected (count = 0);
//   min(s) - lambda > 2 c_max + 1/2: d_0 > c and d_i >= -c + (s_i - lambda) > c, every bin is decided "selected" (count = n).
// The reference's bracket (dp.py:110-111) is min(s) - sum(c) - 1 .. max(s) + sum(c) + 1, about 2 sum(c) wide, while
// counts only vary on [min(s) - 2c, max(s)]: the first ~log2(sum(c) / range(s)) bisection levels land in these two
// regions and are resolved here, with the margins (1/2, strict) far above any rounding of either implementation.
// +1: count = n, -1: count = 0, 0: evaluate.  `cb` bounds every switch cost of the chain (c_max above).
__device__ __forceinline__ int known_side(double smin, double smax, double cb, double lam)
{
    if (!(smin == smin)) return 0;
    if (lam > smax) return -1;
    if (smin - lam > 2.0 * cb + 0.5) return +1;
    return 0;
}
// a chromosome's bound: gamma, or (vector costs) their sum
__device__ __forceinline__ double known_cost_bound(const ChromDev &cd, int vec)
{
    return cd.n >= 2 ? (vec ? cd.cost_sum : cd.gamma) : 0.0;
}

// Walk the bisection (dp.py:141-162) through every level whose midpoint has a known count.
__device__ void skip_known_levels(SearchDev &sd, double cb)
{
    while (sd.iters_left > 0) {
        const double mid = (sd.lower + sd.upper) / 2.0;
        const int k = known_side(sd.smin, sd.smax, cb, mid);
        if (k == 0) break;
        if (k > 0) sd.lower = mid; else sd.upper = mid;           // count = n > target / count = 0 <= target
        sd.iters_left -= 1;
        sd.passes += 1;
    }
}

__device__ void gen_tree(const SearchDev &sd, double *lam, int levels)
{
    // heap-ordered complete tree of the next `levels` bisection midpoints; every midpoint is formed
    // with the reference's own expression (lower + upper) / 2.0 on the bracket it would see (dp.py:143)
    double lo[1 << MAX_LEVELS], hi[1 << MAX_LEVELS];
    lo[1] = sd.lower; hi[1] = sd.upper;
    const int nodes = (1 << levels) - 1;
    for (int i = 1; i <= nodes; ++i) {
        const double mid = (lo[i] + hi[i]) / 2.0;
        lam[i - 1] = mid;
        if (2 * i + 1 <= nodes) {
            lo[2 * i] = lo[i]; hi[2 * i] = mid;
            lo[2 * i + 1] = mid; hi[2 * i + 1] = hi[i];
        }
    }
}

// Bracket lower = min(s) - sum(c) - 1, upper = max(s) + sum(c) + 1 (dp.py:110-111) and the first tree.  Both bracket ends
// usually have known counts (n > target and 0 <= target): the two bracket solves of dp.py:113-138 and the leading bisection
// levels then need no DP pass.
__device__ void search_start(SearchDev &sd, double *lam, double lo, double hi, double cost_sum, int max_iter, double cb, int levels)
{
    sd.lower = lo - cost_sum - 1.0;
    sd.upper = hi + cost_sum + 1.0;
    sd.phase = PH_BRACKET; sd.iters_left = max_iter; sd.levels = levels; sd.nslots = 2;
    lam[0] = sd.lower; lam[1] = sd.upper;
    if (known_side(sd.smin, sd.smax, cb, sd.lower) > 0 && known_side(sd.smin, sd.smax, cb, sd.upper) < 0) {
        sd.phase = PH_BISECT;
        sd.passes = 2;
        skip_known_levels(sd, cb);
        if (sd.iters_left <= 0) {
            sd.phase = PH_DONE; sd.nslots = 1; lam[0] = sd.upper;
        } else {
            const int lv = min(levels, sd.iters_left);
            sd.levels = lv; sd.nslots = (1 << lv) - 1;
            gen_tree(sd, lam, lv);
        }
    }
}

// One controller step after a search round: `cnt` holds the counts at the round's multipliers `lam`.  live >= 0: the tiles
// that did real work in the round (adaptive depth), -1: fixed depth.
__device__ void search_advance(SearchDev &sd, const long long *cnt, double *lam, long long target, double cb, int live,
                               int levels_base, int live_threshold)
{
    // reference-equivalent pass count (dp.py: 2 bracket solves + one per bisection level)
    sd.passes += (sd.phase == PH_BISECT) ? sd.levels : sd.nslots;
    sd.rounds += 1;
    if (sd.phase == PH_BRACKET) {
        // dp.py:113-138: the bracket ends must give count > target (lower) and count <= target (upper)
        if (cnt[0] <= target || cnt[1] > target) {
            sd.phase = PH_HOST;                           // expansion loop handled by the host driver
        } else {
            sd.phase = PH_BISECT;
        }
    } else if (sd.phase == PH_BISECT) {
        int i = 1;
        for (int l = 0; l < sd.levels; ++l) {             // dp.py:141-162
            const double mid = lam[i - 1];
            if (cnt[i - 1] > target) { sd.lower = mid; i = 2 * i + 1; }
            else { sd.upper = mid; i = 2 * i; }
        }
        sd.iters_left -= sd.levels;
    }
    if (sd.phase == PH_BISECT) {
        skip_known_levels(sd, cb);
        if (sd.iters_left <= 0) {
            sd.phase = PH_DONE;
            sd.nslots = 1;
            lam[0] = sd.upper;                            // dp.py:164 returns the upper end
        } else {
            int pref = sd.levels > 0 ? sd.levels : 1;
            if (live >= 0) pref = (live >= live_threshold) ? 1 : levels_base;
            const int lv = min(pref, sd.iters_left);
            sd.levels = lv;
            sd.nslots = (1 << lv) - 1;
            gen_tree(sd, lam, lv);
        }
    }
}

__global__ void __launch_bounds__(256) k_chain_finish(Params P, int emit)
{
    const int c = blockIdx.x;
    const ChromDev cd = P.chroms[c];
    SearchDev sd = P.search[c];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        *P.ticket = 0;
        if (P.live_cnt && !P.lex_pass) P.live_cnt[(P.round_id + 1) & 1] = 0;       // the next round's counter
    }
    const bool active = P.lex_pass ? (sd.need_lex != 0)
                                   : !((sd.phase == PH_DONE && !emit) || sd.phase == PH_HOST);
    // (sequential-kernel chromosomes never set need_lex: their counts are already the reference's)
    if (!active) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __shared__ int s_anytie;
    if (threadIdx.x == 0) s_anytie = 0;
    __syncthreads();

    const bool replayed = P.lex_pass && P.exact_mode;       // counts were written by k_chain_replay
    for (int slot = wid; slot < sd.nslots && !cd.seq && !replayed; slot += nw) {
        const TileOut *to = P.tout + (size_t)slot * P.ntiles + cd.tile0;
        long long total = 0;
        int ties = 0;
        int carry = 0;                                   // value flowing in from the right of the chunk
        const TileSweep *tsw = P.tsweep ? P.tsweep + (size_t)slot * P.ntiles + cd.tile0 : nullptr;
        double sw_ssz = 0.0;
        long long sw_cnt = 0;
        for (int hi = cd.ntiles; hi > 0; hi -= 32) {     // chunks of 32 tiles, right to left
            const int t = hi - 32 + lane;                // this lane's tile (may be < 0)
            int h = 2, pend = 0, cnt = 0, tt = 0;
            if (t >= 0) {
                const TileOut me = to[t];
                cnt = me.cnt; pend = me.pend; tt = me.ties;
                if (t + 1 < cd.ntiles) h = to[t + 1].head;   // head of the right neighbour
            }
            const unsigned D = __ballot_sync(0xffffffffu, h != 2);
            const unsigned Hv = __ballot_sync(0xffffffffu, h == 1);
            const unsigned at_or_above = D >> lane;
            const int zin = at_or_above ? ((Hv >> (lane + __ffs(at_or_above) - 1)) & 1) : carry;
            if (t >= 0) {
                total += cnt + (zin ? pend : 0);
                ties += tt;
                if (emit && slot == 0) P.zin[cd.tile0 + t] = zin;
                if (tsw) {
                    const TileSweep ts = tsw[t];
                    sw_ssz += ts.ssz + (zin ? ts.spend : 0.0);
                    sw_cnt += ts.sw;
                    if (t + 1 < cd.ntiles && ts.zp != 2 && ts.zp != zin) sw_cnt += 1;   // boundary after the last decided bin
                }
            }
            carry = __shfl_sync(0xffffffffu, zin, 0);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            total += __shfl_xor_sync(0xffffffffu, total, d);
            ties += __shfl_xor_sync(0xffffffffu, ties, d);
            sw_ssz += __shfl_xor_sync(0xffffffffu, sw_ssz, d);
            sw_cnt += __shfl_xor_sync(0xffffffffu, sw_cnt, d);
        }
        if (lane == 0 && tsw) { P.sweep_ssz[(size_t)c * MAX_SLOTS + slot] = sw_ssz; P.sweep_sw[(size_t)c * MAX_SLOTS + slot] = sw_cnt; }
        if (lane == 0) {
            P.counts[(size_t)c * MAX_SLOTS + slot] = total;
            P.tiecnt[(size_t)c * MAX_SLOTS + slot] = ties;
            if (ties) atomicOr(&s_anytie, 1);
        }
    }
    __syncthreads();
    if (threadIdx.x != 0) return;

    // ---- controller (thread 0)
    if (!P.lex_pass && s_anytie) {                      // exact ties: redo these multipliers with VL
        sd.need_lex = 1;
        P.search[c] = sd;
        return;
    }
    sd.need_lex = 0;
    // the final mask-emitting solve re-evaluates `upper`; in genome mode the group controller takes the step (k_genome_control)
    if (!emit && !P.group)
        search_advance(sd, P.counts + (size_t)c * MAX_SLOTS, P.lam + (size_t)c * MAX_SLOTS, cd.target,
                       known_cost_bound(cd, P.costs != nullptr), P.live_cnt ? P.live_cnt[P.round_id & 1] : -1,
                       P.levels_base, P.live_threshold);
    P.search[c] = sd;
}

// Bracket initialisation: lower = min(s) - sum(c) - 1, upper = max(s) + sum(c) + 1 (dp.py:110-111).
__global__ void __launch_bounds__(256) k_chain_minmax(const double *scores, const ChromDev *chroms, SearchDev *search,
                                                      double *partial /* [nchrom][gridDim.y][2] */)
{
    const int c = blockIdx.x;
    const ChromDev cd = chroms[c];
    const double *s = scores + cd.offset;
    double lo = INFINITY, hi = -INFINITY;
    int bad = 0;
    for (long long i = (long long)blockIdx.y * blockDim.x + threadIdx.x; i < cd.n; i += (long long)gridDim.y * blockDim.x) {
        const double v = s[i];
        lo = fmin(lo, v); hi = fmax(hi, v);
        bad |= !isfinite(v);
    }
    __shared__ double s_lo[8], s_hi[8];
    __shared__ int s_bad;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, d));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, d));
    }
    if (bad) atomicOr(&s_bad, 1);
    if ((threadIdx.x & 31) == 0) { s_lo[threadIdx.x >> 5] = lo; s_hi[threadIdx.x >> 5] = hi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { lo = fmin(lo, s_lo[w]); hi = fmax(hi, s_hi[w]); }
        double *p = partial + ((size_t)c * gridDim.y + blockIdx.y) * 2;
        p[0] = s_bad ? NAN : lo;
        p[1] = hi;
    }
}

__global__ void k_chain_init(const ChromDev *chroms, SearchDev *search, double *lam, const double *partial,
                             int nparts, int levels, int nchrom, int vec)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchrom) return;
    const ChromDev cd = chroms[c];
    SearchDev sd;
    double lo = INFINITY, hi = -INFINITY;
    bool bad = false;
    for (int k = 0; k < nparts; ++k) {
        const double a = partial[((size_t)c * nparts + k) * 2], b = partial[((size_t)c * nparts + k) * 2 + 1];
        if (isnan(a)) bad = true;
        lo = fmin(lo, a); hi = fmax(hi, b);
    }
    sd.smin = bad ? NAN : lo; sd.smax = hi;
    sd.need_lex = 0; sd.passes = 0; sd.rounds = 0; sd.pad = 0;
    double *l = lam + (size_t)c * MAX_SLOTS;
    if (cd.mode == 0) {
        sd.phase = PH_DONE; sd.lower = sd.upper = l[0];     // host stored the fixed multiplier in slot 0
        sd.iters_left = 0; sd.levels = 0; sd.nslots = 1;
    } else {
        search_start(sd, l, lo, hi, cd.cost_sum, cd.max_iter, known_cost_bound(cd, vec), levels);
    }
    search[c] = sd;
}

// After the bracket round, PH_BRACKET -> PH_BISECT transitions generate the first tree inside k_chain_finish.

// ------------------------------------------------------------------ genome-wide budget: one controller for a group
// The chromosomes of a call (and of every rank taking part) form one chain S = s_1 || s_2 || ..., with zero switch cost at
// the junctions, so at any multiplier the chain's mask is the members' masks laid end to end and count(lambda) is the sum
// of the members' counts.  The members are solved by the kernels above exactly as in a per-chromosome search; only the
// controller step changes: k_chain_finish leaves it out (P.group), k_genome_sum adds the members' counts of every slot,
// the caller's reducer sums those over ranks, and k_genome_control runs search_advance once on the group's state with the
// genome target and copies the result into every member's SearchDev and multiplier row.
struct GroupDev {
    SearchDev sd;
    long long target;       // floor(N * budget) of the whole genome
    double cost_sum;        // correctly rounded sum of every switch cost of the genome
    double cost_max;        // largest switch cost: the bound of known_side
    int max_iter;
    int status;             // 0, or the status a reduce reported (then sd.phase = PH_DONE)
};

// Status slot of a reduce: class k of ST_NOMEM, ST_INVALID, ST_CUDA, ST_NONFINITE (-(k+1)) adds 4096^k, so the summed slot
// counts the failed ranks of each class (up to 4095 ranks) exactly in a double; every rank decodes the same status.
constexpr int STATUS_FIELD_BITS = 12;
__device__ __forceinline__ double status_field(int st)
{
    if (st == 0) return 0.0;
    const int k = (st >= -4 && st < 0) ? -st - 1 : -ST_CUDA - 1;
    return (double)(1LL << (STATUS_FIELD_BITS * k));
}
__host__ __device__ __forceinline__ int status_decode(double v)
{
    const long long x = (long long)v;
    for (int k = 0; k < 4; ++k)
        if ((x >> (STATUS_FIELD_BITS * k)) & ((1LL << STATUS_FIELD_BITS) - 1)) return -(k + 1);
    return 0;
}

// every thread of the block: the group's state and multipliers into each member (their own score extremes stay)
__device__ void group_broadcast(const Params &P, const SearchDev &g, const double *g_lam)
{
    for (int c = threadIdx.x; c < P.nchrom; c += blockDim.x) {
        SearchDev sd = g;
        sd.smin = P.search[c].smin; sd.smax = P.search[c].smax;
        sd.need_lex = 0;
        P.search[c] = sd;
    }
    const int ns = g.nslots;
    for (int i = threadIdx.x; i < P.nchrom * ns; i += blockDim.x)
        P.lam[(size_t)(i / ns) * MAX_SLOTS + i % ns] = g_lam[i % ns];
}

// The group's first state (one block).  member_extremes: min(S) / max(S) from the members' own (single-process calls).
__global__ void __launch_bounds__(256) k_genome_init(Params P, GroupDev *G, double *g_lam, int levels, int member_extremes)
{
    __shared__ SearchDev s_g;
    if (threadIdx.x == 0) {
        GroupDev g = *G;
        if (member_extremes) {
            double lo = INFINITY, hi = -INFINITY;
            for (int c = 0; c < P.nchrom; ++c) { lo = fmin(lo, P.search[c].smin); hi = fmax(hi, P.search[c].smax); }
            g.sd.smin = lo; g.sd.smax = hi;
        }
        g.sd.need_lex = 0; g.sd.passes = 0; g.sd.rounds = 0; g.sd.pad = 0;
        search_start(g.sd, g_lam, g.sd.smin, g.sd.smax, g.cost_sum, g.max_iter, g.cost_max, levels);
        g.status = 0;
        *G = g;
        s_g = g.sd;
    }
    __syncthreads();
    group_broadcast(P, s_g, g_lam);
}

// Copy the group's state (set by the host) into the members.
__global__ void __launch_bounds__(256) k_genome_broadcast(Params P, const GroupDev *G, const double *g_lam)
{
    group_broadcast(P, G->sd, g_lam);
}

// red[0 .. nslots): every slot's count summed over the members (exact integers as doubles); red[nslots]: the tiles that did
// real work this round; red[nslots + 1]: this rank's status.
__global__ void __launch_bounds__(256) k_genome_sum(Params P, double *red, int nslots, int local_status)
{
    for (int s = threadIdx.x; s < nslots; s += blockDim.x) {
        long long t = 0;
        for (int c = 0; c < P.nchrom; ++c) t += P.counts[(size_t)c * MAX_SLOTS + s];
        red[s] = (double)t;
    }
    if (threadIdx.x == 0) {
        red[nslots] = P.live_cnt ? (double)P.live_cnt[P.round_id & 1] : 0.0;
        red[nslots + 1] = status_field(local_status);
    }
}

// The total selected count of the members' final masks and this rank's status, in the layout of k_genome_sum.
__global__ void k_genome_total(const rocco_b200_chain_result *res, int nchrom, double *red, int nslots, int local_status)
{
    if (threadIdx.x != 0) return;
    long long t = 0;
    int bad = 0;
    for (int c = 0; c < nchrom; ++c) { t += res[c].selected_count; bad |= res[c].status != 0; }
    red[0] = (double)t;
    red[nslots] = 0.0;
    red[nslots + 1] = status_field(local_status ? local_status : (bad ? ST_NONFINITE : 0));
}

// The group's controller step on the reduced buffer, then the new state into every member.
__global__ void __launch_bounds__(256) k_genome_control(Params P, GroupDev *G, const double *red, int nslots, double *g_lam,
                                                        long long *g_cnt)
{
    __shared__ SearchDev s_g;
    if (threadIdx.x == 0) {
        GroupDev g = *G;
        const int st = status_decode(red[nslots + 1]);
        if (st != 0) {
            g.status = st;
            g.sd.phase = PH_DONE; g.sd.nslots = 1;
        } else if (g.sd.phase == PH_BRACKET || g.sd.phase == PH_BISECT) {
            for (int s = 0; s < g.sd.nslots; ++s) g_cnt[s] = (long long)red[s];
            search_advance(g.sd, g_cnt, g_lam, g.target, g.cost_max, P.live_cnt ? (int)red[nslots] : -1, P.levels_base,
                           P.live_threshold);
        }
        *G = g;
        s_g = g.sd;
    }
    __syncthreads();
    group_broadcast(P, s_g, g_lam);
}

// ------------------------------------------------------------------ finalize: patch undecided suffixes, objective sums
struct FinalPart { double sum_sz; double sum_cost; long long count; long long switches; };

template <bool VEC_COST>
__global__ void __launch_bounds__(THREADS) k_chain_finalize(Params P, FinalPart *parts /* [tile] */)
{
    const int tile = blockIdx.x;
    const int c = P.tile_chrom[tile];
    const ChromDev cd = P.chroms[c];
    const long long s0 = (long long)(tile - cd.tile0) * TILE;
    const int len = (int)min((long long)TILE, cd.n - s0);
    const TileOut to = P.tout[tile];                      // slot 0
    const int zin = P.zin[tile];
    const int pend_from = len - to.pend;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint8_t *gm = P.mask + cd.offset + s0;
    const double *gs = P.scores + cd.offset + s0;
    const bool last_tile = (s0 + len == cd.n);

    __shared__ uint8_t s_z[TILE + 1];
    for (int e = tid; e < len; e += THREADS) {
        uint8_t z = gm[e];
        if (e >= pend_from) { z = (uint8_t)zin; if (zin) gm[e] = 1; }
        s_z[e] = z;
    }
    if (tid == 0) s_z[len] = last_tile ? 255 : (uint8_t)zin;      // right neighbour of the tile's last bin
    __syncthreads();
    double ssz = 0.0, scost = 0.0;
    long long cntv = 0, sw = 0;
    for (int e = tid; e < len; e += THREADS) {
        const int z = s_z[e];
        if (z) { ssz += gs[e]; ++cntv; }
        const int zr = s_z[e + 1];
        if (zr != 255 && zr != z) {
            ++sw;
            if (VEC_COST) scost += P.costs[cd.offset + s0 + e];
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        ssz += __shfl_xor_sync(0xffffffffu, ssz, d);
        scost += __shfl_xor_sync(0xffffffffu, scost, d);
        cntv += __shfl_xor_sync(0xffffffffu, cntv, d);
        sw += __shfl_xor_sync(0xffffffffu, sw, d);
    }
    __shared__ double r_a[WARPS], r_b[WARPS];
    __shared__ long long r_c[WARPS], r_d[WARPS];
    if (lane == 0) { r_a[wid] = ssz; r_b[wid] = scost; r_c[wid] = cntv; r_d[wid] = sw; }
    __syncthreads();
    if (tid == 0) {
        FinalPart fp{0.0, 0.0, 0, 0};
        for (int w = 0; w < WARPS; ++w) { fp.sum_sz += r_a[w]; fp.sum_cost += r_b[w]; fp.count += r_c[w]; fp.switches += r_d[w]; }
        parts[tile] = fp;
    }
}

__global__ void k_chain_results(Params P, const FinalPart *parts, rocco_b200_chain_result *out, int vec_cost)
{
    const int c = blockIdx.x;
    const ChromDev cd = P.chroms[c];
    const SearchDev sd = P.search[c];
    // fixed order, one warp: deterministic sums
    const int lane = threadIdx.x;
    double ssz = 0.0, scost = 0.0;
    long long cnt = 0, sw = 0;
    for (int t = lane; t < cd.ntiles; t += 32) {
        const FinalPart fp = parts[cd.tile0 + t];
        ssz += fp.sum_sz; scost += fp.sum_cost; cnt += fp.count; sw += fp.switches;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        ssz += __shfl_xor_sync(0xffffffffu, ssz, d);
        scost += __shfl_xor_sync(0xffffffffu, scost, d);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
        sw += __shfl_xor_sync(0xffffffffu, sw, d);
    }
    if (lane == 0) {
        rocco_b200_chain_result r;
        const double lam = P.lam[(size_t)c * MAX_SLOTS];
        const double tv = vec_cost ? scost : cd.gamma * (double)sw;
        r.selection_penalty = lam;
        r.penalized_objective = cd.seq ? P.seq_value[c] : ssz - lam * (double)cnt - tv;
        r.objective = -ssz + tv;
        r.selected_count = cnt;
        r.switch_count = sw;
        r.exact_tie_bins = P.tiecnt[(size_t)c * MAX_SLOTS];
        r.near_tie_bins = P.near_ties[c];
        r.dp_passes = sd.passes + (cd.mode == 0 ? 1 : 0);
        r.search_rounds = sd.rounds;
        r.status = isnan(sd.smin) ? ST_NONFINITE : 0;
        r.reserved = 0;
        out[c] = r;
    }
}

// ------------------------------------------------------------------ host driver
// chromosomes of at most this many bins (<= TILE) use the exact sequential kernel
static std::atomic<int> g_seq_max{TILE};
// 1: re-evaluate multipliers with near-tie decisions by the sequential replay (any length); see k_chain_replay
static std::atomic<int> g_exact_search{0};
// 1 (default): search rounds answer tiles whose decisions cannot change any more from stored outputs; 0: evaluate every tile
static std::atomic<int> g_freeze{1};

struct Workspace {
    ChromDev *d_chroms = nullptr;
    SearchDev *d_search = nullptr;
    int *d_tile_chrom = nullptr;
    double *d_lam = nullptr;
    long long *d_counts = nullptr, *d_tiecnt = nullptr, *d_near = nullptr;
    int *d_flags = nullptr;
    void *d_agg = nullptr, *d_incl = nullptr;
    TileOut *d_tout = nullptr;
    int *d_ticket = nullptr, *d_zin = nullptr;
    double *d_partial = nullptr;
    FinalPart *d_parts = nullptr;
    rocco_b200_chain_result *d_results = nullptr;
};

static size_t smem_bytes(bool vec) { return (size_t)(TILE + THREADS) * sizeof(double) * (vec ? 2 : 1) + (vec ? 64 : 0); }

template <typename V, bool VEC, bool EMIT>
static int launch_tiles(const Params &P, int blocks, cudaStream_t st)
{
    static bool attr_set_dev[64] = {false};
    int attr_set_d = 0;
    cudaGetDevice(&attr_set_d);
    bool &attr_set = attr_set_dev[attr_set_d & 63];
    const size_t sm = smem_bytes(VEC);
    if (!attr_set) {
        RB_CUDA(cudaFuncSetAttribute(k_chain_tiles<V, VEC, EMIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        attr_set = true;
    }
    k_chain_tiles<V, VEC, EMIT><<<blocks, THREADS, sm, st>>>(P);
    RB_LAUNCH_CHECK();
    return 0;
}

template <bool EMIT>
static int launch_round(Params P, bool vec, int nslots_max, int &epoch, bool any_seq, cudaStream_t st)
{
    P.ngroups = (nslots_max + P.slots_per_block - 1) / P.slots_per_block;
    const int blocks = P.ntiles * P.ngroups;
    // algorithmic bytes of a search round: every score read once (8 B/bin) whatever the number of multipliers;
    // the emitting round also writes one mask byte per bin
    RB_PROF(EMIT ? "chain_emit_round" : "chain_search_round", st, (double)P.ntiles * TILE * (EMIT ? 9.0 : 8.0));
    for (int lex = 0; lex < 2; ++lex) {
        P.lex_pass = lex;
        P.epoch = ++epoch;
        if (lex == 0 && any_seq) {
            if (vec) k_chain_seq<true, EMIT><<<P.nchrom, 256, 0, st>>>(P);
            else k_chain_seq<false, EMIT><<<P.nchrom, 256, 0, st>>>(P);
            RB_LAUNCH_CHECK();
        }
        if (lex == 0) {
            if (vec) RB_TRY((launch_tiles<VD, true, EMIT>(P, blocks, st)));
            else RB_TRY((launch_tiles<VD, false, EMIT>(P, blocks, st)));
        } else if (P.exact_mode) {
            if (vec) k_chain_replay<true, EMIT><<<P.nchrom, MAX_SLOTS, 0, st>>>(P);
            else k_chain_replay<false, EMIT><<<P.nchrom, MAX_SLOTS, 0, st>>>(P);
            RB_LAUNCH_CHECK();
        } else {
            if (vec) RB_TRY((launch_tiles<VL, true, EMIT>(P, blocks, st)));
            else RB_TRY((launch_tiles<VL, false, EMIT>(P, blocks, st)));
        }
        k_chain_finish<<<P.nchrom, 256, 0, st>>>(P, EMIT ? 1 : 0);
        RB_LAUNCH_CHECK();
    }
    return 0;
}

// Genome mode of solve_batch: one multiplier searched for the chromosomes of every rank that calls with the same `search`.
struct Genome {
    const rocco_b200_genome_search *search;
    rocco_b200_allreduce_fn reduce;         // nullptr: this call holds the whole genome
    void *user;
    rocco_b200_genome_result *out;
};

static int solve_batch(const double *d_scores, const double *d_costs, const rocco_b200_chain_task *tasks, int ntask,
                       uint8_t *d_masks, rocco_b200_chain_result *results, int levels, cudaStream_t st,
                       const Genome *G = nullptr)
{
    if (ntask <= 0 && !G) return 0;
    if (ntask < 0 || (ntask > 0 && (!d_scores || !tasks || !d_masks || !results))) return ST_INVALID;
    // genome mode: the arguments every rank agrees on, checked before anything is queued
    long long g_target = 0;
    bool g_whole = false, g_own_extremes = false;
    if (G) {
        const rocco_b200_genome_search &gs = *G->search;
        if (g_exact_search.load()) {
            set_error("genome budget: exact search replays one chromosome's recurrence and has no meaning for a genome; "
                      "turn it off (rocco_b200_chain_set_exact_search(0))");
            return ST_INVALID;
        }
        if (gs.total_bins <= 0 || !std::isfinite(gs.cost_sum) || gs.cost_sum < 0.0 || !std::isfinite(gs.cost_max) ||
            gs.cost_max < 0.0 || gs.max_iter < 0 || !G->out)
            return ST_INVALID;
        g_own_extremes = std::isnan(gs.score_min) || std::isnan(gs.score_max);
        if (g_own_extremes ? G->reduce != nullptr
                           : !(std::isfinite(gs.score_min) && std::isfinite(gs.score_max) && gs.score_min <= gs.score_max))
            return ST_INVALID;
        long long local_bins = 0;
        for (int c = 0; c < ntask; ++c) local_bins += (long long)std::min<size_t>(tasks[c].n, (size_t)1 << 41);
        if (G->reduce ? local_bins > gs.total_bins : local_bins != gs.total_bins) return ST_INVALID;
        g_target = std::max<long long>(0, std::min<long long>(gs.target_count, gs.total_bins));
        g_whole = g_target == gs.total_bins;      // dp.py:102-108: every chromosome at lambda = 0
    }
    // levels <= 0 (default): two levels per round, dropping to ONE while more than LIVE_THRESHOLD tiles still do real work
    // (throughput-bound rounds: a 2-level tree evaluates 3 multipliers to advance 2 levels).  An explicit value is used as is.
    const bool adaptive = levels <= 0;
    if (levels <= 0) levels = 2;      // measured on B200: 1 GPU, hg38 x 100: L=2 49 ms, L=3 57 ms, L=4 84 ms per genome search
    levels = std::min(levels, MAX_LEVELS);
    constexpr int LIVE_THRESHOLD = 3072;   // tiles: ~28 ns per tile and multiplier against a ~66 us floor per round (B200); 1950-tile shards measured better at 2 levels
    RB_TRY(ensure_device());

    std::vector<ChromDev> chroms(ntask);
    std::vector<int> tile_chrom;
    int ntiles = 0, max_iter = 0;
    bool any_search = false, any_seq = false;
    for (int c = 0; c < ntask; ++c) {
        const rocco_b200_chain_task &t = tasks[c];
        if (t.n == 0 || !(t.gamma >= 0.0) || t.n > (size_t)1 << 40) return ST_INVALID;
        ChromDev &cd = chroms[c];
        cd.offset = (long long)t.offset; cd.n = (long long)t.n; cd.gamma = t.gamma; cd.cost_sum = t.cost_sum;
        cd.mode = t.mode; cd.max_iter = t.max_iter;
        long long target = std::max<long long>(0, std::min<long long>(t.target_count, (long long)t.n));
        cd.target = target;
        if (t.mode == 1 && target == (long long)t.n) cd.mode = 2;    // dp.py:102-108: solve at lambda = 0
        if (G) { cd.mode = g_whole ? 2 : 1; cd.max_iter = G->search->max_iter; }
        cd.seq = ((long long)t.n <= (long long)g_seq_max.load()) ? 1 : 0;
        cd.pad = 0;
        any_seq |= cd.seq != 0;
        cd.tile0 = ntiles;
        cd.ntiles = (int)((t.n + TILE - 1) / TILE);
        ntiles += cd.ntiles;
        for (int k = 0; k < cd.ntiles; ++k) tile_chrom.push_back(c);
        if (cd.mode == 1) { any_search = true; max_iter = std::max(max_iter, t.max_iter); }
    }
    if (G) any_search = !g_whole;     // the group's round layout comes from agreed data, also on a rank without chromosomes
    const bool vec = d_costs != nullptr;
    const int max_slots = any_search ? std::max(2, (1 << levels) - 1) : 1;
    const int slots_per_block = std::min(max_slots, 8);

    Arena ar(st);
    // genome mode: the reduce buffer [max_slots counts][live tiles][status] and the group's state come first; a local failure
    // after them is carried to the next reduce, which every rank reaches (budget.cu's Shard::local)
    const int nred = max_slots + 2;
    double *d_red = nullptr, *d_glam = nullptr;
    long long *d_gcnt = nullptr;
    GroupDev *d_group = nullptr;
    if (G) {
        RB_TRY(ar.alloc(&d_red, (size_t)nred));
        RB_TRY(ar.alloc(&d_group, 1));
        RB_TRY(ar.alloc(&d_glam, MAX_SLOTS));
        RB_TRY(ar.alloc(&d_gcnt, MAX_SLOTS));
    }
    const bool carry = G && G->reduce;
    int failed = 0;
    auto local = [&](int s) -> int {
        if (s == 0 || !carry) return s;
        if (!failed) failed = s;
        return 0;
    };

    Workspace w;
    Params P{};
    const bool exact = g_exact_search.load() != 0;
    const bool freeze = any_search && !exact && g_freeze.load() != 0;
    int *d_fz[2] = {nullptr, nullptr};
    auto setup = [&]() -> int {
        RB_TRY(ar.alloc(&w.d_chroms, ntask));
        RB_TRY(ar.alloc(&w.d_search, ntask));
        RB_TRY(ar.alloc(&w.d_tile_chrom, ntiles));
        RB_TRY(ar.alloc(&w.d_lam, (size_t)ntask * MAX_SLOTS));
        RB_TRY(ar.alloc(&w.d_counts, (size_t)ntask * MAX_SLOTS));
        RB_TRY(ar.alloc(&w.d_tiecnt, (size_t)ntask * MAX_SLOTS));
        RB_TRY(ar.alloc(&w.d_near, ntask));
        RB_TRY(ar.alloc(&w.d_flags, (size_t)max_slots * ntiles));
        char *agg_bytes = nullptr, *incl_bytes = nullptr;
        RB_TRY(ar.alloc(&agg_bytes, (size_t)max_slots * ntiles * sizeof(Map<VL>)));
        RB_TRY(ar.alloc(&incl_bytes, (size_t)max_slots * ntiles * sizeof(VL)));
        w.d_agg = agg_bytes; w.d_incl = incl_bytes;
        RB_TRY(ar.alloc(&w.d_tout, (size_t)max_slots * ntiles));
        RB_TRY(ar.alloc(&w.d_ticket, 1));
        RB_TRY(ar.alloc(&w.d_zin, ntiles));
        const int nparts = 64;
        RB_TRY(ar.alloc(&w.d_partial, (size_t)ntask * nparts * 2));
        RB_TRY(ar.alloc(&w.d_parts, ntiles));
        RB_TRY(ar.alloc(&w.d_results, ntask));
        uint8_t *d_bt = nullptr;
        double *d_seqv = nullptr;
        RB_TRY(ar.alloc(&d_bt, (any_seq || exact) ? (size_t)ntiles * TILE : 16));
        RB_TRY(ar.alloc(&d_seqv, ntask));

        // modes: 0 fixed (lambda given), 2 fixed at 0.0; both are PH_DONE from the start
        std::vector<double> lam0((size_t)ntask * MAX_SLOTS, 0.0);
        for (int c = 0; c < ntask; ++c) {
            if (chroms[c].mode == 0) lam0[(size_t)c * MAX_SLOTS] = tasks[c].selection_penalty;
            if (chroms[c].mode == 2) { chroms[c].mode = 0; lam0[(size_t)c * MAX_SLOTS] = 0.0; }
        }
        if (ntask > 0) {
            RB_CUDA(cudaMemcpyAsync(w.d_chroms, chroms.data(), sizeof(ChromDev) * ntask, cudaMemcpyHostToDevice, st));
            RB_CUDA(cudaMemcpyAsync(w.d_tile_chrom, tile_chrom.data(), sizeof(int) * ntiles, cudaMemcpyHostToDevice, st));
            RB_CUDA(cudaMemcpyAsync(w.d_lam, lam0.data(), sizeof(double) * lam0.size(), cudaMemcpyHostToDevice, st));
            RB_CUDA(cudaMemsetAsync(w.d_flags, 0, sizeof(int) * (size_t)max_slots * ntiles, st));
            RB_CUDA(cudaMemsetAsync(w.d_ticket, 0, sizeof(int), st));
            RB_CUDA(cudaMemsetAsync(w.d_near, 0, sizeof(long long) * ntask, st));
            RB_CUDA(cudaMemsetAsync(w.d_tiecnt, 0, sizeof(long long) * (size_t)ntask * MAX_SLOTS, st));
            // the group sums every slot of every member: no slot may hold garbage
            if (G) RB_CUDA(cudaMemsetAsync(w.d_counts, 0, sizeof(long long) * (size_t)ntask * MAX_SLOTS, st));

            k_chain_minmax<<<dim3(ntask, nparts), 256, 0, st>>>(d_scores, w.d_chroms, w.d_search, w.d_partial);
            RB_LAUNCH_CHECK();
            const int init_levels = (adaptive && ntiles >= LIVE_THRESHOLD) ? 1 : levels;
            k_chain_init<<<(ntask + 63) / 64, 64, 0, st>>>(w.d_chroms, w.d_search, w.d_lam, w.d_partial, nparts, init_levels, ntask, vec ? 1 : 0);
            RB_LAUNCH_CHECK();
        }

        P.scores = d_scores; P.costs = d_costs; P.chroms = w.d_chroms; P.search = w.d_search;
        P.tile_chrom = w.d_tile_chrom; P.lam = w.d_lam; P.counts = w.d_counts; P.tiecnt = w.d_tiecnt;
        P.flags = w.d_flags; P.agg = w.d_agg; P.incl = w.d_incl; P.tout = w.d_tout; P.ticket = w.d_ticket;
        P.mask = d_masks; P.zin = w.d_zin; P.near_ties = w.d_near; P.ntiles = ntiles; P.nchrom = ntask;
        P.slots_per_block = slots_per_block;
        P.bt = d_bt; P.seq_value = d_seqv;
        P.exact_mode = exact ? 1 : 0;
        P.group = G ? 1 : 0;
        // tile freezing: two state buffers (read = previous round, write = this round), the frozen outputs and hand-on values
        if (freeze) {
            RB_TRY(ar.alloc(&d_fz[0], (size_t)ntiles));
            RB_TRY(ar.alloc(&d_fz[1], (size_t)ntiles));
            RB_TRY(ar.alloc(&P.fz_out, (size_t)ntiles));
            RB_TRY(ar.alloc(&P.fz_incl, (size_t)ntiles));
            RB_CUDA(cudaMemsetAsync(d_fz[0], 0, sizeof(int) * (size_t)ntiles, st));
            RB_CUDA(cudaMemsetAsync(d_fz[1], 0, sizeof(int) * (size_t)ntiles, st));
        }
        if (adaptive && any_search) {
            RB_TRY(ar.alloc(&P.live_cnt, (size_t)2));
            RB_CUDA(cudaMemsetAsync(P.live_cnt, 0, sizeof(int) * 2, st));
            P.levels_base = levels;
            P.live_threshold = LIVE_THRESHOLD;
        }
        return 0;
    };
    RB_TRY(local(setup()));
    int epoch = 0;
    int fz_round = 0, round_id = 0;
    auto search_round = [&](int nslots) -> int {
        P.round_id = round_id++;
        if (freeze) { P.fz_read = d_fz[fz_round & 1]; P.fz_write = d_fz[(fz_round & 1) ^ 1]; ++fz_round; }
        return launch_round<false>(P, vec, nslots, epoch, any_seq, st);
    };
    // the final solve at the chosen multipliers, mask emitted
    auto final_solve = [&]() -> int {
        P.fz_read = nullptr; P.fz_write = nullptr;
        RB_TRY((launch_round<true>(P, vec, 1, epoch, any_seq, st)));
        {
            RB_PROF("k_chain_finalize", st, (double)ntiles * TILE * 9.0);
            if (vec) k_chain_finalize<true><<<ntiles, THREADS, 0, st>>>(P, w.d_parts);
            else k_chain_finalize<false><<<ntiles, THREADS, 0, st>>>(P, w.d_parts);
            RB_LAUNCH_CHECK();
        }
        k_chain_results<<<ntask, 32, 0, st>>>(P, w.d_parts, w.d_results, vec ? 1 : 0);
        RB_LAUNCH_CHECK();
        return 0;
    };
    if (G) {
        // ---- genome mode: the members' rounds as above, the controller step on the group after one reduce per round
        const rocco_b200_genome_search &gs = *G->search;
        auto reduce = [&]() -> int {
            if (!G->reduce) return 0;
            if (G->reduce(d_red, (size_t)nred, (void *)st, G->user) != 0) {
                set_error("genome budget: the all-reduce callback failed");
                return ST_CUDA;
            }
            return 0;
        };
        auto another = [&](int s) -> int {                // every rank returns the status a reduce reported
            if (!failed) set_error("genome budget: another rank failed with status %d", s);
            return s;
        };
        auto group_params = [&]() { Params q = P; if (failed) q.nchrom = 0; return q; };   // a failed rank's members are left alone
        GroupDev hg{};
        auto read_group = [&]() -> int {
            RB_CUDA(cudaMemcpyAsync(&hg, d_group, sizeof(GroupDev), cudaMemcpyDeviceToHost, st));
            RB_CUDA(cudaStreamSynchronize(st));
            return 0;
        };
        if (!g_whole) {
            GroupDev g0{};
            g0.sd.smin = gs.score_min; g0.sd.smax = gs.score_max;
            g0.target = g_target; g0.cost_sum = gs.cost_sum; g0.cost_max = gs.cost_max; g0.max_iter = gs.max_iter;
            // agreed data only: every rank starts from the same state
            const int init_levels = (adaptive && (gs.total_bins + TILE - 1) / TILE >= LIVE_THRESHOLD) ? 1 : levels;
            RB_CUDA(cudaMemcpyAsync(d_group, &g0, sizeof(GroupDev), cudaMemcpyHostToDevice, st));
            k_genome_init<<<1, 256, 0, st>>>(group_params(), d_group, d_glam, init_levels, g_own_extremes ? 1 : 0);
            RB_LAUNCH_CHECK();
            RB_TRY(read_group());
            // rounds in batches, as the per-chromosome search; the batch size depends on the group's state only, so every
            // rank calls the reducer the same number of times
            while (hg.sd.phase == PH_BRACKET || hg.sd.phase == PH_BISECT) {
                const int bound = hg.sd.iters_left + (hg.sd.phase == PH_BRACKET ? 1 : 0);
                const int batch = std::max(1, std::min(bound, 12));
                for (int r = 0; r < batch; ++r) {
                    if (!failed && ntask > 0) RB_TRY(local(search_round(max_slots)));
                    k_genome_sum<<<1, 256, 0, st>>>(group_params(), d_red, max_slots, failed);
                    RB_LAUNCH_CHECK();
                    RB_TRY(reduce());
                    k_genome_control<<<1, 256, 0, st>>>(group_params(), d_group, d_red, max_slots, d_glam, d_gcnt);
                    RB_LAUNCH_CHECK();
                }
                RB_TRY(read_group());
            }
            if (hg.status) return another(hg.status);
            // rare: bracket expansion (dp.py:119-125, 132-138) from the host, each evaluation reduced
            if (hg.sd.phase == PH_HOST) {
                auto eval = [&](double lamv, long long &count) -> int {
                    GroupDev h = hg;
                    h.sd.phase = PH_MANUAL; h.sd.nslots = 1;
                    RB_CUDA(cudaMemcpyAsync(d_group, &h, sizeof(GroupDev), cudaMemcpyHostToDevice, st));
                    RB_CUDA(cudaMemcpyAsync(d_glam, &lamv, sizeof(double), cudaMemcpyHostToDevice, st));
                    k_genome_broadcast<<<1, 256, 0, st>>>(group_params(), d_group, d_glam);
                    RB_LAUNCH_CHECK();
                    if (!failed && ntask > 0) RB_TRY(local(launch_round<false>(P, vec, 1, epoch, any_seq, st)));
                    k_genome_sum<<<1, 256, 0, st>>>(group_params(), d_red, 1, failed);
                    RB_LAUNCH_CHECK();
                    RB_TRY(reduce());
                    double r[3];
                    RB_CUDA(cudaMemcpyAsync(r, d_red, sizeof(r), cudaMemcpyDeviceToHost, st));
                    RB_CUDA(cudaStreamSynchronize(st));
                    const int s = status_decode(r[2]);
                    if (s) return another(s);
                    count = (long long)r[0];
                    return 0;
                };
                double lower = hg.sd.lower, upper = hg.sd.upper;
                long long cl = 0, cu = 0;
                int passes = 0;
                RB_TRY(eval(lower, cl)); ++passes;
                while (cl <= g_target) { lower -= std::max(1.0, fabs(lower)); RB_TRY(eval(lower, cl)); ++passes; if (passes > 4096) return ST_INVALID; }
                RB_TRY(eval(upper, cu)); ++passes;
                while (cu > g_target) { upper += std::max(1.0, fabs(upper)); RB_TRY(eval(upper, cu)); ++passes; if (passes > 4096) return ST_INVALID; }
                for (int it = 0; it < gs.max_iter; ++it) {
                    const double mid = (lower + upper) / 2.0;
                    long long cm = 0;
                    RB_TRY(eval(mid, cm)); ++passes;
                    if (cm > g_target) lower = mid; else upper = mid;
                }
                hg.sd.lower = lower; hg.sd.upper = upper; hg.sd.passes = passes; hg.sd.rounds = passes;
                hg.sd.phase = PH_DONE; hg.sd.nslots = 1;
                RB_CUDA(cudaMemcpyAsync(d_group, &hg, sizeof(GroupDev), cudaMemcpyHostToDevice, st));
                RB_CUDA(cudaMemcpyAsync(d_glam, &hg.sd.upper, sizeof(double), cudaMemcpyHostToDevice, st));
                k_genome_broadcast<<<1, 256, 0, st>>>(group_params(), d_group, d_glam);
                RB_LAUNCH_CHECK();
            }
        }
        // every member at the group's multiplier, then one last reduce: the genome's selected count and every rank's status
        if (!failed && ntask > 0) RB_TRY(local(final_solve()));
        k_genome_total<<<1, 32, 0, st>>>(failed ? nullptr : w.d_results, failed ? 0 : ntask, d_red, max_slots, failed);
        RB_LAUNCH_CHECK();
        RB_TRY(reduce());
        double r[2];
        RB_CUDA(cudaMemcpyAsync(&r[0], d_red, sizeof(double), cudaMemcpyDeviceToHost, st));
        RB_CUDA(cudaMemcpyAsync(&r[1], d_red + max_slots + 1, sizeof(double), cudaMemcpyDeviceToHost, st));
        if (!failed && ntask > 0)
            RB_CUDA(cudaMemcpyAsync(results, w.d_results, sizeof(rocco_b200_chain_result) * ntask, cudaMemcpyDeviceToHost, st));
        RB_CUDA(cudaStreamSynchronize(st));
        const int s = status_decode(r[1]);
        if (s) return another(s);
        rocco_b200_genome_result &o = *G->out;
        o.selection_penalty = g_whole ? 0.0 : hg.sd.upper;
        o.selected_count = (long long)r[0];
        o.dp_passes = g_whole ? 1 : hg.sd.passes;
        o.search_rounds = g_whole ? 0 : hg.sd.rounds;
        o.status = 0;
        o.reserved = 0;
        return 0;
    }


    std::vector<SearchDev> hsearch(ntask);
    if (any_search) {
        // the controller has already walked through the levels that need no DP pass: fetch its state (a few hundred
        // bytes, behind two tiny kernels) so that only the rounds that still have work are launched
        RB_CUDA(cudaMemcpyAsync(hsearch.data(), w.d_search, sizeof(SearchDev) * ntask, cudaMemcpyDeviceToHost, st));
        RB_CUDA(cudaStreamSynchronize(st));
        bool need_bracket = false;
        int rounds = 0;
        for (int c = 0; c < ntask; ++c) {
            if (chroms[c].mode != 1) continue;
            if (hsearch[c].phase == PH_BRACKET) { need_bracket = true; rounds = std::max(rounds, (chroms[c].max_iter + levels - 1) / levels); }
            else if (hsearch[c].phase == PH_BISECT) rounds = std::max(rounds, (hsearch[c].iters_left + levels - 1) / levels);
        }
        if (need_bracket) RB_TRY(search_round(2));     // bracket ends
        // PH_BRACKET -> PH_BISECT generates the first tree in the same finish kernel
        if (!P.live_cnt) {
            for (int r = 0; r < rounds; ++r) RB_TRY(search_round(max_slots));
            RB_CUDA(cudaMemcpyAsync(hsearch.data(), w.d_search, sizeof(SearchDev) * ntask, cudaMemcpyDeviceToHost, st));
            RB_CUDA(cudaStreamSynchronize(st));
        } else {
            // the depth of each round is chosen on the device, so the number of rounds is not known here: launch them in
            // batches and look at the controllers' state (a few hundred bytes) after each; a round launched for chromosomes
            // that are already done costs ~20 us
            int upper = 0;                             // rounds still needed if every one of them took a single level
            for (int c = 0; c < ntask; ++c)
                if (chroms[c].mode == 1 && (hsearch[c].phase == PH_BRACKET || hsearch[c].phase == PH_BISECT))
                    upper = std::max(upper, hsearch[c].phase == PH_BRACKET ? chroms[c].max_iter : hsearch[c].iters_left);
            for (;;) {
                const int batch = std::min(upper, 12);
                for (int r = 0; r < batch; ++r) RB_TRY(search_round(max_slots));
                RB_CUDA(cudaMemcpyAsync(hsearch.data(), w.d_search, sizeof(SearchDev) * ntask, cudaMemcpyDeviceToHost, st));
                RB_CUDA(cudaStreamSynchronize(st));
                upper = 0;
                for (int c = 0; c < ntask; ++c)
                    if (chroms[c].mode == 1 && hsearch[c].phase == PH_BISECT) upper = std::max(upper, hsearch[c].iters_left);
                if (upper <= 0) break;
            }
        }
        // rare: bracket expansion (dp.py:119-125, 132-138) is driven from the host with single solves
        bool any_host = false;
        for (int c = 0; c < ntask; ++c) any_host |= (hsearch[c].phase == PH_HOST);
        if (any_host) {
            std::vector<double> hl((size_t)ntask * MAX_SLOTS);
            std::vector<long long> hc((size_t)ntask * MAX_SLOTS);
            auto eval = [&](int c, double lamv, long long &count) -> int {
                // PH_MANUAL for chromosome c only; everything else parked as PH_HOST (skipped)
                for (int k = 0; k < ntask; ++k) {
                    hsearch[k].phase = (k == c) ? PH_MANUAL : PH_HOST;
                    hsearch[k].nslots = 1; hsearch[k].need_lex = 0;
                }
                RB_CUDA(cudaMemcpyAsync(w.d_search, hsearch.data(), sizeof(SearchDev) * ntask, cudaMemcpyHostToDevice, st));
                RB_CUDA(cudaMemcpyAsync(w.d_lam + (size_t)c * MAX_SLOTS, &lamv, sizeof(double), cudaMemcpyHostToDevice, st));
                RB_TRY((launch_round<false>(P, vec, 1, epoch, any_seq, st)));
                RB_CUDA(cudaMemcpyAsync(&count, w.d_counts + (size_t)c * MAX_SLOTS, sizeof(long long), cudaMemcpyDeviceToHost, st));
                RB_CUDA(cudaStreamSynchronize(st));
                return 0;
            };
            std::vector<SearchDev> fin = hsearch;
            std::vector<SearchDev> saved = hsearch;
            for (int c = 0; c < ntask; ++c) {
                if (saved[c].phase != PH_HOST) continue;
                const long long target = chroms[c].target;
                double lower = saved[c].lower, upper = saved[c].upper;
                long long cl = 0, cu = 0;
                int passes = 0;
                RB_TRY(eval(c, lower, cl)); ++passes;
                while (cl <= target) { lower -= std::max(1.0, fabs(lower)); RB_TRY(eval(c, lower, cl)); ++passes; if (passes > 4096) return ST_INVALID; }
                RB_TRY(eval(c, upper, cu)); ++passes;
                while (cu > target) { upper += std::max(1.0, fabs(upper)); RB_TRY(eval(c, upper, cu)); ++passes; if (passes > 4096) return ST_INVALID; }
                for (int it = 0; it < chroms[c].max_iter; ++it) {
                    const double mid = (lower + upper) / 2.0;
                    long long cm = 0;
                    RB_TRY(eval(c, mid, cm)); ++passes;
                    if (cm > target) lower = mid; else upper = mid;
                }
                fin[c] = saved[c];
                fin[c].lower = lower; fin[c].upper = upper; fin[c].passes = passes; fin[c].rounds = passes;
            }
            for (int c = 0; c < ntask; ++c) {
                if (saved[c].phase != PH_HOST) fin[c] = saved[c];
                fin[c].phase = PH_DONE; fin[c].nslots = 1; fin[c].need_lex = 0;
                hl[(size_t)c * MAX_SLOTS] = fin[c].upper;
            }
            RB_CUDA(cudaMemcpyAsync(w.d_search, fin.data(), sizeof(SearchDev) * ntask, cudaMemcpyHostToDevice, st));
            for (int c = 0; c < ntask; ++c)
                RB_CUDA(cudaMemcpyAsync(w.d_lam + (size_t)c * MAX_SLOTS, &hl[(size_t)c * MAX_SLOTS], sizeof(double),
                                        cudaMemcpyHostToDevice, st));
        }
    }

    RB_TRY(final_solve());
    RB_CUDA(cudaMemcpyAsync(results, w.d_results, sizeof(rocco_b200_chain_result) * ntask, cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    for (int c = 0; c < ntask; ++c)
        if (results[c].status == ST_NONFINITE) return ST_NONFINITE;
    return 0;
}

// Multiplier sweep: counts and objectives of one chromosome for up to MAX_SLOTS multipliers per launch set.
static int sweep(const double *d_scores, size_t n, double gamma, const double *lambdas, int K, long long *count_out,
                 double *pen_out, double *obj_out, cudaStream_t st)
{
    if (!d_scores || !lambdas || n == 0 || K <= 0 || !(gamma >= 0.0)) return ST_INVALID;
    RB_TRY(ensure_device());
    const int ntiles = (int)((n + TILE - 1) / TILE);
    Arena ar(st);
    ChromDev cd{};
    cd.offset = 0; cd.n = (long long)n; cd.gamma = gamma; cd.tile0 = 0; cd.ntiles = ntiles; cd.mode = 0; cd.seq = 0;
    ChromDev *d_cd = nullptr; SearchDev *d_sd = nullptr; int *d_tc = nullptr, *d_flags = nullptr, *d_ticket = nullptr, *d_zin = nullptr;
    double *d_lam = nullptr, *d_ssz = nullptr; long long *d_cnt = nullptr, *d_tie = nullptr, *d_near = nullptr, *d_sw = nullptr;
    char *agg = nullptr, *incl = nullptr; TileOut *d_to = nullptr; TileSweep *d_ts = nullptr;
    const int batch = std::min(K, MAX_SLOTS);
    RB_TRY(ar.alloc(&d_cd, 1)); RB_TRY(ar.alloc(&d_sd, 1)); RB_TRY(ar.alloc(&d_tc, ntiles));
    RB_TRY(ar.alloc(&d_lam, MAX_SLOTS)); RB_TRY(ar.alloc(&d_cnt, MAX_SLOTS)); RB_TRY(ar.alloc(&d_tie, MAX_SLOTS));
    RB_TRY(ar.alloc(&d_near, 1)); RB_TRY(ar.alloc(&d_ssz, MAX_SLOTS)); RB_TRY(ar.alloc(&d_sw, MAX_SLOTS));
    RB_TRY(ar.alloc(&d_flags, (size_t)batch * ntiles)); RB_TRY(ar.alloc(&agg, (size_t)batch * ntiles * sizeof(Map<VL>)));
    RB_TRY(ar.alloc(&incl, (size_t)batch * ntiles * sizeof(VL))); RB_TRY(ar.alloc(&d_to, (size_t)batch * ntiles));
    RB_TRY(ar.alloc(&d_ts, (size_t)batch * ntiles)); RB_TRY(ar.alloc(&d_ticket, 1)); RB_TRY(ar.alloc(&d_zin, ntiles));
    RB_CUDA(cudaMemcpyAsync(d_cd, &cd, sizeof(cd), cudaMemcpyHostToDevice, st));
    RB_CUDA(cudaMemsetAsync(d_tc, 0, sizeof(int) * ntiles, st));
    RB_CUDA(cudaMemsetAsync(d_flags, 0, sizeof(int) * (size_t)batch * ntiles, st));
    RB_CUDA(cudaMemsetAsync(d_ticket, 0, sizeof(int), st));
    Params P{};
    P.scores = d_scores; P.costs = nullptr; P.chroms = d_cd; P.search = d_sd; P.tile_chrom = d_tc; P.lam = d_lam;
    P.counts = d_cnt; P.tiecnt = d_tie; P.flags = d_flags; P.agg = agg; P.incl = incl; P.tout = d_to; P.ticket = d_ticket;
    P.mask = nullptr; P.zin = d_zin; P.near_ties = d_near; P.ntiles = ntiles; P.nchrom = 1; P.slots_per_block = 8;
    P.tsweep = d_ts; P.sweep_ssz = d_ssz; P.sweep_sw = d_sw;
    int epoch = 0;
    std::vector<double> ssz(MAX_SLOTS);
    std::vector<long long> cnt(MAX_SLOTS), sw(MAX_SLOTS);
    for (int k0 = 0; k0 < K; k0 += batch) {
        const int kb = std::min(batch, K - k0);
        SearchDev sd{};
        sd.phase = PH_MANUAL; sd.nslots = kb; sd.need_lex = 0;
        RB_CUDA(cudaMemcpyAsync(d_sd, &sd, sizeof(sd), cudaMemcpyHostToDevice, st));
        RB_CUDA(cudaMemcpyAsync(d_lam, lambdas + k0, sizeof(double) * kb, cudaMemcpyHostToDevice, st));
        RB_TRY((launch_round<false>(P, false, kb, epoch, false, st)));
        RB_CUDA(cudaMemcpyAsync(cnt.data(), d_cnt, sizeof(long long) * kb, cudaMemcpyDeviceToHost, st));
        RB_CUDA(cudaMemcpyAsync(ssz.data(), d_ssz, sizeof(double) * kb, cudaMemcpyDeviceToHost, st));
        RB_CUDA(cudaMemcpyAsync(sw.data(), d_sw, sizeof(long long) * kb, cudaMemcpyDeviceToHost, st));
        RB_CUDA(cudaStreamSynchronize(st));
        for (int k = 0; k < kb; ++k) {
            const double tv = gamma * (double)sw[k];
            if (count_out) count_out[k0 + k] = cnt[k];
            if (pen_out) pen_out[k0 + k] = ssz[k] - lambdas[k0 + k] * (double)cnt[k] - tv;
            if (obj_out) obj_out[k0 + k] = -ssz[k] + tv;
        }
    }
    return 0;
}

}  // namespace chain
}  // namespace rb

// ====================================================================== C-ABI
using namespace rb;

extern "C" __attribute__((visibility("default"))) int rocco_b200_chain_set_seq_max(int max_bins)
{
    const int prev = chain::g_seq_max.load();
    chain::g_seq_max.store(std::max(0, std::min(max_bins, chain::TILE)));
    return prev;
}

extern "C" __attribute__((visibility("default"))) int rocco_b200_chain_set_tile_freezing(int on)
{
    return chain::g_freeze.exchange(on ? 1 : 0);
}

extern "C" __attribute__((visibility("default"))) int rocco_b200_chain_set_exact_search(int on)
{
    return chain::g_exact_search.exchange(on ? 1 : 0);
}

extern "C" __attribute__((visibility("default"))) int rocco_b200_chain_solve_batch_dev(
    const double *d_scores, const double *d_switch_costs, const rocco_b200_chain_task *tasks, int task_count,
    uint8_t *d_masks_out, rocco_b200_chain_result *results_out, int levels_per_round, void *cuda_stream)
{
    return chain::solve_batch(d_scores, d_switch_costs, tasks, task_count, d_masks_out, results_out,
                              levels_per_round, (cudaStream_t)cuda_stream);
}

extern "C" __attribute__((visibility("default"))) int rocco_b200_chain_solve_genome_dev(
    const double *d_scores, const double *d_switch_costs, const rocco_b200_chain_task *tasks, int task_count,
    const rocco_b200_genome_search *search, rocco_b200_allreduce_fn allreduce, void *user, uint8_t *d_masks_out,
    rocco_b200_chain_result *results_out, rocco_b200_genome_result *genome_out, int levels_per_round, void *cuda_stream)
{
    if (!search || !genome_out) return ST_INVALID;
    const chain::Genome g{search, allreduce, user, genome_out};
    return chain::solve_batch(d_scores, d_switch_costs, tasks, task_count, d_masks_out, results_out, levels_per_round,
                              (cudaStream_t)cuda_stream, &g);
}

extern "C" __attribute__((visibility("default"))) int rocco_b200_chain_sweep_dev(
    const double *d_scores, size_t n, double gamma, const double *lambdas, int lambda_count, long long *selected_count_out,
    double *penalized_objective_out, double *objective_out, void *cuda_stream)
{
    return chain::sweep(d_scores, n, gamma, lambdas, lambda_count, selected_count_out, penalized_objective_out, objective_out,
                        (cudaStream_t)cuda_stream);
}

static int host_chain(const double *scores, const double *costs, size_t n, int mode, double lam, long long target,
                      int max_iter, uint8_t *mask_out, rocco_b200_chain_result *res)
{
    if (!scores || !mask_out || n == 0) return ST_INVALID;
    if (n > 1 && !costs) return ST_INVALID;
    // validate before anything is queued: negative / NaN switch costs are outside the clamp-map form of the DP
    double csum = 0.0;
    if (n > 1) {
        for (size_t i = 0; i + 1 < n; ++i)
            if (!(costs[i] >= 0.0)) return ST_INVALID;
        csum = numpy_sum_f64(costs, n - 1);                  // dp.py:110-111 uses numpy.sum; its rounding defines the bracket
    }
    RB_TRY(ensure_device());
    HostScope lease(true);
    cudaStream_t st = lease.stream();
    Arena ar(st);
    double *d_s = nullptr, *d_c = nullptr;
    uint8_t *d_m = nullptr;
    RB_TRY(ar.alloc(&d_s, n));
    RB_TRY(ar.alloc(&d_c, n));
    RB_TRY(ar.alloc(&d_m, n));
    double *stage = static_cast<double *>(lease.staging(2 * n * sizeof(double)));
    const double *src_s = scores, *src_c = costs;
    if (stage) {
        memcpy(stage, scores, n * sizeof(double)); src_s = stage;
        if (n > 1) { memcpy(stage + n, costs, (n - 1) * sizeof(double)); src_c = stage + n; }
    }
    if (stage) RB_TRY(pull_from_pinned(d_s, src_s, n * sizeof(double), st));
    else RB_CUDA(cudaMemcpyAsync(d_s, src_s, n * sizeof(double), cudaMemcpyHostToDevice, st));
    RB_CUDA(cudaMemsetAsync(d_c, 0, n * sizeof(double), st));
    if (n > 1) {
        if (stage) RB_TRY(pull_from_pinned(d_c, src_c, (n - 1) * sizeof(double), st));
        else RB_CUDA(cudaMemcpyAsync(d_c, src_c, (n - 1) * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    rocco_b200_chain_task t{};
    t.offset = 0; t.n = n; t.gamma = 0.0; t.cost_sum = csum; t.selection_penalty = lam;
    t.target_count = target; t.mode = mode; t.max_iter = max_iter;
    int s = chain::solve_batch(d_s, d_c, &t, 1, d_m, res, 0, st);
    if (s != 0) return s;
    RB_CUDA(cudaMemcpyAsync(mask_out, d_m, n, cudaMemcpyDeviceToHost, st));
    RB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

extern "C" __attribute__((visibility("default"))) int rocco_solve_penalized_chain_f64(
    const double *scores, const double *switch_costs, size_t n, double selection_penalty,
    uint8_t *solution_out, double *penalized_objective_out, long long *selected_count_out)
{
    rocco_b200_chain_result r{};
    int s = host_chain(scores, switch_costs, n, 0, selection_penalty, 0, 0, solution_out, &r);
    if (s != 0) return s;
    if (penalized_objective_out) *penalized_objective_out = r.penalized_objective;
    if (selected_count_out) *selected_count_out = r.selected_count;
    return 0;
}

extern "C" __attribute__((visibility("default"))) int rocco_calibrate_selection_penalty_f64(
    const double *scores, const double *switch_costs, size_t n, long long target_count, int max_iter,
    double *selection_penalty_out, uint8_t *solution_out, double *penalized_objective_out,
    long long *selected_count_out)
{
    rocco_b200_chain_result r{};
    int s = host_chain(scores, switch_costs, n, 1, 0.0, target_count, max_iter, solution_out, &r);
    if (s != 0) return s;
    if (selection_penalty_out) *selection_penalty_out = r.selection_penalty;
    if (penalized_objective_out) *penalized_objective_out = r.penalized_objective;
    if (selected_count_out) *selected_count_out = r.selected_count;
    return 0;
}
