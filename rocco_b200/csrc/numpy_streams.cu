// NumPy's default_rng(seed).standard_normal streams generated on the device: the innovations of the reference's budget
// null (one generator per draw, samples served in order) without a host array.
//
// The stream: PCG64 (XSL-RR 128/64) seeded through SeedSequence, and NumPy's 256-level ziggurat (random_standard_normal
// of numpy/random/src/distributions/distributions.c; tables in numpy_ziggurat.cuh).  An attempt takes one word on the
// fast path (99.2 % of normals), two on the wedge path (accepted or rejected) and 1 + 2k in the tail, so whether word p
// starts an attempt depends on every word before it.  The parse is made parallel by speculation:
//   * a segment of words is cut into chunks of C words, one thread per chunk (T chunks per block);
//   * k_np_parse: every chunk parses itself from each entry overhang e in [0, E) -- the first attempt starting at word
//     e of the chunk -- and records the exit overhang into the next chunk and the normals it returned; a block composes
//     the maps of its chunks the same way;
//   * k_np_scan: one CTA follows the true path through the block maps (groups of blocks composed in parallel first) and
//     gives every block its true entry and the index of its first normal;
//   * k_np_emit: a block follows the true path through its chunk maps, and every chunk re-parses itself from its true
//     entry and writes its normals.
// An overhang of E or more (a tail loop running past a chunk's end: rare) has no precomputed map; wherever one is met,
// the chunk is re-parsed serially from it (apply_chunk), so every path is exact.  A chunk's first state comes from a
// jump-ahead table of the LCG (MULT^(2^k) and 1 + MULT + .. + MULT^(2^k - 1)), never from stepping the generator.
//
// Exactness: the words every normal consumes, and every accept/reject decision, are NumPy's.  Fast-path and wedge normals
// are bit-identical (rabs * wi[idx] with a sign); the wedge and tail formulas are evaluated with explicit round-to-nearest
// operations (no FMA contraction: NumPy's x86-64 baseline build has none).  Tail normals go through log1p, which glibc
// does not round correctly and whose result NumPy takes from the host's libm, so they can differ from a given host's
// NumPy in the last bit.
#include <algorithm>
#include <atomic>
#include <mutex>

#include "numpy_streams.cuh"
#include "numpy_ziggurat.cuh"

namespace rb {
namespace npz {

constexpr int E = 4;                   // entry overhangs with a precomputed map
constexpr int T = 128;                 // chunks (threads) per block
constexpr int MAX_BLOCKS = 8192;       // blocks per segment (2^26 words at 64 words per chunk)
constexpr int SCAN_GROUPS = 256;       // k_np_scan: groups of blocks composed in parallel
constexpr int MAX_CHUNK_WORDS = 256;   // keeps a block's normal count and every overhang within int
static std::atomic<int> g_chunk_words{64};  // measured on a B200: 64 words parse 1.45x faster than 32, emit the same

constexpr double NOR_R = 3.6541528853610087963519472518;
constexpr double NOR_INV_R = 0.27366123732975827203338247596;
constexpr unsigned long long MULT_HI = 0x2360ED051FC65DA4ull, MULT_LO = 0x4385DF649FCCF645ull;

struct Jump { unsigned long long a_lo, a_hi, g_lo, g_hi; };     // 2^k steps: s -> A s + inc G
__constant__ Jump c_jump[64];

__host__ __device__ __forceinline__ u128 mk128(unsigned long long lo, unsigned long long hi) { return ((u128)hi << 64) | lo; }

__device__ __forceinline__ unsigned long long next64(u128 &s, u128 inc)
{
    s = s * mk128(MULT_LO, MULT_HI) + inc;
    const unsigned long long hi = (unsigned long long)(s >> 64), x = hi ^ (unsigned long long)s;
    const unsigned rot = (unsigned)(hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
}

__device__ u128 jump(u128 s, u128 inc, unsigned long long k)
{
    for (int b = 0; k; ++b, k >>= 1)
        if (k & 1) {
            const Jump j = c_jump[b];
            s = s * mk128(j.a_lo, j.a_hi) + inc * mk128(j.g_lo, j.g_hi);
        }
    return s;
}

struct Tables { unsigned long long ki[256]; double wi[256], fi[256]; };

__device__ void load_tables(Tables &z)
{
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        z.ki[i] = ZIG_KI[i];
        z.wi[i] = __longlong_as_double((long long)ZIG_WI_BITS[i]);
        z.fi[i] = __longlong_as_double((long long)ZIG_FI_BITS[i]);
    }
    __syncthreads();
}

__device__ __forceinline__ double unit_double(unsigned long long w) { return (double)(w >> 11) * (1.0 / 9007199254740992.0); }

// The attempt that starts with word w0; w1 is the next word and s the generator after it.  Returns the words the attempt
// takes; *ok: it returned a normal, *val.
__device__ __forceinline__ int attempt(unsigned long long w0, unsigned long long w1, u128 s, u128 inc, const Tables &z, bool *ok,
                                       double *val)
{
    const int idx = (int)(w0 & 0xFF);
    const unsigned long long r = w0 >> 8;
    const unsigned long long rabs = (r >> 1) & 0x000FFFFFFFFFFFFFull;
    double x = __dmul_rn((double)rabs, z.wi[idx]);
    if (r & 1) x = -x;
    *val = x;
    if (rabs < z.ki[idx]) { *ok = true; return 1; }
    if (idx == 0) {                                       // tail: pairs of doubles until one is accepted
        unsigned long long a = w1;
        for (int len = 3;; len += 2) {
            const unsigned long long b = next64(s, inc);
            const double xx = __dmul_rn(-NOR_INV_R, log1p(-unit_double(a)));
            const double yy = -log1p(-unit_double(b));
            if (__dadd_rn(yy, yy) > __dmul_rn(xx, xx)) {
                const double v = __dadd_rn(NOR_R, xx);
                *val = ((rabs >> 8) & 1) ? -v : v;
                *ok = true;
                return len;
            }
            a = next64(s, inc);
        }
    }
    const double lhs = __dadd_rn(__dmul_rn(__dadd_rn(z.fi[idx - 1], -z.fi[idx]), unit_double(w1)), z.fi[idx]);
    *ok = lhs < exp(__dmul_rn(__dmul_rn(-0.5, x), x));
    return 2;
}

struct Emit {
    double *out;
    long long lo, hi;                  // window of normal indices written to out[g - lo]
    long long g;                       // index of the path's next normal
    unsigned long long w;              // absolute index of the chunk's first word
    unsigned long long *end;           // word after the attempt of normal hi - 1
};

// Parse the attempts that start in words [0, C) of a chunk (s: the generator at the chunk's first word).  Path q's first
// attempt starts at word pos[q]; on return pos[q] - C is its overhang into the next chunk and cnt[q] the normals it got.
template <int NP, bool EMIT>
__device__ __forceinline__ void parse_chunk(u128 s, u128 inc, int C, int (&pos)[NP], int (&cnt)[NP], const Tables &z, Emit *em)
{
    int first = pos[0];
#pragma unroll
    for (int q = 1; q < NP; ++q) first = min(first, pos[q]);
    if (first >= C) return;
    if (first > 0) s = jump(s, inc, (unsigned long long)first);
    unsigned long long w0 = next64(s, inc), w1 = next64(s, inc);
    for (int p = first; p < C; ++p) {
        bool hit = false;
#pragma unroll
        for (int q = 0; q < NP; ++q) hit |= pos[q] == p;
        if (hit) {
            bool ok;
            double v;
            const int len = attempt(w0, w1, s, inc, z, &ok, &v);
#pragma unroll
            for (int q = 0; q < NP; ++q)
                if (pos[q] == p) { pos[q] += len; cnt[q] += ok ? 1 : 0; }
            if (EMIT && ok) {
                const long long g = em->g++;
                if (g >= em->lo) em->out[g - em->lo] = v;
                if (g == em->hi - 1) { *em->end = em->w + (unsigned long long)(p + len); return; }
            }
        }
        w0 = w1;
        w1 = next64(s, inc);
    }
}

// Chunk j of the segment (first state s0) entered with any overhang x: the exit overhang; *cnt the normals.
__device__ int apply_chunk(u128 s0, u128 inc, int C, long long j, int x, const Tables &z, long long *cnt)
{
    if (x >= C) return x - C;
    int pos[1] = {x}, c[1] = {0};
    parse_chunk<1, false>(jump(s0, inc, (unsigned long long)j * (unsigned long long)C), inc, C, pos, c, z, nullptr);
    *cnt += c[0];
    return pos[0] - C;
}

__device__ __forceinline__ int lane_of(const int4 &v, int e) { return e == 0 ? v.x : e == 1 ? v.y : e == 2 ? v.z : v.w; }

// one step of a path through chunk j, from the chunk's map or (overhang >= E) by re-parsing it
__device__ __forceinline__ int step_chunk(const int4 &ex, const int4 &cn, u128 s0, u128 inc, int C, long long j, int x,
                                          const Tables &z, long long *cnt)
{
    if (x < E) { *cnt += lane_of(cn, x); return lane_of(ex, x); }
    return apply_chunk(s0, inc, C, j, x, z, cnt);
}

__device__ __forceinline__ u128 block_state(u128 s0, u128 inc, int C, u128 *s_state)
{
    if (threadIdx.x == 0) *s_state = jump(s0, inc, (unsigned long long)blockIdx.x * T * (unsigned long long)C);
    __syncthreads();
    return jump(*s_state, inc, (unsigned long long)threadIdx.x * (unsigned long long)C);
}

// ------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(T) k_np_parse(unsigned long long s_lo, unsigned long long s_hi, unsigned long long i_lo,
                                                unsigned long long i_hi, int C, int4 *__restrict__ cex, int4 *__restrict__ ccn,
                                                int *__restrict__ bex, int *__restrict__ bcn)
{
    __shared__ Tables z;
    __shared__ int4 s_ex[T], s_cn[T];
    __shared__ u128 s_state;
    load_tables(z);
    const u128 s0 = mk128(s_lo, s_hi), inc = mk128(i_lo, i_hi);
    const u128 s = block_state(s0, inc, C, &s_state);
    int pos[E], cnt[E];
#pragma unroll
    for (int e = 0; e < E; ++e) { pos[e] = e; cnt[e] = 0; }
    parse_chunk<E, false>(s, inc, C, pos, cnt, z, nullptr);
    const int4 ex = make_int4(pos[0] - C, pos[1] - C, pos[2] - C, pos[3] - C), cn = make_int4(cnt[0], cnt[1], cnt[2], cnt[3]);
    const long long j = (long long)blockIdx.x * T + threadIdx.x;
    cex[j] = ex;
    ccn[j] = cn;
    s_ex[threadIdx.x] = ex;
    s_cn[threadIdx.x] = cn;
    __syncthreads();
    if (threadIdx.x < E) {
        int x = threadIdx.x;
        long long c = 0;
        for (int t = 0; t < T; ++t) x = step_chunk(s_ex[t], s_cn[t], s0, inc, C, (long long)blockIdx.x * T + t, x, z, &c);
        bex[blockIdx.x * E + threadIdx.x] = x;
        bcn[blockIdx.x * E + threadIdx.x] = (int)c;
    }
}

// block b entered with overhang x: the exit overhang; *cnt += its normals
__device__ int apply_block(const int4 *__restrict__ cex, const int4 *__restrict__ ccn, const int *__restrict__ bex,
                           const int *__restrict__ bcn, u128 s0, u128 inc, int C, long long b, int x, const Tables &z, long long *cnt)
{
    if (x < E) { *cnt += bcn[b * E + x]; return bex[b * E + x]; }
    for (int t = 0; t < T; ++t) {
        const long long j = b * T + t;
        x = step_chunk(cex[j], ccn[j], s0, inc, C, j, x, z, cnt);
    }
    return x;
}

// One CTA of SCAN_GROUPS * E threads: true entry and first normal (relative to the segment) of every block; tot = {exit
// overhang, normals} of the segment.
__global__ void __launch_bounds__(SCAN_GROUPS *E) k_np_scan(unsigned long long s_lo, unsigned long long s_hi, unsigned long long i_lo,
                                                            unsigned long long i_hi, int C, int nblocks, int entry,
                                                            const int4 *__restrict__ cex, const int4 *__restrict__ ccn,
                                                            const int *__restrict__ bex, const int *__restrict__ bcn,
                                                            int *__restrict__ bent, long long *__restrict__ bbase, long long *tot)
{
    __shared__ Tables z;
    __shared__ int g_ex[E][SCAN_GROUPS], g_ent[SCAN_GROUPS];
    __shared__ long long g_cn[E][SCAN_GROUPS], g_base[SCAN_GROUPS];
    load_tables(z);
    const u128 s0 = mk128(s_lo, s_hi), inc = mk128(i_lo, i_hi);
    const int per = (nblocks + SCAN_GROUPS - 1) / SCAN_GROUPS;
    const int g = threadIdx.x % SCAN_GROUPS, e = threadIdx.x / SCAN_GROUPS;
    const int b0 = min(nblocks, g * per), b1 = min(nblocks, b0 + per);
    {
        int x = e;
        long long c = 0;
        for (int b = b0; b < b1; ++b) x = apply_block(cex, ccn, bex, bcn, s0, inc, C, b, x, z, &c);
        g_ex[e][g] = x;
        g_cn[e][g] = c;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int x = entry;
        long long base = 0;
        for (int q = 0; q < SCAN_GROUPS; ++q) {
            g_ent[q] = x;
            g_base[q] = base;
            if (x < E) { base += g_cn[x][q]; x = g_ex[x][q]; }
            else
                for (int b = min(nblocks, q * per); b < min(nblocks, q * per + per); ++b)
                    x = apply_block(cex, ccn, bex, bcn, s0, inc, C, b, x, z, &base);
        }
        tot[0] = x;
        tot[1] = base;
        bbase[nblocks] = base;
    }
    __syncthreads();
    if (e == 0) {
        int x = g_ent[g];
        long long c = g_base[g];
        for (int b = b0; b < b1; ++b) {
            bent[b] = x;
            bbase[b] = c;
            x = apply_block(cex, ccn, bex, bcn, s0, inc, C, b, x, z, &c);
        }
    }
}

// Every chunk re-parses itself from its true entry and writes its normals in [lo, hi) to out[g - lo].  (Staging a block's
// normals in shared memory for coalesced stores was measured no faster: the kernel is bound by the parse, not the stores.)
__global__ void __launch_bounds__(T) k_np_emit(unsigned long long s_lo, unsigned long long s_hi, unsigned long long i_lo,
                                               unsigned long long i_hi, int C, const int4 *__restrict__ cex, const int4 *__restrict__ ccn,
                                               const int *__restrict__ bent, const long long *__restrict__ bbase, long long seg_normal,
                                               unsigned long long seg_word, long long lo, long long hi, double *__restrict__ out,
                                               unsigned long long *end)
{
    const long long b = blockIdx.x;
    const long long g0 = seg_normal + bbase[b], g1 = seg_normal + bbase[b + 1];
    if (g1 <= lo || g0 >= hi) return;                      // uniform over the block
    __shared__ Tables z;
    __shared__ int4 s_ex[T], s_cn[T];
    __shared__ int s_ent[T];
    __shared__ long long s_g[T + 1];
    __shared__ u128 s_state;
    const long long j = b * T + threadIdx.x;
    s_ex[threadIdx.x] = cex[j];
    s_cn[threadIdx.x] = ccn[j];
    load_tables(z);
    const u128 s0 = mk128(s_lo, s_hi), inc = mk128(i_lo, i_hi);
    const u128 s = block_state(s0, inc, C, &s_state);
    if (threadIdx.x == 0) {
        int x = bent[b];
        long long c = g0;
        for (int t = 0; t < T; ++t) {
            s_ent[t] = x;
            s_g[t] = c;
            x = step_chunk(s_ex[t], s_cn[t], s0, inc, C, b * T + t, x, z, &c);
        }
        s_g[T] = c;
    }
    __syncthreads();
    const int t = threadIdx.x;
    if (s_g[t + 1] <= lo || s_g[t] >= hi || s_g[t + 1] == s_g[t]) return;
    int pos[1] = {s_ent[t]}, cnt[1] = {0};
    Emit em{out, lo, hi, s_g[t], seg_word + (unsigned long long)j * (unsigned long long)C, end};
    parse_chunk<1, true>(s, inc, C, pos, cnt, z, &em);
}

// ------------------------------------------------------------------ host side
static Jump h_jump[64];
static std::once_flag h_jump_once;

static void init_jump()
{
    u128 A = mk128(MULT_LO, MULT_HI), G = 1;
    for (int k = 0; k < 64; ++k) {
        h_jump[k] = Jump{(unsigned long long)A, (unsigned long long)(A >> 64), (unsigned long long)G, (unsigned long long)(G >> 64)};
        G = G + A * G;
        A = A * A;
    }
}

static u128 host_jump(u128 s, u128 inc, unsigned long long k)
{
    std::call_once(h_jump_once, init_jump);
    for (int b = 0; k; ++b, k >>= 1)
        if (k & 1) s = s * mk128(h_jump[b].a_lo, h_jump[b].a_hi) + inc * mk128(h_jump[b].g_lo, h_jump[b].g_hi);
    return s;
}

static int ensure_jump(cudaStream_t st)
{
    std::call_once(h_jump_once, init_jump);
    static std::atomic<bool> done[64];
    int dev = 0;
    RB_CUDA(cudaGetDevice(&dev));
    if (!done[dev & 63].load()) {
        RB_CUDA(cudaMemcpyToSymbolAsync(c_jump, h_jump, sizeof(h_jump), 0, cudaMemcpyHostToDevice, st));
        RB_CUDA(cudaStreamSynchronize(st));
        done[dev & 63].store(true);
    }
    return 0;
}

Cursor seed_cursor(u128 seed)
{
    // SeedSequence(seed): entropy = little-endian 32-bit words (at least one), pool of 4, then generate_state(4, uint64)
    constexpr uint32_t INIT_A = 0x43B0D7E5u, MULT_A = 0x931E8875u, INIT_B = 0x8B51F9DDu, MULT_B = 0x58F38DEDu;
    constexpr uint32_t MIX_L = 0xCA01F9DDu, MIX_R = 0x4973F715u;
    std::vector<uint32_t> ent;
    do { ent.push_back((uint32_t)seed); seed >>= 32; } while (seed != 0);
    uint32_t hc = INIT_A;
    auto hashmix = [&hc](uint32_t v) { v ^= hc; hc *= MULT_A; v *= hc; v ^= v >> 16; return v; };
    auto mix = [](uint32_t x, uint32_t y) { uint32_t r = MIX_L * x - MIX_R * y; r ^= r >> 16; return r; };
    uint32_t pool[4];
    for (int i = 0; i < 4; ++i) pool[i] = hashmix(i < (int)ent.size() ? ent[(size_t)i] : 0u);
    for (int src = 0; src < 4; ++src)
        for (int dst = 0; dst < 4; ++dst)
            if (src != dst) pool[dst] = mix(pool[dst], hashmix(pool[src]));
    for (size_t src = 4; src < ent.size(); ++src)
        for (int dst = 0; dst < 4; ++dst) pool[dst] = mix(pool[dst], hashmix(ent[src]));
    uint32_t hb = INIT_B, w[8];
    for (int i = 0; i < 8; ++i) {
        uint32_t v = pool[i & 3];
        v ^= hb; hb *= MULT_B; v *= hb; v ^= v >> 16;
        w[i] = v;
    }
    unsigned long long v[4];
    for (int k = 0; k < 4; ++k) v[k] = (unsigned long long)w[2 * k] | ((unsigned long long)w[2 * k + 1] << 32);
    Cursor c;
    const u128 initstate = mk128(v[1], v[0]);
    c.inc = (mk128(v[3], v[2]) << 1) | 1;
    c.state = (c.inc + initstate) * mk128(MULT_LO, MULT_HI) + c.inc;
    return c;
}

int Scratch::alloc(Arena &ar, long long max_normals)
{
    chunk_words = g_chunk_words.load();
    const long long W = (long long)T * chunk_words;
    const long long words = max_normals + max_normals / 32 + 64;
    blocks = (int)std::min<long long>(MAX_BLOCKS, std::max<long long>(1, (words + W - 1) / W));
    const size_t chunks = (size_t)blocks * T;
    RB_TRY(ar.alloc(&cex, chunks));
    RB_TRY(ar.alloc(&ccn, chunks));
    RB_TRY(ar.alloc(&bex, (size_t)blocks * E));
    RB_TRY(ar.alloc(&bcn, (size_t)blocks * E));
    RB_TRY(ar.alloc(&bent, (size_t)blocks));
    RB_TRY(ar.alloc(&bbase, (size_t)blocks + 1));
    RB_TRY(ar.alloc(&tot, 2));
    return ar.alloc(&end, 1);
}

int generate(Cursor &cur, long long lo, long long hi, double *d_out, unsigned long long *words_end, Scratch &sc, cudaStream_t st)
{
    if (hi <= lo || lo < cur.normal || !d_out || sc.blocks <= 0) { set_error("numpy streams: bad normal window"); return ST_INVALID; }
    RB_TRY(ensure_jump(st));
    const int C = sc.chunk_words;
    const long long W = (long long)T * C;
    for (;;) {
        if (cur.overhang >= (1LL << 30)) { set_error("numpy streams: overhang out of range"); return ST_INVALID; }
        const unsigned long long a = (unsigned long long)cur.state, b = (unsigned long long)(cur.state >> 64);
        const unsigned long long c = (unsigned long long)cur.inc, d = (unsigned long long)(cur.inc >> 64);
        // a call that continues the previous one starts in the segment that call parsed last: its maps are still here
        const bool cached = sc.seg_valid && sc.seg.state == cur.state && sc.seg.inc == cur.inc && sc.seg.word == cur.word &&
                            sc.seg.overhang == cur.overhang && sc.seg.normal == cur.normal;
        int nb = sc.seg_blocks;
        long long tot[2] = {sc.seg_tot[0], sc.seg_tot[1]};
        if (!cached) {
            const long long need = hi - cur.normal;
            const long long words = need + need / 32 + 64 + cur.overhang;
            nb = (int)std::min<long long>(sc.blocks, std::max<long long>(1, (words + W - 1) / W));
            sc.seg_valid = false;
            {
                RB_PROF("k_np_parse", st, (double)nb * T * 32.0);
                k_np_parse<<<nb, T, 0, st>>>(a, b, c, d, C, sc.cex, sc.ccn, sc.bex, sc.bcn);
                RB_LAUNCH_CHECK();
            }
            k_np_scan<<<1, SCAN_GROUPS * E, 0, st>>>(a, b, c, d, C, nb, (int)cur.overhang, sc.cex, sc.ccn, sc.bex, sc.bcn,
                                                     sc.bent, sc.bbase, sc.tot);
            RB_LAUNCH_CHECK();
            RB_CUDA(cudaMemcpyAsync(tot, sc.tot, sizeof(tot), cudaMemcpyDeviceToHost, st));
            RB_CUDA(cudaStreamSynchronize(st));
            sc.seg = cur;
            sc.seg_blocks = nb;
            sc.seg_tot[0] = tot[0];
            sc.seg_tot[1] = tot[1];
            sc.seg_valid = true;
        }
        const long long seg_end = cur.normal + tot[1];
        if (seg_end > lo) {
            RB_PROF("k_np_emit", st, (double)(std::min(seg_end, hi) - std::max(cur.normal, lo)) * 8.0);
            k_np_emit<<<nb, T, 0, st>>>(a, b, c, d, C, sc.cex, sc.ccn, sc.bent, sc.bbase, cur.normal, cur.word, lo, hi, d_out, sc.end);
            RB_LAUNCH_CHECK();
        }
        if (seg_end >= hi) {
            if (words_end) {
                RB_CUDA(cudaMemcpyAsync(words_end, sc.end, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
                RB_CUDA(cudaStreamSynchronize(st));
            }
            return 0;
        }
        cur.state = host_jump(cur.state, cur.inc, (unsigned long long)(nb * W));
        cur.word += (unsigned long long)(nb * W);
        cur.overhang = tot[0];
        cur.normal = seg_end;
    }
}

}  // namespace npz
}  // namespace rb

// ==================================================================================== C ABI
using namespace rb;
#define RB_API __attribute__((visibility("default")))

extern "C" {

RB_API int rocco_b200_numpy_seed_state(unsigned long long seed_lo, unsigned long long seed_hi, unsigned long long out[4])
{
    if (!out) return ST_INVALID;
    const npz::Cursor c = npz::seed_cursor(npz::mk128(seed_lo, seed_hi));
    out[0] = (unsigned long long)c.state; out[1] = (unsigned long long)(c.state >> 64);
    out[2] = (unsigned long long)c.inc; out[3] = (unsigned long long)(c.inc >> 64);
    return 0;
}

RB_API int rocco_b200_numpy_normals_dev(unsigned long long seed_lo, unsigned long long seed_hi, unsigned long long skip,
                                        unsigned long long count, double *d_out, unsigned long long *words_consumed,
                                        void *cuda_stream)
{
    if (!d_out || count == 0 || skip > (1ull << 62) || count > (1ull << 62)) return ST_INVALID;
    RB_TRY(ensure_device());
    cudaStream_t st = (cudaStream_t)cuda_stream;
    Arena ar(st);
    npz::Scratch sc;
    RB_TRY(sc.alloc(ar, (long long)(skip + count)));
    npz::Cursor cur = npz::seed_cursor(npz::mk128(seed_lo, seed_hi));
    unsigned long long end = 0;
    RB_TRY(npz::generate(cur, (long long)skip, (long long)(skip + count), d_out, &end, sc, st));
    if (words_consumed) *words_consumed = end;
    return 0;
}

RB_API int rocco_b200_numpy_streams_set_chunk_words(int words)
{
    const int w = std::max(1, std::min(npz::MAX_CHUNK_WORDS, words > 0 ? words : 64));
    return npz::g_chunk_words.exchange(w);
}

}  // extern "C"
