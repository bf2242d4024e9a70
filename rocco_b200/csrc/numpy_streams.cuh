// NumPy's Generator(PCG64).standard_normal streams on the device (numpy_streams.cu): what the budget null needs to draw
// the reference's own innovations without a host array.
#pragma once
#include "common.cuh"

namespace rb {
namespace npz {

typedef unsigned __int128 u128;

// A position in one generator's stream: the generator state at word `word` (the next next_u64 returns word `word`), the
// first attempt of the ziggurat starting at word + overhang, whose normal (if it returns one) has index `normal`.
struct Cursor {
    u128 state = 0, inc = 0;
    unsigned long long word = 0;
    long long overhang = 0, normal = 0;
};

// default_rng(seed) for an integer seed >= 0 (SeedSequence -> PCG64), positioned at its first word.
Cursor seed_cursor(u128 seed);

// Scratch of generate(): sized for `max_normals` (the largest count a call asks for; bounds the segment length).
struct Scratch {
    int4 *cex = nullptr, *ccn = nullptr;       // per chunk, per entry overhang: exit overhang, normals
    int *bex = nullptr, *bcn = nullptr;        // the same per block, [block][entry]
    int *bent = nullptr;                       // per block: true entry overhang
    long long *bbase = nullptr;                // per block (+1): first normal, relative to the segment
    long long *tot = nullptr;                  // segment: exit overhang, normals
    unsigned long long *end = nullptr;         // word after the attempt that returned the last requested normal
    int blocks = 0, chunk_words = 0;
    // the segment parsed last (maps above): a call continuing from it emits from these maps without parsing again
    Cursor seg;
    int seg_blocks = 0;
    long long seg_tot[2] = {0, 0};
    bool seg_valid = false;
    int alloc(Arena &ar, long long max_normals);
};

// Write normals [lo, hi) of the stream into d_out[0 .. hi - lo) (hi > lo, lo >= cur.normal).  The cursor is advanced to
// the start of the segment that holds normal hi - 1, so a following call with lo >= hi continues from there.
// words_end (host, optional): the number of words the stream has consumed once normal hi - 1 is returned.
int generate(Cursor &cur, long long lo, long long hi, double *d_out, unsigned long long *words_end, Scratch &sc, cudaStream_t st);

}  // namespace npz
}  // namespace rb
