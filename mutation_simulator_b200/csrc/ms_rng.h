// ms_rng.h — counter-based randomness shared by host and device code.
//
//  * Philox4x32-10 (Salmon et al., SC'11) for every iid draw.  The stream is a
//    pure function of (seed, contig, purpose, index), so results do not depend
//    on the GPU count, the partition of contigs over GPUs, or launch geometry
//    (BASELINE.json north_star (a)).
//  * A Philox-keyed Feistel permutation with cycle walking (a uniform random
//    injection without any redraw round) pairs TLs with TLIs (mutator.py:277-285).
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define MS_HD __host__ __device__ __forceinline__
#else
#define MS_HD inline
#endif

namespace ms {

struct U4 { uint32_t x, y, z, w; };

MS_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

MS_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// Philox4x32-10.  ctr = 128-bit counter, key = 64-bit key.
MS_HD U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = mulhi32(M0, c.x), lo0 = M0 * c.x;
        uint32_t hi1 = mulhi32(M1, c.z), lo1 = M1 * c.z;
        U4 n;
        n.x = hi1 ^ c.y ^ k0;
        n.y = lo1;
        n.z = hi0 ^ c.w ^ k1;
        n.w = lo0;
        c = n;
        k0 += W0;
        k1 += W1;
    }
    return c;
}

// Purposes (second counter word).  One purpose per independent stream.
enum Purpose : uint32_t {
    P_RANGE_KEY = 1,   // sub-key of one RMT range: bucket-count splits and in-bucket position draws (util.py:104)
    P_TYPE_LEN  = 2,   // type + length of one candidate                            (mutator.py:170-174, 229-265)
    P_SNP       = 3,   // ti/tv decision + transversion coin of one SNP             (mutator.py:429-455)
    P_INSERT    = 4,   // random insert bases, 64 per Philox block                  (mutator.py:466-471)
    P_TL_PRP    = 5,   // round keys of the TL<->TLI pairing permutation of a contig (mutator.py:277-285)
    P_TL_REV    = 6,   // inversion coin of one translocation                       (mutator.py:307-316)
    P_IT_KEY    = 7,   // the same for the breakpoint ranges of an interchromosomal pair (it_mutator.py:94-118)
    P_GENOME    = 8,   // synthetic genome generator (bench only)
    P_GENOTYPE  = 9,   // haplotype mask of one record of a polyploid run (ms_genotype_core.h)
    P_READS     = 10,  // fragment, start, strand and errors of one read pair (ms_reads_core.h)
};

struct Seed { uint32_t k0, k1; };

MS_HD Seed make_seed(uint64_t s) { return Seed{(uint32_t)s, (uint32_t)(s >> 32)}; }

// One Philox block addressed by (contig, purpose, 64-bit index).
MS_HD U4 draw(Seed s, uint32_t contig, uint32_t purpose, uint64_t idx) {
    U4 c{contig, purpose, (uint32_t)idx, (uint32_t)(idx >> 32)};
    return philox4x32_10(c, s.k0, s.k1);
}

MS_HD uint64_t u64_of(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// 53-bit uniform double in [0,1), like random.random()/numpy's random_sample.
MS_HD double unit_double(uint32_t lo, uint32_t hi) {
    return (double)(u64_of(lo, hi) >> 11) * (1.0 / 9007199254740992.0);
}

// Uniform integer in [0, n) from 64 random bits (multiply-high; bias < n/2^64).
MS_HD uint64_t bounded(uint64_t r, uint64_t n) { return mulhi64(r, n); }

// ---------------------------------------------------------------------------
// Pseudo-random permutation of range(n), n < 2^32: a Feistel network over the
// mixed-radix domain [0,a) x [0,b) with a = ceil(sqrt n), b = ceil(n / a) and
// modular addition as the combiner, plus cycle walking for the a*b - n < a + b
// values that fall outside the range (re-encrypted until they land inside).
// Because a*b exceeds n by at most ~2 sqrt(n), a walk is needed with probability
// ~2/sqrt(n): on a GPU every lane of a warp finishes in the same pass (the
// power-of-two Feistel this replaces walked with probability up to 1/2 and ran
// at 16-18 active lanes, profiles/r1e, r1m).
// ---------------------------------------------------------------------------
// Rounds: 8 on domains of >= 2^12 values (statistically flat for k-subsets of genome-sized ranges);
// 16 on tiny domains, where each round function has only a few output values (tests/test_emu.py checks
// that all arrangements of small domains are equally likely over keys).
constexpr int PRP_MAX_ROUNDS = 16;

struct Prp {
    uint32_t key[PRP_MAX_ROUNDS];
    uint32_t n;        // domain size
    uint32_t rounds;
    uint32_t a;        // radix of the high digit
    uint32_t b;        // radix of the low digit (a * b >= n)
};

MS_HD uint32_t mix32(uint32_t x, uint32_t k) {
    x ^= k;
    x *= 0x9E3779B1u;
    x ^= x >> 15;
    x *= 0x85EBCA77u;
    x ^= x >> 13;
    x *= 0xC2B2AE3Du;
    x ^= x >> 16;
    return x;
}

MS_HD Prp make_prp(Seed s, uint32_t contig, uint32_t purpose, uint64_t idx, uint32_t n) {
    Prp p;
    p.n = n;
    p.rounds = n >= 4096u ? 8u : 16u;
    for (uint32_t b = 0; b < PRP_MAX_ROUNDS / 4; ++b) {
        U4 r{0, 0, 0, 0};
        if (4 * b < p.rounds) r = draw(s, contig, purpose | ((uint32_t)(b + 1) << 8), idx);
        p.key[4 * b + 0] = r.x; p.key[4 * b + 1] = r.y; p.key[4 * b + 2] = r.z; p.key[4 * b + 3] = r.w;
    }
    // a = ceil(sqrt(n)) by integer correction of the floating-point root (n < 2^32: a <= 65536)
    uint32_t a = (uint32_t)sqrt((double)n);
    while ((uint64_t)a * a < (uint64_t)n) ++a;
    while (a > 1u && (uint64_t)(a - 1u) * (a - 1u) >= (uint64_t)n) --a;
    if (a == 0u) a = 1u;
    p.a = a;
    p.b = n == 0u ? 1u : (uint32_t)(((uint64_t)n + a - 1u) / a);
    return p;
}

MS_HD uint32_t prp_apply(const Prp& p, uint32_t j) {
    const uint32_t a = p.a, b = p.b;
    uint32_t x = j;
    do {
        uint32_t hi = x / b, lo = x - hi * b;          // hi < a because x < n <= a * b
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int r = 0; r < 8; r += 2) {
            hi += mulhi32(mix32(lo, p.key[r]), a);      if (hi >= a) hi -= a;
            lo += mulhi32(mix32(hi, p.key[r + 1]), b);  if (lo >= b) lo -= b;
        }
        if (p.rounds > 8u) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 8; r < PRP_MAX_ROUNDS; r += 2) {
                hi += mulhi32(mix32(lo, p.key[r]), a);      if (hi >= a) hi -= a;
                lo += mulhi32(mix32(hi, p.key[r + 1]), b);  if (lo >= b) lo -= b;
            }
        }
        x = hi * b + lo;
    } while (x >= p.n);
    return x;
}

}  // namespace ms
