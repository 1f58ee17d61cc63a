// ms_reads_core.h — paired-end reads drawn from the mutated genome of the last full apply (--reads), host/device
// shared: ms_reads.cu runs it on the device, tests/emu/reads_emu.cpp builds it with g++.
//
// Pair i of a contig (gid, mutated length Lp) on haplotype h, attempt a (0..7), reads words w0, w1, ... from the
// Philox blocks draw(seed, gid, P_READS | h << 8 | b << 12, i * 16 + a), b = 0, 1, 2, ... (word k = component k % 4
// of block k / 4):
//   fragment  Z = w0 + ... + w11 - 6 * 2^32 (Irwin-Hall(12), exact in int64), f = M + ((S * Z + 2^31) >> 32),
//             clamped to [L, Lp]
//   start     s = mulhi32(w12, Lp - f + 1); strand '+' when bit 0 of w13 is 0, else '-'
//   '+'       R1 = [s, s + L) forward, R2 = reverse complement of [s + f - L, s + f); '-' swaps the two ends
//   redraw    while either template end holds a byte other than A, C, G, T, with a + 1; attempt 7 is kept as drawn
//   errors    base j of R1 (as sequenced) uses v = w(16 + j), base j of R2 v = w(16 + L + j): an A/C/G/T base becomes
//             the (v mod 3)-th of the other three bases in ACGT order iff v < llround(E * 2^32); other bytes stay
// Only integer arithmetic decides bytes, so the g++ build and the device agree to the byte.  The truth in the read
// name lifts the leftmost template position of each read to the input genome along the primary chain (read_lift).
#pragma once
#include "ms_vcf_core.h"

namespace ms {

constexpr int32_t READS_MAX_LEN = 1000;
constexpr int32_t READS_MAX_FRAG_MEAN = 1000000;
constexpr int32_t READS_MAX_FRAG_SD = 100000;
constexpr uint32_t READS_ATTEMPTS = 8;

struct ReadsCfg {
    Seed seed;
    uint32_t hap;        // 1..8
    int32_t L, M, S;     // read length, fragment mean, fragment SD
    uint64_t err_thr;    // llround(E * 2^32)
    uint8_t qual;        // quality character of every base
};

// llround(E * 2^32) for 0 <= E < 1 (host side)
inline uint64_t read_error_threshold(double e) { return (uint64_t)llround(e * 4294967296.0); }

// One pair's draw and truth, kept by the size pass for the write pass.  24 bytes.
struct PairInfo {
    uint32_t s, f;           // template start and fragment length on the mutated contig
    int32_t lift1, lift2;    // input position of the leftmost template base of R1 / R2, -1 for '*'
    uint32_t meta;           // bit 0: strand ('-' = 1), bits 1..3: the attempt kept
    uint32_t size;           // bytes of one record (R1 and R2 records have the same size)
};
static_assert(sizeof(PairInfo) == 24, "PairInfo layout");

MS_HD U4 reads_block(const ReadsCfg& g, uint32_t gid, uint64_t i, uint32_t a, uint32_t b) {
    return draw(g.seed, gid, (uint32_t)P_READS | (g.hap << 8) | (b << 12), i * 16u + a);
}

MS_HD uint32_t u4_word(const U4& v, uint32_t k) { return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w; }

// mutated base q of contig k in the FASTA image (lines of bpl bases, each followed by '\n'); q < 2^31, so the line
// number is a 32-bit division (the write pass does one per base)
MS_HD int64_t image_off(const Contig& k, int64_t q) { return k.body_off + q + (int64_t)((uint32_t)q / (uint32_t)k.bpl); }

MS_HD bool is_acgt(uint8_t c) { return c == 'A' || c == 'C' || c == 'G' || c == 'T'; }

// all of [q, q + n) of contig k are A/C/G/T; walks the line layout instead of dividing per base
MS_HD bool run_acgt(const uint8_t* img, const Contig& k, int64_t q, int32_t n) {
    int64_t o = image_off(k, q);
    int64_t col = (int64_t)((uint32_t)q % (uint32_t)k.bpl);
    for (int32_t j = 0; j < n; ++j) {
        if (!is_acgt(img[o])) return false;
        ++o;
        if (++col == k.bpl) { col = 0; ++o; }
    }
    return true;
}

// fragment length, start and strand of attempt a (Lp >= L)
MS_HD void pair_geometry(const ReadsCfg& g, uint32_t gid, uint64_t i, uint32_t a, int64_t Lp, uint32_t& s, uint32_t& f,
                         uint32_t& strand) {
    int64_t z = -6ll * 4294967296ll;
    for (uint32_t b = 0; b < 3; ++b) {
        const U4 v = reads_block(g, gid, i, a, b);
        z += (int64_t)v.x + (int64_t)v.y + (int64_t)v.z + (int64_t)v.w;
    }
    int64_t fl = (int64_t)g.M + (((int64_t)g.S * z + (1ll << 31)) >> 32);
    if (fl < g.L) fl = g.L;
    if (fl > Lp) fl = Lp;
    const U4 v3 = reads_block(g, gid, i, a, 3);
    f = (uint32_t)fl;
    s = mulhi32(v3.x, (uint32_t)(Lp - fl + 1));
    strand = v3.y & 1u;
}

// the attempt kept for pair i: the first whose two template ends are A/C/G/T only, else attempt 7
MS_HD uint32_t pair_draw(const ReadsCfg& g, const uint8_t* img, const Contig& k, uint64_t i, uint32_t& s, uint32_t& f,
                         uint32_t& strand) {
    uint32_t a = 0;
    for (;; ++a) {
        pair_geometry(g, k.gid, i, a, k.out_len, s, f, strand);
        if (a + 1 == READS_ATTEMPTS) break;
        if (run_acgt(img, k, s, g.L) && run_acgt(img, k, (int64_t)s + f - g.L, g.L)) break;
    }
    return a;
}

// Input position of mutated position q of contig k (records [rec_lo, rec_hi) with out filled in), -1 for a base that
// no input base maps to along the primary chain (inserted, duplicated, inverted or translocated).  r = the last
// record with out <= q: q inside its payload lifts to pos for a SNP, else to nothing; past it, the copy run after r.
MS_HD int64_t read_lift(const Rec* recs, const Contig& k, int64_t q) {
    int64_t lo = k.rec_lo, hi = k.rec_hi;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((int64_t)recs[mid].out <= q) lo = mid + 1; else hi = mid;
    }
    if (lo == k.rec_lo) return q;
    const Rec& r = recs[lo - 1];
    if (q < (int64_t)r.out + r.prod) return r.kind == K_SNP ? (int64_t)r.pos : -1;
    return (int64_t)r.pos + r.cons + (q - (int64_t)r.out - r.prod);
}

MS_HD PairInfo pair_info(const ReadsCfg& g, const uint8_t* img, const Rec* recs, const Contig& k, uint64_t i) {
    PairInfo p;
    uint32_t strand;
    const uint32_t a = pair_draw(g, img, k, i, p.s, p.f, strand);
    const int64_t left = p.s, right = (int64_t)p.s + p.f - g.L;
    p.lift1 = (int32_t)read_lift(recs, k, strand ? right : left);
    p.lift2 = (int32_t)read_lift(recs, k, strand ? left : right);
    p.meta = strand | (a << 1);
    p.size = 0;
    return p;
}

// "@name:h:i:s+1:f:strand:lift1+1:lift2+1/m\n" (lifts '*' when -1)
template <class S>
MS_HD void read_header(S& s, const uint8_t* names, const Contig& k, uint32_t hap, uint32_t i, const PairInfo& p, uint8_t mate) {
    s.put('@');
    if constexpr (S::counting) s.skip((uint32_t)k.name_len);
    else for (int32_t j = 0; j < k.name_len; ++j) s.put(names[k.name_src + j]);
    s.put(':'); put_uint(s, hap); s.put(':'); put_uint(s, i); s.put(':'); put_uint(s, p.s + 1u); s.put(':');
    put_uint(s, p.f); s.put(':'); s.put((p.meta & 1u) ? '-' : '+'); s.put(':');
    if (p.lift1 < 0) s.put('*'); else put_uint(s, (uint32_t)p.lift1 + 1u);
    s.put(':');
    if (p.lift2 < 0) s.put('*'); else put_uint(s, (uint32_t)p.lift2 + 1u);
    s.put('/'); s.put(mate); s.put('\n');
}

MS_HD uint32_t read_record_size(const Contig& k, uint32_t hap, uint32_t i, const PairInfo& p, int32_t L) {
    CountSink c;
    read_header(c, nullptr, k, hap, i, p, '1');
    return c.n + 2u * (uint32_t)L + 4u;
}

// base j (0..L-1) of mate m (1 or 2) as sequenced, before errors
MS_HD uint8_t read_template_base(const uint8_t* img, const uint8_t* comp, const Contig& k, const PairInfo& p, int32_t L, int mate,
                                 int32_t j) {
    const bool forward = (mate == 1) == ((p.meta & 1u) == 0u);
    if (forward) return img[image_off(k, (int64_t)p.s + j)];
    return comp[img[image_off(k, (int64_t)p.s + p.f - 1 - j)]];
}

MS_HD uint8_t read_error(uint8_t b, uint32_t v, uint64_t thr) {
    if (!is_acgt(b) || (uint64_t)v >= thr) return b;
    const uint32_t me = b == 'A' ? 0u : b == 'C' ? 1u : b == 'G' ? 2u : 3u;
    uint32_t x = v % 3u;
    if (x >= me) ++x;
    return (uint8_t)"ACGT"[x];
}

// error word k (16 + j for R1 base j, 16 + L + j for R2 base j) of the attempt kept
MS_HD uint32_t read_error_word(const ReadsCfg& g, uint32_t gid, uint64_t i, const PairInfo& p, uint32_t k) {
    return u4_word(reads_block(g, gid, i, (p.meta >> 1) & 7u, k >> 2), k & 3u);
}

// One whole record of mate m, base by base (the host build; the device writes the sequence a warp at a time)
template <class S>
MS_HD void read_record(S& s, const ReadsCfg& g, const uint8_t* img, const uint8_t* comp, const uint8_t* names, const Contig& k,
                       uint32_t i, const PairInfo& p, int mate) {
    read_header(s, names, k, g.hap, i, p, (uint8_t)('0' + mate));
    const uint32_t w0 = 16u + (mate == 1 ? 0u : (uint32_t)g.L);
    for (int32_t j = 0; j < g.L; ++j)
        s.put(read_error(read_template_base(img, comp, k, p, g.L, mate, j), read_error_word(g, k.gid, i, p, w0 + (uint32_t)j),
                         g.err_thr));
    put_str(s, "\n+\n", 3);
    for (int32_t j = 0; j < g.L; ++j) s.put(g.qual);
    s.put('\n');
}

}  // namespace ms
