// ms_records.h — the splice descriptor shared by every apply-side kernel, plus
// the byte tables of mutator.py:75-77.  Host/device shared (no CUDA types).
#pragma once
#include <stdint.h>
#include "ms_rng.h"

namespace ms {

// Reference mutation types in the reference's ARGS dict order
// (rmt.py:443-450 + :91-94; mut_types.py:4-12).  IT_SEG is ours: one
// partner-contig interval of an interchromosomal swap (it_mutator.py:133-142).
enum MutType : uint8_t { T_SN = 0, T_IN = 1, T_DE = 2, T_IV = 3, T_DU = 4, T_TL = 5, T_TLI = 6, T_IT = 7, T_DEAD = 0xFF };

// What a record writes before its trailing copy run.
enum Kind : uint8_t {
    K_NONE = 0,  // nothing (DE, TL)
    K_SNP  = 1,  // one byte: rec.alt
    K_LIT  = 2,  // prod bytes from the literal pool at src (random inserts, replayed ALT strings)
    K_RAW  = 3,  // prod raw genome bytes from src          (DU, IT partner interval)
    K_CONV = 4,  // prod IUPAC-converted genome bytes from src (TLI)
    K_RC   = 5,  // reverse complement of the converted bytes [src, src+prod) (IV, reversed TLI)
    K_RAND = 6,  // prod random bases (mutator.py:466-471), a pure function of (seed, contig id, pos): base j of the
                 // insert at pos comes from Philox block j/64 — generated where it is consumed, never stored.
                 // src caches the first 64 bits of block 0 = bases 0..31 (2 bits each), so inserts of up to 32
                 // bases never touch Philox again
};

// One applied mutation.  32 bytes, sorted by (contig, pos).
// The walk of mutator.py:318-426 becomes: for each record copy input up to pos,
// emit `prod` payload bytes, skip `cons` input bytes, continue copying.
struct alignas(16) Rec {
    uint32_t pos;     // contig-relative start (the reference's dict key)
    uint32_t cons;    // input bases skipped at pos
    uint32_t prod;    // payload bytes produced at pos
    uint32_t out;     // contig-relative output base index of the payload (filled by the delta scan)
    int64_t  src;     // payload source: genome index (RAW/CONV/RC) or literal-pool offset (LIT)
    uint8_t  kind;    // Kind
    uint8_t  type;    // MutType (selects the VCF wording)
    uint8_t  ref;     // SN: converted reference base (VCF REF)
    uint8_t  alt;     // SN: substituted base (FASTA + VCF ALT)
    uint32_t contig;  // local contig index
};
static_assert(sizeof(Rec) == 32, "Rec must be 32 bytes");

// Per-contig geometry, device resident.
struct Contig {
    int64_t goff;       // index of base 0 in the genome array (16-byte aligned)
    int64_t len;        // input length L
    int64_t out_len;    // mutated length L'
    int64_t rec_lo;     // first record index
    int64_t rec_hi;     // one past the last record index
    int64_t hdr_off;    // file offset of '>' in the output FASTA image
    int64_t body_off;   // file offset of the first body byte
    int64_t body_bytes; // L' + floor(L'/bpl)
    int64_t blk_lo;     // first entry of this contig in the coarse block index
    int64_t piece_lo;   // first splice piece (tile) of this contig
    int64_t hdr_src;    // offset of the header text in the header blob
    int32_t hdr_len;    // header text length (without '>' and '\n')
    int32_t bpl;        // bases per line (pyfaidx lenc of the input record, mutator.py:133-134)
    int64_t name_src;   // offset of the contig name in the names blob
    int32_t name_len;
    uint32_t gid;       // global contig index in the FASTA (RNG key; independent of partitioning)
    uint32_t sep;       // 1 if a '\n' separator follows the body (partial last line, fasta_writer.py:44-45)
    uint32_t pad;
};

// What ms_load_records requires of record i of a table r (checked in this order): RF_OK or the first check it fails.
// src_end = end of the genome buffer (resident bases, pad and staging region) that K_RAW / K_CONV / K_RC sources index.
enum RecFault : int { RF_OK = 0, RF_CONTIG = 1, RF_ORDER = 2, RF_LIT = 3, RF_SRC = 4 };
MS_HD int rec_fault(const Rec* r, int64_t i, int32_t n_contigs, int64_t lit_bytes, int64_t src_end) {
    const Rec& x = r[i];
    if (x.contig >= (uint32_t)n_contigs) return RF_CONTIG;
    if (i && (x.contig < r[i - 1].contig || (x.contig == r[i - 1].contig && x.pos <= r[i - 1].pos))) return RF_ORDER;
    if (x.kind == K_LIT && (x.src < 0 || x.src + x.prod > lit_bytes)) return RF_LIT;
    if ((x.kind == K_RAW || x.kind == K_CONV || x.kind == K_RC) && (x.src < 0 || x.src + x.prod > src_end)) return RF_SRC;
    return RF_OK;
}

// mutator.py:75-77 as 256-entry tables.
struct Tables {
    uint8_t conv[256];   // non_ambiguous
    uint8_t comp[256];   // complement
    uint8_t trans[256];  // transitions
};

// per-record VCF line size arrays carry in bit 31 whether the record moves bases (goes to the SvRec stream) or is a SNP
constexpr uint32_t VSIZE_SV = 0x80000000u;

// first 32 bases of the random insert at `pos`, 2 bits each (what Rec.src caches for K_RAND)
MS_HD int64_t rand_insert_cache(Seed seed, uint32_t gid, uint32_t pos) {
    const U4 blk = draw(seed, gid, P_INSERT, pos);
    return (int64_t)u64_of(blk.x, blk.y);
}
MS_HD uint8_t cached_insert_base(int64_t cache, uint32_t j) { return (uint8_t)("ATGC"[((uint64_t)cache >> (2u * j)) & 3u]); }

// base j of the random insert at contig position `pos` (64 bases per Philox block, 2 bits each, "ATGC")
MS_HD uint8_t rand_insert_base(Seed seed, uint32_t gid, uint32_t pos, uint32_t j) {
    const U4 blk = draw(seed, gid, P_INSERT | ((j >> 6) << 8), pos);
    const uint32_t wsel = (j >> 4) & 3u;
    const uint32_t wv = wsel == 0 ? blk.x : wsel == 1 ? blk.y : wsel == 2 ? blk.z : blk.w;
    return (uint8_t)("ATGC"[(wv >> ((j & 15u) * 2u)) & 3u]);
}

inline void fill_tables(Tables& t) {
    for (int i = 0; i < 256; ++i) t.conv[i] = t.comp[i] = t.trans[i] = (uint8_t)i;
    const char* a = "KSYMWRBDHV-"; const char* b = "GCCAAACAAAN";
    for (int i = 0; a[i]; ++i) t.conv[(uint8_t)a[i]] = (uint8_t)b[i];
    const char* c = "ACGTUMRWSYKVHDB"; const char* d = "TGCAAKYWSRMBDHV";
    for (int i = 0; c[i]; ++i) t.comp[(uint8_t)c[i]] = (uint8_t)d[i];
    const char* e = "AGTC"; const char* f = "GACT";
    for (int i = 0; e[i]; ++i) t.trans[(uint8_t)e[i]] = (uint8_t)f[i];
}

// mutator.py:444-455 transversion pairs; letters outside ACGTN map to themselves
// (the reference raises KeyError there; SURVEY.md Q6).
MS_HD uint8_t transversion(uint8_t ref, uint32_t coin) {
    switch (ref) {
        case 'A': return coin ? 'C' : 'T';
        case 'G': return coin ? 'T' : 'C';
        case 'T': return coin ? 'A' : 'G';
        case 'C': return coin ? 'G' : 'A';
        default: return ref;
    }
}

// Blocks of the coarse index: entry k of a contig = number of that contig's
// records whose `out` is < k * BLK_BASES  (a lower bound for the record lookup).
constexpr int BLK_SHIFT = 8;
constexpr int64_t BLK_BASES = 1 << BLK_SHIFT;

}  // namespace ms
