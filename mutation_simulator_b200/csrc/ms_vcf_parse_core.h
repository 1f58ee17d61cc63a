// ms_vcf_parse_core.h — one VCF line -> one splice descriptor (records.py:119-191 records_from_vcf), host/device
// shared: ms_vcf_parse.cu runs it one thread per line, tests/emu/vcf_parse_emu.cpp builds it with g++.
//
// Only the regular shape is parsed here: the lines VcfWriter.write emits (the reference's vcf_writer.py:118-126 and
// this package's k_vcf_write).  Anything else makes the line IRREGULAR and the whole text goes to the host parser,
// which owns the error messages:
//   - the text holds none of '\r' '\x0b' '\x0c' '\x1c' '\x1d' '\x1e' '\x85' (str.splitlines() breaks lines there);
//   - empty lines and lines starting with '#' are skipped;
//   - every other line has >= 8 tab-separated fields, POS is ASCII digits;
//   - INFO is '.' (single-base REF and ALT) or exactly SVTYPE=<INS|DEL|INV|DUP|DEL:ME|INS:ME>;END=<digits>;SVLEN=<digits>;
//   - INS / DEL anchoring as records_from_vcf reads it, every record inside its contig.
#pragma once
#include <stdint.h>
#include "ms_records.h"

namespace ms {
namespace vcfp {

// per contig: where its CHROM name lies in the names blob, and its genome geometry
struct VcfContig {
    int64_t name_off;
    int64_t goff;
    int32_t name_len;
    int32_t len;
};

// CHROM -> local contig index: open addressing over a power-of-two table of contig indices (-1 = empty)
struct NameTable {
    const int32_t* slot;
    uint32_t mask;
    const uint8_t* names;
    const VcfContig* contig;
};

enum LineKind : int { VL_SKIP = 0, VL_REC = 1, VL_IRREGULAR = 2 };

// a byte str.splitlines() treats as a line break besides '\n' (the text is decoded as latin-1)
MS_HD bool irregular_byte(uint8_t b) {
    return b == '\r' || b == 0x0b || b == 0x0c || b == 0x1c || b == 0x1d || b == 0x1e || b == 0x85;
}

MS_HD uint32_t name_hash(const uint8_t* p, int64_t n) {
    uint32_t h = 2166136261u;                          // FNV-1a
    for (int64_t i = 0; i < n; ++i) h = (h ^ p[i]) * 16777619u;
    return h;
}

MS_HD int32_t find_contig(const NameTable& t, const uint8_t* p, int64_t n) {
    for (uint32_t s = name_hash(p, n) & t.mask;; s = (s + 1) & t.mask) {
        const int32_t ci = t.slot[s];
        if (ci < 0) return -1;
        const VcfContig& k = t.contig[ci];
        if (k.name_len != n) continue;
        bool eq = true;
        for (int64_t i = 0; i < n && eq; ++i) eq = t.names[k.name_off + i] == p[i];
        if (eq) return ci;
    }
}

// slot count for n contigs (load factor <= 1/2)
inline uint32_t table_size(int32_t n) {
    uint32_t s = 16;
    while (s < 2u * (uint32_t)n) s <<= 1;
    return s;
}

// Fills slot[table_size(n)].  A name given twice maps to its last contig, like the dict records_from_vcf builds.
inline void build_table(const uint8_t* names, const VcfContig* contig, int32_t n, int32_t* slot, uint32_t size) {
    for (uint32_t s = 0; s < size; ++s) slot[s] = -1;
    const NameTable t{slot, size - 1, names, contig};
    for (int32_t ci = 0; ci < n; ++ci) {
        const uint8_t* p = names + contig[ci].name_off;
        const int32_t have = find_contig(t, p, contig[ci].name_len);
        uint32_t s = name_hash(p, contig[ci].name_len) & t.mask;
        if (have >= 0) while (slot[s] != have) s = (s + 1) & t.mask;
        else while (slot[s] >= 0) s = (s + 1) & t.mask;
        slot[s] = ci;
    }
}

constexpr uint64_t NUM_CAP = 1ull << 40;   // digits saturate here: far beyond any contig length (< 2^31)

// ASCII digits [lo, hi) -> value (saturated at NUM_CAP); false when empty or anything else is there
MS_HD bool parse_digits(const uint8_t* t, int64_t lo, int64_t hi, uint64_t* v) {
    if (lo >= hi) return false;
    uint64_t x = 0;
    for (int64_t i = lo; i < hi; ++i) {
        const uint32_t d = (uint32_t)t[i] - '0';
        if (d > 9) return false;
        x = x * 10 + d;
        if (x > NUM_CAP) x = NUM_CAP;
    }
    *v = x;
    return true;
}

MS_HD bool same_bytes(const uint8_t* t, int64_t a, int64_t b, int64_t n) {
    for (int64_t i = 0; i < n; ++i)
        if (t[a + i] != t[b + i]) return false;
    return true;
}

// bytes [lo, hi) of t == the NUL-terminated word w
MS_HD bool is_word(const uint8_t* t, int64_t lo, int64_t hi, const char* w) {
    int64_t i = 0;
    for (; w[i]; ++i)
        if (lo + i >= hi || t[lo + i] != (uint8_t)w[i]) return false;
    return lo + i == hi;
}

// Line [lo, hi) of t (without its '\n') -> LineKind.  For VL_REC, *out is the record records_from_vcf builds, except
// that out->out holds POS (the block order check needs it) and, for K_LIT, out->src is the text offset of the inserted
// bytes (their pool offset comes from a scan over the literal lengths in file order).
MS_HD int parse_line(const uint8_t* t, int64_t lo, int64_t hi, const NameTable& names, int skip_unknown, Rec* out) {
    if (lo >= hi || t[lo] == '#') return VL_SKIP;
    int64_t f[9];                       // f[k] = start of field k, f[k+1] - 1 = its end (fields 0..7)
    f[0] = lo;
    int nf = 1;
    for (int64_t i = lo; i < hi && nf < 9; ++i)
        if (t[i] == '\t') f[nf++] = i + 1;
    if (nf < 8) return VL_IRREGULAR;    // "expected at least 8 tab-separated fields"
    int64_t info_hi = hi;               // INFO ends at the next tab or the end of the line
    if (nf == 9) info_hi = f[8] - 1;
    const int32_t ci = find_contig(names, t + f[0], f[1] - 1 - f[0]);
    if (ci < 0) return skip_unknown ? VL_SKIP : VL_IRREGULAR;
    const VcfContig k = names.contig[ci];
    const int64_t L = k.len;
    uint64_t pos1u;
    if (!parse_digits(t, f[1], f[2] - 1, &pos1u)) return VL_IRREGULAR;
    const int64_t pos1 = (int64_t)pos1u;
    const int64_t r0 = f[3], lr = f[4] - 1 - f[3];
    const int64_t a0 = f[4], la = f[5] - 1 - f[4];
    const int64_t i0 = f[7];
    if (la >= 0x7FFFFFFF || lr >= 0x7FFFFFFF) return VL_IRREGULAR;
    Rec r{};
    r.contig = (uint32_t)ci;
    r.out = (uint32_t)(pos1 < 0x7FFFFFFF ? pos1 : 0x7FFFFFFF);
    if (info_hi - i0 == 1 && t[i0] == '.') {
        if (lr != 1 || la != 1 || pos1 < 1 || pos1 > L) return VL_IRREGULAR;
        r.pos = (uint32_t)(pos1 - 1); r.cons = 1; r.prod = 1; r.kind = K_SNP; r.type = T_SN;
        r.ref = t[r0]; r.alt = t[a0];
        *out = r;
        return VL_REC;
    }
    // SVTYPE=<type>;END=<digits>;SVLEN=<digits>
    if (!is_word(t, i0, i0 + 7 < info_hi ? i0 + 7 : info_hi, "SVTYPE=")) return VL_IRREGULAR;
    int64_t s1 = i0 + 7;
    while (s1 < info_hi && t[s1] != ';') ++s1;
    int type;
    if (is_word(t, i0 + 7, s1, "INS")) type = T_IN;
    else if (is_word(t, i0 + 7, s1, "DEL")) type = T_DE;
    else if (is_word(t, i0 + 7, s1, "INV")) type = T_IV;
    else if (is_word(t, i0 + 7, s1, "DUP")) type = T_DU;
    else if (is_word(t, i0 + 7, s1, "DEL:ME")) type = T_TL;
    else if (is_word(t, i0 + 7, s1, "INS:ME")) type = T_TLI;
    else return VL_IRREGULAR;
    if (s1 + 5 > info_hi || !is_word(t, s1, s1 + 5, ";END=")) return VL_IRREGULAR;
    int64_t s2 = s1 + 5;
    while (s2 < info_hi && t[s2] != ';') ++s2;
    uint64_t end_v, svlen;
    if (!parse_digits(t, s1 + 5, s2, &end_v)) return VL_IRREGULAR;
    if (s2 + 7 > info_hi || !is_word(t, s2, s2 + 7, ";SVLEN=")) return VL_IRREGULAR;
    if (!parse_digits(t, s2 + 7, info_hi, &svlen)) return VL_IRREGULAR;
    r.type = (uint8_t)type;
    int64_t pos, cons = 0, prod = 0;
    if (type == T_IN || type == T_TLI) {
        // ALT = REF + insert (POS = pos), or insert + REF at POS 1 (pos 0)
        if (la >= lr && same_bytes(t, a0, r0, lr)) { pos = pos1; prod = la - lr; r.src = a0 + lr; }
        else if (la >= lr && pos1 == 1 && same_bytes(t, a0 + la - lr, r0, lr)) { pos = 0; prod = la - lr; r.src = a0; }
        else return VL_IRREGULAR;
        r.kind = K_LIT;
    } else if (type == T_DE || type == T_TL) {
        // ALT = REF[:1] (POS = pos), or REF[-1:] at POS 1 (pos 0)
        if (la == (lr > 0 ? 1 : 0) && (lr == 0 || t[a0] == t[r0])) pos = pos1;
        else if (la == 1 && lr > 0 && pos1 == 1 && t[a0] == t[r0 + lr - 1]) pos = 0;
        else return VL_IRREGULAR;
        if (pos >= L) return VL_IRREGULAR;
        cons = (int64_t)svlen < L - pos ? (int64_t)svlen : L - pos;
        r.kind = K_NONE;
    } else {
        pos = pos1 - 1;
        if (pos < 0 || pos >= L) return VL_IRREGULAR;
        if (type == T_IV) { cons = lr; prod = lr; r.kind = K_RC; }
        else { prod = lr; r.kind = K_RAW; }
        r.src = k.goff + pos;
    }
    if (pos < 0 || pos >= L || pos + cons > L) return VL_IRREGULAR;   // "record outside contig"
    r.pos = (uint32_t)pos; r.cons = (uint32_t)cons; r.prod = (uint32_t)prod;
    *out = r;
    return VL_REC;
}

}  // namespace vcfp
}  // namespace ms
