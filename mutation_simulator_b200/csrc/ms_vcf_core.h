// ms_vcf_core.h — one VCF line per applied mutation (K7), host/device shared.
//
// Restates vcf_writer.py:44-52,118-126 and the per-type REF/ALT/POS/END/SVLEN
// rules of mutator.py:334-421.  The same templated emitter is instantiated with
// a counting sink (pass 1: sizes) and a writing sink (pass 2: bytes), so the two
// passes cannot disagree.
#pragma once
#include "ms_records.h"

namespace ms {

struct VcfView {
    const uint8_t* genome;
    const uint8_t* lit;
    const uint8_t* names;   // contig names blob
    const uint8_t* conv;
    const uint8_t* comp;
    Seed seed;              // for K_RAND payloads
};

struct CountSink {
    uint32_t n = 0;
    MS_HD void put(uint8_t) { ++n; }
    MS_HD void skip(uint32_t k) { n += k; }
    static constexpr bool counting = true;
};

struct WriteSink {
    uint8_t* p;
    MS_HD void put(uint8_t c) { *p++ = c; }
    MS_HD void skip(uint32_t) {}
    static constexpr bool counting = false;
};

MS_HD uint32_t ndigits(uint32_t v) {   // (a clz + power-of-ten table version was measured: its indexed constant loads cost k_vcf_write 5 %)
    return v < 10u ? 1u : v < 100u ? 2u : v < 1000u ? 3u : v < 10000u ? 4u : v < 100000u ? 5u : v < 1000000u ? 6u
         : v < 10000000u ? 7u : v < 100000000u ? 8u : v < 1000000000u ? 9u : 10u;
}

// every POS / END / SVLEN of this build is < 2^32 (contigs < 2^31 bases)
template <class S> MS_HD void put_uint(S& s, uint32_t v) {
    if constexpr (S::counting) s.skip(ndigits(v));
    else {
        char buf[10];
        int n = 0;
        do { const uint32_t q = v / 10u; buf[n++] = (char)('0' + (v - q * 10u)); v = q; } while (v);
        while (n) s.put((uint8_t)buf[--n]);
    }
}

template <class S> MS_HD void put_str(S& s, const char* t, int n) {
    if constexpr (S::counting) s.skip((uint32_t)n);
    else for (int i = 0; i < n; ++i) s.put((uint8_t)t[i]);
}

// n bytes of genome from g, optionally IUPAC-converted
template <class S> MS_HD void put_bases(S& s, const VcfView& v, int64_t g, uint32_t n, bool convert) {
    if constexpr (S::counting) s.skip(n);
    else for (uint32_t i = 0; i < n; ++i) { uint8_t c = v.genome[g + i]; s.put(convert ? v.conv[c] : c); }
}

// reverse complement of the converted bases [g, g+n)
template <class S> MS_HD void put_rc(S& s, const VcfView& v, int64_t g, uint32_t n) {
    if constexpr (S::counting) s.skip(n);
    else for (uint32_t i = 0; i < n; ++i) s.put(v.comp[v.conv[v.genome[g + (int64_t)(n - 1 - i)]]]);
}

// payload bytes of a record as the FASTA shows them (insert of IN / TLI)
template <class S> MS_HD void put_payload(S& s, const VcfView& v, const Rec& r, uint32_t gid = 0) {
    if constexpr (S::counting) { s.skip(r.prod); return; }
    else switch (r.kind) {
        case K_RAND:
            for (uint32_t i = 0; i < r.prod; ++i) s.put(i < 32u ? cached_insert_base(r.src, i) : rand_insert_base(v.seed, gid, r.pos, i));
            break;
        case K_LIT:  for (uint32_t i = 0; i < r.prod; ++i) s.put(v.lit[r.src + i]); break;
        case K_RAW:  put_bases(s, v, r.src, r.prod, false); break;
        case K_CONV: put_bases(s, v, r.src, r.prod, true); break;
        case K_RC:   put_rc(s, v, r.src, r.prod); break;
        default: break;
    }
}

// vcf_writer.py:123 — records with REF == ALT are not written.
MS_HD bool vcf_omitted(const VcfView& v, const Contig& c, const Rec& r) {
    switch (r.type) {
        case T_SN: return r.ref == r.alt;
        case T_IV: {  // REF == reverse complement of itself
            const int64_t g = c.goff + r.pos;
            for (uint32_t i = 0; i < r.cons; ++i)
                if (v.conv[v.genome[g + i]] != v.comp[v.conv[v.genome[g + (int64_t)(r.cons - 1 - i)]]]) return false;
            return true;
        }
        case T_DE: case T_TL:  // only a deletion of a whole 1-base contig degenerates to REF == ALT
            return r.pos == 0 && c.len == 1;
        case T_IT: case T_DEAD: return true;
        default: return false;
    }
}

template <class S> MS_HD void put_info(S& s, const char* sv, int svn, uint32_t end, uint32_t len) {
    put_str(s, "SVTYPE=", 7); put_str(s, sv, svn);
    put_str(s, ";END=", 5); put_uint(s, end);
    put_str(s, ";SVLEN=", 7); put_uint(s, len);
}

// the GT column of a haploid line (K7's)
struct HaploidGt {
    template <class S> MS_HD void operator()(S& s) const { put_str(s, "\tGT\t1\n", 6); }
};

// Emits the whole line (caller has checked vcf_omitted); gt writes everything from the tab before FORMAT on
// (ms_genotype_core.h's PhasedGt for a polyploid run).
template <class S, class Gt = HaploidGt> MS_HD void vcf_emit(S& s, const VcfView& v, const Contig& c, const Rec& r, Gt gt = Gt()) {
    const int64_t g0 = c.goff;
    const uint32_t p = r.pos;
    if constexpr (S::counting) s.skip((uint32_t)c.name_len);
    else for (int i = 0; i < c.name_len; ++i) s.put(v.names[c.name_src + i]);
    s.put('\t');
    const char* sv = ""; int svn = 0; uint32_t pos1 = 0, end = 0, svlen = 0;
    // POS first, REF/ALT below
    switch (r.type) {
        case T_SN: pos1 = p + 1; break;
        case T_IN: pos1 = p > 0 ? p : 1; end = pos1; svlen = r.prod; sv = "INS"; svn = 3; break;
        case T_TLI: pos1 = p > 0 ? p : 1; end = pos1; svlen = r.prod; sv = "INS:ME"; svn = 6; break;
        case T_DE: case T_TL:
            pos1 = p > 0 ? p : 1; end = p > 0 ? p + r.cons : r.cons + 1u; svlen = r.cons;
            if (r.type == T_DE) { sv = "DEL"; svn = 3; } else { sv = "DEL:ME"; svn = 6; }
            break;
        case T_IV: pos1 = p + 1; end = p + r.cons; svlen = 0; sv = "INV"; svn = 3; break;
        case T_DU: pos1 = p + 1; end = p + r.prod; svlen = r.prod; sv = "DUP"; svn = 3; break;
        default: break;
    }
    put_uint(s, pos1);
    put_str(s, "\t.\t", 3);
    switch (r.type) {
        case T_SN:  // mutator.py:334-341
            s.put(r.ref); s.put('\t'); s.put(r.alt);
            break;
        case T_IN: case T_TLI: {  // mutator.py:343-358, 401-421
            const uint8_t anchor = v.conv[v.genome[g0 + (p > 0 ? (int64_t)p - 1 : 0)]];
            s.put(anchor); s.put('\t');
            if (p > 0) { s.put(anchor); put_payload(s, v, r, c.gid); }
            else       { put_payload(s, v, r, c.gid); s.put(anchor); }
        } break;
        case T_DE: case T_TL: {  // mutator.py:360-377
            if (p > 0) {
                put_bases(s, v, g0 + (int64_t)p - 1, r.cons + 1, true); s.put('\t');
                s.put(v.conv[v.genome[g0 + (int64_t)p - 1]]);
            } else {
                uint64_t rl = (uint64_t)r.cons + 1;  // sequence[0:stop+2], truncated at the contig end
                if (rl > (uint64_t)c.len) rl = (uint64_t)c.len;
                put_bases(s, v, g0, (uint32_t)rl, true); s.put('\t');
                s.put(v.conv[v.genome[g0 + (int64_t)rl - 1]]);
            }
        } break;
        case T_IV:  // mutator.py:379-387
            put_bases(s, v, g0 + (int64_t)p, r.cons, true); s.put('\t');
            put_rc(s, v, g0 + (int64_t)p, r.cons);
            break;
        case T_DU:  // mutator.py:389-399 (raw bases)
            put_bases(s, v, g0 + (int64_t)p, r.prod, false); s.put('\t');
            put_bases(s, v, g0 + (int64_t)p, r.prod, false); put_bases(s, v, g0 + (int64_t)p, r.prod, false);
            break;
        default: break;
    }
    put_str(s, "\t.\t.\t", 5);
    if (r.type == T_SN) s.put('.'); else put_info(s, sv, svn, end, svlen);
    gt(s);
}

// Size of the line vcf_emit() writes, in closed form (the sampler sizes 40 M records per genome: running the
// emitter against a counting sink there cost a type switch with seven divergent bodies per record).
// tests/emu checks it against the emitter on every golden record.
MS_HD uint32_t vcf_line_len(const Contig& c, const Rec& r) {
    const uint32_t p = r.pos;
    uint32_t pos1, end = 0, svlen = 0, ref_len, alt_len, svn = 0;
    switch (r.type) {
        case T_SN:  pos1 = p + 1; ref_len = 1; alt_len = 1; break;
        case T_IN:  pos1 = p > 0 ? p : 1; end = pos1; svlen = r.prod; ref_len = 1; alt_len = 1 + r.prod; svn = 3; break;
        case T_TLI: pos1 = p > 0 ? p : 1; end = pos1; svlen = r.prod; ref_len = 1; alt_len = 1 + r.prod; svn = 6; break;
        case T_DE: case T_TL: {
            pos1 = p > 0 ? p : 1; end = p > 0 ? p + r.cons : r.cons + 1u; svlen = r.cons; svn = r.type == T_DE ? 3 : 6;
            uint64_t rl = (uint64_t)r.cons + 1;
            if (p == 0 && rl > (uint64_t)c.len) rl = (uint64_t)c.len;
            ref_len = (uint32_t)rl; alt_len = 1;
        } break;
        case T_IV:  pos1 = p + 1; end = p + r.cons; svlen = 0; ref_len = r.cons; alt_len = r.cons; svn = 3; break;
        case T_DU:  pos1 = p + 1; end = p + r.prod; svlen = r.prod; ref_len = r.prod; alt_len = 2 * r.prod; svn = 3; break;
        default:    return 0;
    }
    // name \t POS \t.\t REF \t ALT \t.\t.\t INFO \tGT\t1\n
    uint32_t n = (uint32_t)c.name_len + 1u + ndigits(pos1) + 3u + ref_len + 1u + alt_len + 5u + 6u;
    n += svn ? 7u + svn + 5u + ndigits(end) + 7u + ndigits(svlen) : 1u;
    return n;
}

MS_HD uint32_t vcf_line_size(const VcfView& v, const Contig& c, const Rec& r) {
    if (vcf_omitted(v, c, r)) return 0;
    return vcf_line_len(c, r);
}

// the same through the emitter (reference for the closed form above)
MS_HD uint32_t vcf_line_size_emitted(const VcfView& v, const Contig& c, const Rec& r) {
    if (vcf_omitted(v, c, r)) return 0;
    CountSink s;
    vcf_emit(s, v, c, r);
    return s.n;
}

// Line size if the record is written: an upper bound that does not look at the bases (the streamed run lays out
// the VCF buffer before the genome has arrived; whether a SNP / inversion has REF == ALT is decided later).
MS_HD uint32_t vcf_line_bound(const VcfView& v, const Contig& c, const Rec& r) {
    (void)v;
    if (r.type == T_IT || r.type == T_DEAD) return 0;
    if ((r.type == T_DE || r.type == T_TL) && r.pos == 0 && c.len == 1) return 0;
    return vcf_line_len(c, r);
}

}  // namespace ms
