// ms_genotype_core.h — the genotype of each record in a polyploid run (--ploidy), host/device shared: ms_genotype.cu runs
// it on the device, tests/emu/genotype_emu.cpp builds it with g++.
//
// Every record of the (haploid) table gets a haplotype mask m: bit h-1 set = haplotype h carries the record.
//   blk = draw(seed, gid, P_GENOTYPE, key)   key = r.pos, or for a TLI its TL's position (r.src - goff), so that both
//                                              halves of a translocation land on the same haplotypes
//   homozygous (m = 2^P - 1)  iff  blk.x < thr,  thr = min(2^32, llround(F * 2^32))
//   else m = 1 + mulhi(blk.y, 2^P - 2): uniform over the masks that are neither empty nor full
// The phased VCF line is the haploid line with GT = the P alleles of haplotypes 1..P joined by '|'.
#pragma once
#include <math.h>
#include "ms_vcf_core.h"

namespace ms {

constexpr int MAX_PLOIDY = 8;

// F in [0, 1] -> the threshold on blk.x (host side; 2^32 makes every record homozygous)
inline uint64_t hom_threshold(double f) {
    const long long t = llround(f * 4294967296.0);
    return t > (1ll << 32) ? (1ull << 32) : (uint64_t)t;
}

MS_HD uint32_t genotype_key(const Contig& c, const Rec& r) {
    return r.type == T_TLI ? (uint32_t)(r.src - c.goff) : r.pos;
}

MS_HD uint8_t genotype_mask(Seed seed, uint32_t gid, uint32_t key, int ploidy, uint64_t thr) {
    const U4 blk = draw(seed, gid, P_GENOTYPE, key);
    const uint32_t full = (1u << ploidy) - 1u;
    if ((uint64_t)blk.x < thr) return (uint8_t)full;
    return (uint8_t)(1u + mulhi32(blk.y, full - 1u));
}

// GT tail of a phased line: "\tGT\t" a|b|...\n
struct PhasedGt {
    uint32_t mask;
    int32_t ploidy;
    template <class S> MS_HD void operator()(S& s) const {
        put_str(s, "\tGT\t", 4);
        for (int h = 0; h < ploidy; ++h) {
            if (h) s.put('|');
            s.put((mask >> h) & 1u ? '1' : '0');
        }
        s.put('\n');
    }
};

// the phased line is the haploid one with 2 (P - 1) more bytes of GT; 0 when the record writes no line
MS_HD uint32_t phased_line_size(const VcfView& v, const Contig& c, const Rec& r, int ploidy) {
    const uint32_t n = vcf_line_size(v, c, r);
    return n ? n + 2u * (uint32_t)(ploidy - 1) : 0u;
}

}  // namespace ms
