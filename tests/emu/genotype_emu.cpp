// Host build of ms_genotype_core.h (and the GT parse of ms_vcf_parse_core.h) for tests/test_genotype_core.py (g++, no
// CUDA): the masks k_genotype draws, the phased lines K7p writes and their closed-form size, one record at a time.
#include <stdint.h>
#include <vector>
#include "../../mutation_simulator_b200/csrc/ms_genotype_core.h"
#include "../../mutation_simulator_b200/csrc/ms_vcf_parse_core.h"

using namespace ms;

static std::vector<Contig> contigs(const int64_t* lens, int32_t n, const int64_t* name_off) {
    std::vector<Contig> k((size_t)n);
    int64_t goff = 0;
    for (int32_t c = 0; c < n; ++c) {
        k[c] = Contig{};
        k[c].goff = goff; k[c].len = lens[c]; k[c].out_len = lens[c]; k[c].gid = (uint32_t)c;
        if (name_off) { k[c].name_src = name_off[c]; k[c].name_len = (int32_t)(name_off[c + 1] - name_off[c]); }
        goff += lens[c];
    }
    return k;
}

extern "C" {

// masks of a table whose contig c holds lens[c] bases at genome index sum(lens[:c]) and has gid c
void genotype_emu(const Rec* recs, int64_t n, const int64_t* lens, int32_t n_contigs, uint64_t seed, int32_t ploidy,
                  double hom_fraction, uint8_t* mask) {
    const std::vector<Contig> k = contigs(lens, n_contigs, nullptr);
    const uint64_t thr = hom_threshold(hom_fraction);
    for (int64_t i = 0; i < n; ++i) {
        const Contig& c = k[recs[i].contig];
        mask[i] = genotype_mask(make_seed(seed), c.gid, genotype_key(c, recs[i]), ploidy, thr);
    }
}

// Line of record i: ploidy 0 = the haploid emitter (vcf_emit's default tail), else the phased one with `mask`.
// Returns the emitted size (0 when omitted); *closed gets vcf_line_size / phased_line_size.  Returns -1 if the
// counting and writing sinks disagree.
int64_t phased_line_emu(const uint8_t* genome, const int64_t* lens, int32_t n_contigs, const uint8_t* names,
                        const int64_t* name_off, const uint8_t* lit, const Rec* recs, int64_t i, int32_t ploidy,
                        uint32_t mask, uint8_t* out, int64_t* closed) {
    const std::vector<Contig> k = contigs(lens, n_contigs, name_off);
    Tables tab; fill_tables(tab);
    const VcfView v{genome, lit, names, tab.conv, tab.comp, Seed{0, 0}};
    const Contig& c = k[recs[i].contig];
    const Rec& r = recs[i];
    *closed = ploidy ? phased_line_size(v, c, r, ploidy) : vcf_line_size(v, c, r);
    if (vcf_omitted(v, c, r)) return 0;
    CountSink cs;
    WriteSink ws{out};
    if (ploidy) { vcf_emit(cs, v, c, r, PhasedGt{mask, ploidy}); vcf_emit(ws, v, c, r, PhasedGt{mask, ploidy}); }
    else { vcf_emit(cs, v, c, r); vcf_emit(ws, v, c, r); }
    if ((int64_t)cs.n != ws.p - out) return -1;
    return cs.n;
}

// the device parser's GT check of one line [0, n): 1 and *mask, or 0 (irregular)
int32_t parse_gt_emu(const uint8_t* line, int64_t n, int32_t ploidy, uint8_t* mask) {
    return vcfp::parse_gt(line, 0, n, ploidy, mask) ? 1 : 0;
}

}  // extern "C"
