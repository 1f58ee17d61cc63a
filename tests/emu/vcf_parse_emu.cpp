// Host build of ms_vcf_parse_core.h for tests/test_vcf_parse_core.py (g++, no CUDA): the steps of ms_load_vcf's
// kernels done one after the other — irregular bytes, line starts, one parse per line, compaction with the literal
// pool in file order, the one-block-per-contig check, and the placement of the blocks in contig order.
#include <stdint.h>
#include <string.h>
#include <vector>
#include "../../mutation_simulator_b200/csrc/ms_vcf_parse_core.h"

using namespace ms;
using namespace ms::vcfp;

extern "C" {

// names: blob with name_off[n_contigs + 1]; out: room for one record per line; lit: room for n bytes.
// Returns 1 (regular: out / lit hold the table) or 0 (irregular).
int vcf_parse(const uint8_t* t, int64_t n, const uint8_t* names, const int64_t* name_off, const int64_t* lens,
              int32_t n_contigs, int32_t skip_unknown, Rec* out, int64_t* n_recs, uint8_t* lit, int64_t* lit_bytes) {
    for (int64_t i = 0; i < n; ++i)
        if (irregular_byte(t[i])) return 0;
    std::vector<VcfContig> vc((size_t)n_contigs);
    int64_t goff = 0;
    for (int32_t i = 0; i < n_contigs; ++i) {
        vc[i] = VcfContig{name_off[i], goff, (int32_t)(name_off[i + 1] - name_off[i]), (int32_t)lens[i]};
        goff += lens[i];
    }
    const uint32_t size = table_size(n_contigs);
    std::vector<int32_t> slot(size);
    build_table(names, vc.data(), n_contigs, slot.data(), size);
    const NameTable nt{slot.data(), size - 1, names, vc.data()};

    std::vector<Rec> kept;
    int64_t pool = 0;
    for (int64_t lo = 0; lo < n;) {
        int64_t hi = lo;
        while (hi < n && t[hi] != '\n') ++hi;
        Rec r;
        const int k = parse_line(t, lo, hi, nt, skip_unknown, &r);
        if (k == VL_IRREGULAR) return 0;
        if (k == VL_REC) {
            if (r.kind == K_LIT) {
                memcpy(lit + pool, t + r.src, r.prod);
                r.src = pool;
                pool += r.prod;
            }
            kept.push_back(r);
        }
        lo = hi + 1;
    }
    std::vector<int64_t> first((size_t)n_contigs, 0), last((size_t)n_contigs, 0);
    std::vector<int32_t> blocks((size_t)n_contigs, 0);
    const int64_t m = (int64_t)kept.size();
    for (int64_t j = 0; j < m; ++j) {
        const uint32_t c = kept[j].contig;
        if (j == 0 || kept[j - 1].contig != c) {
            if (blocks[c]++) return 0;          // a contig in two blocks
            first[c] = j;
        } else if (kept[j].out <= kept[j - 1].out) {
            return 0;                            // POS not increasing
        }
        if (j == m - 1 || kept[j + 1].contig != c) last[c] = j + 1;
    }
    int64_t base = 0;
    for (int32_t c = 0; c < n_contigs; ++c) {
        for (int64_t j = first[c]; j < last[c]; ++j) {
            out[base + j - first[c]] = kept[j];
            out[base + j - first[c]].out = 0;
        }
        base += last[c] - first[c];
    }
    *n_recs = m;
    *lit_bytes = pool;
    return 1;
}

}  // extern "C"
