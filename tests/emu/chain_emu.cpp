// Host build of ms_chain_core.h for tests/test_chain_core.py (g++, no CUDA): the steps of ms_chain_count /
// ms_chain_write done one after the other — the SvRec stream and contig lengths the plan pass builds, the per-contig
// summary, the copy numbering, the source check, and every work item sized and then written.
#include <stdint.h>
#include <vector>
#include "../../mutation_simulator_b200/csrc/ms_chain_core.h"

using namespace ms;

extern "C" {

// recs: the table ms_load_records takes (sorted by (contig, pos)); contig c holds lens[c] bases at genome index
// sum(lens[:c]); names blob with name_off[n_contigs + 1].  first_id NULL: ids 1, 2, ... through the file.
// Fills n_chains[n_contigs] and chain_off[n_contigs + 1]; out (NULL: size query) receives the text.
// Returns the text size, or -1 - slot of the first copy record whose source leaves its contig.
int64_t chain_emu(const Rec* recs, int64_t n_recs, const int64_t* lens, int32_t n_contigs, const uint8_t* names,
                  const int64_t* name_off, const int64_t* first_id, int64_t* n_chains, uint8_t* out, int64_t* chain_off) {
    std::vector<Contig> k((size_t)n_contigs);
    int64_t goff = 0;
    for (int32_t c = 0; c < n_contigs; ++c) {
        k[c] = Contig{};
        k[c].goff = goff; k[c].len = lens[c]; k[c].out_len = lens[c];
        k[c].name_src = name_off[c]; k[c].name_len = (int32_t)(name_off[c + 1] - name_off[c]);
        goff += lens[c];
    }
    std::vector<SvRec> sv;
    std::vector<ChainCtg> cc((size_t)n_contigs);
    int64_t i = 0;
    for (int32_t c = 0; c < n_contigs; ++c) {
        cc[c].n_lo = (int64_t)sv.size();
        int64_t shift = 0;
        for (; i < n_recs && recs[i].contig == (uint32_t)c; ++i) {
            const Rec& r = recs[i];
            if (r.kind != K_SNP)
                sv.push_back(SvRec{(uint32_t)(r.pos + shift), r.prod, r.pos + r.cons, r.pos, r.src, (uint32_t)r.kind, 0u});
            shift += (int64_t)r.prod - (int64_t)r.cons;
        }
        cc[c].n_hi = (int64_t)sv.size();
        k[c].out_len = lens[c] + shift;
    }
    const int64_t n_sv = (int64_t)sv.size();
    sv.push_back(SvRec{});                             // keeps sv.data() valid for an empty stream
    std::vector<uint32_t> copy_pre((size_t)n_sv + 1, 0u);
    for (int64_t s = 0; s < n_sv; ++s) copy_pre[s + 1] = copy_pre[s] + (chain_copy(sv[s]) ? 1u : 0u);
    int64_t next_id = 1;
    for (int32_t c = 0; c < n_contigs; ++c) {
        ChainCtg& x = cc[c];
        x.item_lo = 2 * x.n_lo + 2 * (int64_t)c;
        chain_bounds(sv.data(), k[c], x);
        int64_t cons = 0;
        for (int64_t s = x.n_lo; s < x.n_hi; ++s) {
            cons += sv[s].run_in - sv[s].pos;
            if (chain_copy(sv[s])) {
                const int64_t src = sv[s].src - k[c].goff;
                if (src < 0 || src + (int64_t)sv[s].prod > k[c].len) return -1 - s;
            }
        }
        x.score = (uint32_t)(k[c].len - cons);
        x.n_copies = copy_pre[x.n_hi] - copy_pre[x.n_lo];
        n_chains[c] = (int64_t)x.primary + x.n_copies;
        x.first_id = first_id ? first_id[c] : next_id;
        next_id += n_chains[c];
    }
    const ChainView v{sv.data(), k.data(), names, cc.data(), copy_pre.data(), n_contigs};
    const int64_t n_items = 2 * n_sv + 2 * (int64_t)n_contigs;
    int64_t total = 0;
    for (int64_t x = 0; x < n_items; ++x) {
        const int32_t c = chain_item_contig(cc.data(), n_contigs, x);
        if (x == cc[c].item_lo) chain_off[c] = total;
        const uint32_t n = chain_item_size(v, c, x);
        if (out && n) {
            WriteSink s{out + total};
            chain_item(s, v, c, x);
            if (s.p != out + total + n) return -1 - n_sv - x;     // the two sinks disagree
        }
        total += n;
    }
    chain_off[n_contigs] = total;
    return total;
}

}  // extern "C"
