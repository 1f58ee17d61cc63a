// Host build of ms_reads_core.h for tests/test_reads_core.py and tests/test_gpu_reads.py (g++, no CUDA): the pairs
// k_reads_size draws and the records k_reads_write formats, for one contig at a time.
#include <stdint.h>
#include "../../mutation_simulator_b200/csrc/ms_reads_core.h"

using namespace ms;

extern "C" {

// Pairs [first, first + n) of one contig whose mutated bases are img[body_off + q + q / bpl] (Lp of them), with gid and
// name, and whose records (out filled in) are recs[0, n_recs).  R1 records go to out1, R2 records to out2 (each at
// least the returned size); info receives 6 int64 per pair: s, f, strand, attempt, lift1, lift2.  Returns the bytes of
// one file, or -1 if the counting and writing sinks disagree.
int64_t reads_emu(const uint8_t* img, int64_t body_off, int32_t bpl, int64_t Lp, const uint8_t* name, int32_t name_len,
                  uint32_t gid, const Rec* recs, int64_t n_recs, uint64_t seed, int32_t hap, int32_t L, int32_t M, int32_t S,
                  double E, uint8_t qual, int64_t first, int64_t n, uint8_t* out1, uint8_t* out2, int64_t* info) {
    Contig k{};
    k.body_off = body_off; k.bpl = bpl; k.out_len = Lp; k.len = Lp; k.gid = gid;
    k.rec_lo = 0; k.rec_hi = n_recs; k.name_src = 0; k.name_len = name_len;
    Tables tab; fill_tables(tab);
    const ReadsCfg g{make_seed(seed), (uint32_t)hap, L, M, S, read_error_threshold(E), qual};
    int64_t o = 0;
    for (int64_t j = 0; j < n; ++j) {
        const uint32_t i = (uint32_t)(first + j);
        PairInfo p = pair_info(g, img, recs, k, i);
        p.size = read_record_size(k, g.hap, i, p, L);
        int64_t* x = info + 6 * j;
        x[0] = p.s; x[1] = p.f; x[2] = p.meta & 1u; x[3] = p.meta >> 1; x[4] = p.lift1; x[5] = p.lift2;
        for (int mate = 1; mate <= 2; ++mate) {
            uint8_t* base = (mate == 1 ? out1 : out2) + o;
            WriteSink w{base};
            read_record(w, g, img, tab.comp, name, k, i, p, mate);
            CountSink c;
            read_record(c, g, img, tab.comp, name, k, i, p, mate);
            if (w.p - base != (int64_t)p.size || c.n != p.size) return -1;
        }
        o += p.size;
    }
    return o;
}

// lift of mutated positions q[0, n) along recs[0, n_recs) (out filled in); -1 = '*'
void lift_emu(const Rec* recs, int64_t n_recs, const int64_t* q, int64_t n, int64_t* out) {
    Contig k{};
    k.rec_lo = 0; k.rec_hi = n_recs;
    for (int64_t j = 0; j < n; ++j) out[j] = read_lift(recs, k, q[j]);
}

}  // extern "C"
