// ms_chain_core.h — UCSC chain text from the input genome to the mutated genome (K8), host/device shared.
//
// The SvRec stream of the plan pass is the list of copy runs: between two base-moving records the output is one
// shifted copy of the input, so a chain's aligned blocks are those runs, and every DU / IV / TLI payload copied out
// of the contig is one more single-block chain.  The text is cut into work items, per contig in FASTA order:
//   item 0             the primary chain's header (nothing when the contig has no block)
//   items 1 .. k+1     run j = item - 1: one block line, or nothing when the run is empty or continues a block
//   items k+2 .. 2k+1  the copy chain of SvRec item - k - 2 (nothing when the record copies nothing)
// with k the contig's SvRecs; contig c's items start at 2 * (its first SvRec slot) + 2c.  The same templated emitter
// runs with a counting sink (sizes) and a writing sink (bytes), so the two passes cannot disagree.
//
// A record with cons = prod = 0 (an unpaired translocation half left in the table as a no-op) moves no base: it
// neither ends a block nor starts one.  Line layout follows kent's chainWrite: header fields separated by spaces,
// block fields by tabs, the last block line holds its size only, and every chain ends with an empty line.
#pragma once
#include "ms_tile_core.h"
#include "ms_vcf_core.h"

namespace ms {

// Per-contig summary built by ms_chain_count (k_chain_contigs, the copy scan, k_chain_finish).
struct alignas(16) ChainCtg {
    int64_t n_lo, n_hi;        // the contig's SvRec slots [n_lo, n_hi)
    int64_t item_lo;           // first work item: 2 * n_lo + 2 * contig
    int64_t first_id;          // id of the contig's first chain (ms_chain_write)
    uint32_t score;            // L - sum of cons = sum of the block sizes
    uint32_t t0, q0, t1, q1;   // start of the first block, end of the last block
    uint32_t primary;          // 1 if the contig has a block
    uint32_t n_copies;
    uint32_t pad;
};
static_assert(sizeof(ChainCtg) == 64, "ChainCtg layout");

struct ChainView {
    const SvRec* sv;
    const Contig* contigs;
    const uint8_t* names;
    const ChainCtg* cc;
    const uint32_t* copy_pre;   // copy_pre[i]: copy records in slots [0, i)
    int32_t n_contigs;
};

MS_HD bool chain_null(const SvRec& r) { return r.run_in == r.pos && r.prod == 0u; }
MS_HD bool chain_copy(const SvRec& r) { return (r.kind == K_RAW || r.kind == K_CONV || r.kind == K_RC) && r.prod > 0u; }

// first slot in [i, n_hi) that moves bases, or n_hi
MS_HD int64_t chain_next_real(const SvRec* sv, int64_t i, int64_t n_hi) {
    while (i < n_hi && chain_null(sv[i])) ++i;
    return i;
}

// The run after slot m (m = n_lo - 1: run 0): start (ts, qs), end (te, qe) at the next record that moves bases (slot
// e) or at the contig end (e = n_hi).
struct ChainRun { uint32_t ts, qs, te, qe; int64_t e; };
MS_HD ChainRun chain_run(const SvRec* sv, const Contig& k, int64_t n_lo, int64_t n_hi, int64_t m) {
    ChainRun r;
    if (m < n_lo) { r.ts = 0u; r.qs = 0u; }
    else { const SvRec& x = sv[m]; r.ts = x.run_in; r.qs = x.out + x.prod; }
    r.e = chain_next_real(sv, m + 1, n_hi);
    if (r.e < n_hi) { r.te = sv[r.e].pos; r.qe = sv[r.e].out; }
    else { r.te = (uint32_t)k.len; r.qe = (uint32_t)k.out_len; }
    return r;
}

// First and last block of a contig (two short walks over the empty runs at its ends).
MS_HD void chain_bounds(const SvRec* sv, const Contig& k, ChainCtg& cc) {
    const int64_t n_lo = cc.n_lo, n_hi = cc.n_hi;
    cc.primary = 0u; cc.t0 = cc.q0 = cc.t1 = cc.q1 = 0u;
    for (int64_t m = n_lo - 1;;) {
        const ChainRun r = chain_run(sv, k, n_lo, n_hi, m);
        if (r.te > r.ts) { cc.primary = 1u; cc.t0 = r.ts; cc.q0 = r.qs; break; }
        if (r.e >= n_hi) return;                      // no block at all
        m = r.e;
    }
    for (int64_t e = n_hi;;) {                        // e: the record (or contig end) that ends the candidate run
        int64_t m = e - 1;
        while (m >= n_lo && chain_null(sv[m])) --m;
        const uint32_t ts = m >= n_lo ? sv[m].run_in : 0u;
        const uint32_t te = e < n_hi ? sv[e].pos : (uint32_t)k.len;
        if (te > ts) { cc.t1 = te; cc.q1 = e < n_hi ? sv[e].out : (uint32_t)k.out_len; return; }
        e = m;                                        // m >= n_lo here: run 0 is not empty when a block exists
    }
}

template <class S> MS_HD void chain_name(S& s, const ChainView& v, const Contig& k) {
    if constexpr (S::counting) s.skip((uint32_t)k.name_len);
    else for (int i = 0; i < k.name_len; ++i) s.put(v.names[k.name_src + i]);
}

// "chain score tName tSize + tStart tEnd qName qSize qStrand qStart qEnd id\n"
template <class S>
MS_HD void chain_header(S& s, const ChainView& v, const Contig& k, uint32_t score, uint32_t t0, uint32_t t1, uint8_t strand,
                        uint32_t q0, uint32_t q1, uint32_t id) {
    put_str(s, "chain ", 6); put_uint(s, score); s.put(' ');
    chain_name(s, v, k); s.put(' '); put_uint(s, (uint32_t)k.len); put_str(s, " + ", 3);
    put_uint(s, t0); s.put(' '); put_uint(s, t1); s.put(' ');
    chain_name(s, v, k); s.put(' '); put_uint(s, (uint32_t)k.out_len); s.put(' '); s.put(strand); s.put(' ');
    put_uint(s, q0); s.put(' '); put_uint(s, q1); s.put(' '); put_uint(s, id); s.put('\n');
}

// The block line of run j (the run after slot n_lo + j - 1).
template <class S> MS_HD void chain_block(S& s, const SvRec* sv, const Contig& k, int64_t n_lo, int64_t n_hi, int64_t j) {
    const int64_t m = n_lo + j - 1;
    if (j > 0 && chain_null(sv[m])) return;           // continues the block before the no-op record
    const ChainRun r = chain_run(sv, k, n_lo, n_hi, m);
    if (r.te == r.ts) return;                         // empty run: its gaps add into the neighbouring blocks' gap
    put_uint(s, r.te - r.ts);
    for (int64_t x = r.e; x < n_hi;) {                // the next non-empty run
        const ChainRun n = chain_run(sv, k, n_lo, n_hi, x);
        if (n.te > n.ts) {
            s.put('\t'); put_uint(s, n.ts - r.te); s.put('\t'); put_uint(s, n.qs - r.qe); s.put('\n');
            return;
        }
        x = n.e;
    }
    put_str(s, "\n\n", 2);                            // the last block
}

// The single-block chain of a copy record (DU, IV, TLI payloads).
template <class S> MS_HD void chain_copy_item(S& s, const ChainView& v, const Contig& k, const ChainCtg& cc, int64_t i) {
    const SvRec r = v.sv[i];
    if (!chain_copy(r)) return;
    const uint32_t src = (uint32_t)(r.src - k.goff);  // inside the contig: checked by ms_chain_count
    const uint32_t id = (uint32_t)(cc.first_id + cc.primary + (int64_t)(v.copy_pre[i] - v.copy_pre[cc.n_lo]));
    const bool rc = r.kind == K_RC;
    const uint32_t q0 = rc ? (uint32_t)k.out_len - r.out - r.prod : r.out;
    chain_header(s, v, k, r.prod, src, src + r.prod, rc ? (uint8_t)'-' : (uint8_t)'+', q0, q0 + r.prod, id);
    put_uint(s, r.prod);
    put_str(s, "\n\n", 2);
}

// contig of work item x: the last c with item_lo <= x
MS_HD int32_t chain_item_contig(const ChainCtg* cc, int32_t n_contigs, int64_t x) {
    int32_t lo = 0, hi = n_contigs;
    while (hi - lo > 1) { const int32_t mid = (lo + hi) >> 1; if (cc[mid].item_lo <= x) lo = mid; else hi = mid; }
    return lo;
}

// Work item x (of contig c) into the sink.
template <class S> MS_HD void chain_item(S& s, const ChainView& v, int32_t c, int64_t x) {
    const ChainCtg& cc = v.cc[c];
    const Contig& k = v.contigs[c];
    const int64_t l = x - cc.item_lo, n = cc.n_hi - cc.n_lo;
    if (l == 0) {
        if (cc.primary) chain_header(s, v, k, cc.score, cc.t0, cc.t1, (uint8_t)'+', cc.q0, cc.q1, (uint32_t)cc.first_id);
    } else if (l <= n + 1) {
        chain_block(s, v.sv, k, cc.n_lo, cc.n_hi, l - 1);
    } else {
        chain_copy_item(s, v, k, cc, cc.n_lo + (l - n - 2));
    }
}

MS_HD uint32_t chain_item_size(const ChainView& v, int32_t c, int64_t x) {
    CountSink s;
    chain_item(s, v, c, x);
    return s.n;
}

}  // namespace ms
