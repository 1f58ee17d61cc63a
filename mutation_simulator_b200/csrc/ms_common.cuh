// ms_common.cuh — context, device buffers and error plumbing of libmutsim_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include "ms_records.h"
#include "ms_sample_core.h"
#include "ms_tile_core.h"
#include "ms_chain_core.h"
#include "ms_reads_core.h"
#include "../../include/mutsim_b200.h"

namespace ms {

constexpr int NUM_SMS_B200 = 148;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
    // grow-only; contents are NOT preserved
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = want;
        return cudaSuccess;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// Device-side scalars a pipeline produces and the host needs (one small D2H copy).
struct Totals {
    int64_t fasta_bytes;
    int64_t vcf_bytes;
    int64_t n_blk;        // (number of SvRecs of the last plan)
    int64_t n_pieces;
    int64_t n_recs;       // records after sampling / linking
    int64_t lit_bytes;
    int64_t n_candidates;
    int64_t n_accepted;
    int64_t error;        // first error code raised by a kernel (0 = none)
    int64_t error_arg;
    int64_t n_long_gaps;
    int64_t counts[8];    // accepted mutations per MutType
    int64_t pad[5];
};

enum Stage { ST_UPLOAD = 0, ST_SAMPLE_POS, ST_SAMPLE_TYPE, ST_SAMPLE_RESOLVE, ST_SAMPLE_LINK, ST_SAMPLE_FINAL,
             ST_PLAN, ST_INDEX, ST_SPLICE, ST_VCF, ST_DOWNLOAD, ST_CHAIN, ST_GENOTYPE, ST_SELECT, ST_VCF_PHASED, ST_READS, ST_COUNT };
static_assert(ST_COUNT <= (int)(sizeof(ms_stats::stage_ms) / sizeof(float)), "ms_stats.stage_ms has a slot per stage");

}  // namespace ms

namespace ms {
// One FASTA record as the device indexer sees it (ms_ingest.cu): what pyfaidx keeps per .fai line, plus the defline.
struct FaRec {
    int64_t hdr_lo, hdr_hi;   // '>' and the line break that ends the defline
    int64_t seq_lo;           // file offset of the first base
    int64_t goff;             // index of the first base in the stripped genome
    int64_t len;              // bases
    int64_t nfull;            // lines of exactly lenc bases followed by a line break
    int32_t lenc, lenb;       // bases / bytes per line
};
}  // namespace ms

struct ms_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    std::string err;

    // genome
    ms::DevBuf genome, contigs, headers, names, tables;
    std::vector<ms::Contig> h_contigs;
    int32_t n_contigs = 0;
    int64_t total_bases = 0;
    int64_t foreign_cap = 0;   // staging bytes behind the genome (ms_genome_reserve)
    struct PeerWindow { void* base; int64_t bytes; };   // another GPU's genome buffer, mapped with CUDA IPC (ms_peer_open)
    std::vector<PeerWindow> peers;
    const void* peer_anchor = nullptr;   // genome pointer the windows' offsets are relative to (stale once it moves)
    ms::DevBuf tmp_contigs;

    // ranges / sampling
    ms::DevBuf ranges, cand_val, big_ranges, bucket_cnt, bucket_off, cand_type, cand_len, cand_reach, cand_pm,
               cand_accept, acc_idx, tl_list, tli_list, link, keep, contig_tl, scan_tmp, scan_tmp2, scan_mid, svec, vvec, lvec, bucket_range;
    std::vector<ms::Range> h_ranges;
    int32_t n_ranges = 0;
    int64_t n_candidates = 0;
    int64_t n_buckets = 0;
    int split_levels = 0;         // levels k_split_top runs (bucket-tree nodes wider than SPLIT_LEAF)
    int32_t n_big = 0;            // ranges that have such nodes
    int32_t block[7] = {1, 1, 1, 1, 1, 1, 1};
    double p_ti = 0.5;
    int32_t min_dist = 1;
    int64_t maxspan = 2;          // longest blocking span of any candidate (set with the ranges)
    int any_small = 0, any_large = 0;
    bool counts_valid = false;
    bool rec_out_valid = false;   // Rec.out of the device table is filled in (done lazily when the records are handed out)
    bool sizes_valid = false;     // keep/cand_val hold (delta, vcf size) of the current records (written by k_build_records)
    ms::Seed seed_last{0, 0};     // seed of the last ms_sample (K_RAND payloads are a function of it)

    // records + outputs
    ms::DevBuf recs, lit, piece_lo, piece_desc, fasta, vcf, vcf_off, totals, nvec, sv_stream, snp_stream;
    int64_t n_recs = 0, lit_bytes = 0, fasta_bytes = 0, vcf_bytes = 0, n_pieces = 0, n_sv = 0;
    ms::Totals* h_totals = nullptr;  // pinned
    static constexpr int N_STAGE = 6;            // pinned staging buffers of ms_download_to_fd / ms_fasta_ingest_fd:
    static constexpr int64_t STAGE_BYTES = 16 << 20;   // one file read / write per buffer in flight, each on its own thread
    uint8_t* h_stage[N_STAGE] = {};
    cudaEvent_t h_stage_ev[N_STAGE] = {};
    ms::Totals last_totals{};

    // timing
    cudaEvent_t ev[ms::ST_COUNT][2];
    bool ev_used[ms::ST_COUNT];
    float stage_ms[ms::ST_COUNT];
    int64_t kernel_launches = 0;
    int tile_bytes = ms::TL_TILE;
    bool splice_attr_set = false, vcf_attr_set = false;   // cudaFuncSetAttribute done on this context's device

    // device FASTA ingest (ms_fasta_ingest_fd .. ms_fasta_commit)
    std::vector<ms::FaRec> fa_recs;
    ms::DevBuf fa_index;
    int64_t fa_bytes = 0;

    // streamed run (ms_mutate_streamed): copy streams and per-group events
    cudaStream_t s_up = nullptr, s_down = nullptr, s_vcf = nullptr;
    std::vector<cudaEvent_t> ev_up, ev_done, ev_sized;
    ms::DevBuf vend;                 // VCF bytes up to the end of each contig group
    int64_t* h_vend = nullptr;       // pinned copy
    size_t h_vend_cap = 0;

    // BGZF output of the last ms_bgzf_compress (buffer 5), its block table and per-member scratch
    ms::DevBuf bgzf, bgzf_blocks, bgzf_slots, bgzf_zsize;
    int64_t bgzf_bytes = 0;

    // ms_load_vcf: text, line starts, per-line records (then the new table), compacted records, the new literal pool,
    // the CHROM hash table, scalars and per-contig block bounds
    ms::DevBuf vp_text, vp_lines, vp_lrec, vp_krec, vp_lit, vp_names, vp_contig;

    // chain file of the last apply (buffer 6): per-contig summary, per-SvRec prefixes of cons and of copy records
    ms::DevBuf chain, chain_cc, chain_cons, chain_copy, chain_off, chain_err;
    std::vector<ms::ChainCtg> h_chain_cc;
    int64_t chain_bytes = 0;
    bool chain_ready = false;     // the SvRec stream and contig table describe the last ms_apply / ms_apply_window
    bool chain_counted = false;   // h_chain_cc holds ms_chain_count's summary of that output

    // polyploid runs (ms_genotype.cu): haplotype masks of the full table (buffer 8), the full table while a haplotype's
    // records are the active table, the phased VCF body (buffer 7), its per-record and per-contig offsets
    ms::DevBuf gt_mask, recs_full, gt_vcf, gt_voff, gt_ctg_off, vp_lmask, vp_kmask;
    int32_t gt_ploidy = 0;        // 0: the current table has no masks
    int32_t gt_selected = 0;      // haplotype whose records are the active table (0: the full table is)
    int64_t gt_n_full = 0;        // records of the full table while a haplotype is selected
    bool gt_sizes_valid_full = false;
    int64_t gt_vcf_bytes = 0;

    // paired-end reads (ms_reads.cu): FASTQ records of the last ms_reads_write (buffer 9), the per-pair draws and record
    // offsets of the last sized range, the prefix of n_pairs, per-contig bytes
    ms::DevBuf reads, reads_info, reads_off, reads_pre, reads_ctg;
    int64_t reads_bytes = 0;
    bool apply_full = false;      // buffer 0 and the active table's out positions describe the last full ms_apply
    bool reads_sized = false;     // reads_info / reads_off hold the range below (ms_reads_size)
    ms::ReadsCfg reads_cfg{};
    int64_t reads_first = 0, reads_count = 0, reads_sized_total = 0;
    std::vector<int64_t> h_reads_pre, reads_sized_pre;
};

#define MS_CUDA(ctx, call)                                                                        \
    do {                                                                                          \
        cudaError_t _e = (call);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            char _b[512];                                                                         \
            snprintf(_b, sizeof(_b), "%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            (ctx)->err = _b;                                                                      \
            return MS_ERR_CUDA;                                                                   \
        }                                                                                         \
    } while (0)

#define MS_FAIL(ctx, code, ...)                                \
    do {                                                       \
        char _b[512];                                          \
        snprintf(_b, sizeof(_b), __VA_ARGS__);                 \
        (ctx)->err = _b;                                       \
        return (code);                                         \
    } while (0)

#define MS_LAUNCH_CHECK(ctx)                                   \
    do {                                                       \
        (ctx)->kernel_launches++;                              \
        MS_CUDA(ctx, cudaGetLastError());                      \
    } while (0)

namespace ms {
inline void stage_begin(ms_ctx* c, Stage s) { cudaEventRecord(c->ev[s][0], c->stream); }
inline void stage_end(ms_ctx* c, Stage s) { cudaEventRecord(c->ev[s][1], c->stream); c->ev_used[s] = true; }
inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// pipeline entry points implemented in the .cu files
int apply_pipeline(ms_ctx* c);
int apply_window(ms_ctx* c, int part, int n_parts, int64_t* win);
int adopt_output(ms_ctx* c);
int ensure_stage_buffers(ms_ctx* c);
int fasta_ingest(ms_ctx* c, int fd, int32_t n_ranges, const int64_t* off, const int64_t* len, int32_t* n_records, int32_t* regular);
int fasta_index(ms_ctx* c, int64_t* hdr_off, int64_t* seq_off, int64_t* length, int32_t* lenc, int32_t* lenb, uint8_t* hdr_blob,
                int64_t blob_cap);
int fasta_strip(ms_ctx* c, int64_t total, int32_t* regular);
int sample_pipeline(ms_ctx* c, uint64_t seed, bool defer_bases = false);
int mutate_streamed(ms_ctx* c, uint64_t seed, const uint8_t* h_bases, uint8_t* h_fasta, int64_t fasta_cap, uint8_t* h_vcf,
                    int64_t vcf_cap, int64_t* fasta_bytes, int64_t* vcf_bytes, int64_t group_min);
int count_types(ms_ctx* c);
int fill_record_out(ms_ctx* c);
int hash_ranges(ms_ctx* c, const uint8_t* buf, int32_t n, const int64_t* start, const int64_t* end, uint64_t* out);
int vcf_load(ms_ctx* c, const uint8_t* text, int64_t nbytes, int32_t skip_unknown, int32_t ploidy, int32_t* regular,
             int64_t* n_recs);
int record_fault(ms_ctx* c, int fault, int64_t i);
void records_loaded(ms_ctx* c, int64_t n_recs, int64_t lit_bytes);
int bgzf_compress(ms_ctx* c, int which, int32_t n_seg, const int64_t* src_off, const int64_t* nbytes, const int64_t* file_off,
                  const uint8_t* add_nl, int64_t* seg_zbytes, int64_t* total_zbytes);
void chain_invalidate(ms_ctx* c);
int chain_count(ms_ctx* c, int64_t* n_chains);
int chain_write(ms_ctx* c, const int64_t* first_id, int64_t* chain_off);
void genotype_clear(ms_ctx* c);
int genotype_draw(ms_ctx* c, uint64_t seed, int32_t ploidy, double hom_fraction);
int genotype_load(ms_ctx* c, const uint8_t* masks, int64_t n, int32_t ploidy);
int select_haplotype(ms_ctx* c, int32_t h);
int vcf_phased(ms_ctx* c, int64_t* vcf_off);
void reads_invalidate(ms_ctx* c);
int reads_size(ms_ctx* c, const ms_reads_cfg* cfg, const int64_t* n_pairs, int64_t first, int64_t count, int64_t* bytes);
int reads_write(ms_ctx* c, const ms_reads_cfg* cfg, const int64_t* n_pairs, int64_t first, int64_t count, int64_t* nbytes);
}  // namespace ms
