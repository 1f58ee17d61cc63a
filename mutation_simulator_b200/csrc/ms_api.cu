// ms_api.cu — extern "C" entry points of libmutsim_b200.so (include/mutsim_b200.h):
// lifecycle, genome residency, record loading, downloads and introspection.
#include <errno.h>
#include <string.h>
#include <unistd.h>
#include <algorithm>
#include <future>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/statvfs.h>
#include "ms_bgzf_core.h"
#include "ms_common.cuh"
#include "ms_genotype_core.h"

using namespace ms;

static thread_local std::string g_create_error;

namespace ms {
// The error ms_load_records reports for record i failing check `fault` (rec_fault).
int record_fault(ms_ctx* c, int fault, int64_t i) {
    switch (fault) {
        case RF_CONTIG: MS_FAIL(c, MS_ERR_ARG, "record %lld: contig out of range", (long long)i);
        case RF_ORDER: MS_FAIL(c, MS_ERR_OVERLAP, "record %lld: records must be sorted by (contig, pos) with distinct positions", (long long)i);
        case RF_LIT: MS_FAIL(c, MS_ERR_ARG, "record %lld: literal range outside the pool", (long long)i);
        default: MS_FAIL(c, MS_ERR_ARG, "record %lld: source range outside the genome", (long long)i);
    }
}

// The record table and literal pool of c are now a loaded table (ms_load_records, ms_load_vcf).
void records_loaded(ms_ctx* c, int64_t n_recs, int64_t lit_bytes) {
    c->n_recs = n_recs;
    c->lit_bytes = lit_bytes;
    c->counts_valid = false;
    c->sizes_valid = false;
    c->rec_out_valid = true;
    chain_invalidate(c);
    genotype_clear(c);
}
}  // namespace ms

static const char* STAGE_NAMES[ST_COUNT] = {"upload", "sample_positions", "sample_type_len", "sample_resolve",
                                            "sample_link", "sample_finalize", "plan_scan_layout", "block_index",
                                            "splice_emit_fasta", "vcf_format", "download", "chain_format",
                                            "genotype", "select", "vcf_phased", "reads"};

extern "C" {

int ms_abi_version(void) { return 1; }

const char* ms_stage_name(int s) { return (s >= 0 && s < ST_COUNT) ? STAGE_NAMES[s] : ""; }

const char* ms_last_error(const ms_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int ms_create(int device, ms_ctx** out) {
    if (!out) return MS_ERR_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        g_create_error = std::string("no CUDA device available (") + cudaGetErrorString(e) +
                         "); libmutsim_b200 has no CPU fallback";
        return MS_ERR_CUDA;
    }
    if (device < 0 || device >= n) { g_create_error = "device index out of range"; return MS_ERR_ARG; }
    if ((e = cudaSetDevice(device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return MS_ERR_CUDA; }
    ms_ctx* c = new ms_ctx();
    c->device = device;
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e); delete c; return MS_ERR_CUDA;
    }
    for (int s = 0; s < ST_COUNT; ++s) {
        cudaEventCreate(&c->ev[s][0]); cudaEventCreate(&c->ev[s][1]);
        c->ev_used[s] = false; c->stage_ms[s] = 0.f;
    }
    if ((e = cudaMallocHost((void**)&c->h_totals, sizeof(Totals))) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e); delete c; return MS_ERR_CUDA;
    }
    memset(c->h_totals, 0, sizeof(Totals));
    Tables t; fill_tables(t);
    if (c->tables.ensure(sizeof(Tables)) != cudaSuccess || c->totals.ensure(sizeof(Totals)) != cudaSuccess ||
        cudaMemcpy(c->tables.p, &t, sizeof(Tables), cudaMemcpyHostToDevice) != cudaSuccess) {
        g_create_error = "device allocation failed"; delete c; return MS_ERR_CUDA;
    }
    *out = c;
    return MS_OK;
}

// [src, src + n) — relative to this context's genome pointer — lies inside one of the mapped peer buffers
static bool source_in_peer_window(const ms_ctx* c, int64_t src, int64_t n) {
    if (c->peer_anchor != c->genome.p) return false;   // the genome moved since ms_peer_open
    const uint8_t* a = (const uint8_t*)c->genome.p + src;
    for (const auto& w : c->peers)
        if (a >= (const uint8_t*)w.base && a + n <= (const uint8_t*)w.base + w.bytes) return true;
    return false;
}

int ms_destroy(ms_ctx* c) {
    if (!c) return MS_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto& w : c->peers) cudaIpcCloseMemHandle(w.base);
    c->peers.clear();
    DevBuf* bufs[] = {&c->genome, &c->contigs, &c->headers, &c->names, &c->tables, &c->ranges, &c->cand_val, &c->big_ranges,
                      &c->bucket_cnt, &c->bucket_off, &c->cand_type, &c->cand_len, &c->cand_reach, &c->cand_pm, &c->cand_accept,
                      &c->acc_idx, &c->tl_list, &c->tli_list, &c->link, &c->keep, &c->contig_tl, &c->scan_tmp, &c->scan_tmp2,
                      &c->svec, &c->vvec, &c->lvec, &c->tmp_contigs, &c->recs, &c->lit, &c->scan_mid, &c->nvec, &c->sv_stream, &c->snp_stream, &c->piece_lo, &c->piece_desc, &c->fasta, &c->vcf,
                      &c->vcf_off, &c->totals, &c->bucket_range, &c->vend, &c->fa_index, &c->bgzf, &c->bgzf_blocks,
                      &c->bgzf_slots, &c->bgzf_zsize, &c->vp_text, &c->vp_lines, &c->vp_lrec, &c->vp_krec,
                      &c->vp_lit, &c->vp_names, &c->vp_contig, &c->chain, &c->chain_cc, &c->chain_cons, &c->chain_copy,
                      &c->chain_off, &c->chain_err, &c->gt_mask, &c->recs_full, &c->gt_vcf, &c->gt_voff, &c->gt_ctg_off,
                      &c->vp_lmask, &c->vp_kmask, &c->reads, &c->reads_info, &c->reads_off, &c->reads_pre, &c->reads_ctg};
    for (DevBuf* b : bufs) b->release();
    for (cudaStream_t* s : {&c->s_up, &c->s_down, &c->s_vcf})
        if (*s) { cudaStreamSynchronize(*s); cudaStreamDestroy(*s); }
    for (auto* evs : {&c->ev_up, &c->ev_done, &c->ev_sized})
        for (cudaEvent_t e : *evs) cudaEventDestroy(e);
    if (c->h_vend) cudaFreeHost(c->h_vend);
    for (int s = 0; s < ST_COUNT; ++s) { cudaEventDestroy(c->ev[s][0]); cudaEventDestroy(c->ev[s][1]); }
    if (c->h_totals) cudaFreeHost(c->h_totals);
    for (int i = 0; i < ms_ctx::N_STAGE; ++i) {
        if (c->h_stage[i]) cudaFreeHost(c->h_stage[i]);
        if (c->h_stage_ev[i]) cudaEventDestroy(c->h_stage_ev[i]);
    }
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return MS_OK;
}

int ms_set_stream(ms_ctx* c, void* stream) {
    if (!c) return MS_ERR_ARG;
    cudaStreamSynchronize(c->stream);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    c->stream = (cudaStream_t)stream;
    c->own_stream = false;
    return MS_OK;
}

int ms_synchronize(ms_ctx* c) {
    if (!c) return MS_ERR_ARG;
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    return MS_OK;
}

// util.py:87 sequence_always_upper: done on the device, 16 bytes per thread
__global__ void __launch_bounds__(256) k_upper(uint8_t* g, int64_t n16) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n16) return;
    uint4 v = reinterpret_cast<uint4*>(g)[i];
    uint32_t* w = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t x = w[k];
        // bytes in 'a'..'z' get bit 5 cleared: SWAR range test on 7-bit ASCII (bytes >= 0x80 are left alone)
        const uint32_t lo7 = x & 0x7F7F7F7Fu;
        const uint32_t ge_a = (lo7 + 0x1F1F1F1Fu) & 0x80808080u;          // byte >= 0x61
        const uint32_t gt_z = (lo7 + 0x05050505u) & 0x80808080u;          // byte >= 0x7B
        const uint32_t is_lower = ge_a & ~gt_z & ~(x & 0x80808080u);
        w[k] = x & ~(is_lower >> 2);
    }
    reinterpret_cast<uint4*>(g)[i] = v;
}

// ---- genome ---------------------------------------------------------------------------
static int set_contig_table(ms_ctx* c, int64_t total_bases, int32_t n_contigs, const int64_t* contig_len, const int32_t* bpl,
                            const uint32_t* gid, const uint8_t* headers, const int64_t* hdr_off, const uint8_t* names,
                            const int64_t* name_off) {
    if (n_contigs <= 0 || !contig_len || !bpl || !headers || !hdr_off || !names || !name_off)
        MS_FAIL(c, MS_ERR_ARG, "ms_genome: null argument or no contigs");
    c->h_contigs.assign(n_contigs, Contig{});
    int64_t off = 0;
    for (int i = 0; i < n_contigs; ++i) {
        Contig& k = c->h_contigs[i];
        if (contig_len[i] < 0 || contig_len[i] >= (int64_t)0x7FFFFFF0)
            MS_FAIL(c, MS_ERR_LIMIT, "contig %d has %lld bases; this build supports < 2^31 per contig", i, (long long)contig_len[i]);
        k.goff = off; k.len = contig_len[i]; k.out_len = contig_len[i];
        k.bpl = bpl[i] > 0 ? bpl[i] : 60;  // FastaWriter default (fasta_writer.py:26)
        k.hdr_src = hdr_off[i]; k.hdr_len = (int32_t)(hdr_off[i + 1] - hdr_off[i]);
        k.name_src = name_off[i]; k.name_len = (int32_t)(name_off[i + 1] - name_off[i]);
        k.gid = gid ? gid[i] : (uint32_t)i;
        off += contig_len[i];
    }
    if (off != total_bases) MS_FAIL(c, MS_ERR_ARG, "sum of contig lengths (%lld) != total_bases (%lld)", (long long)off, (long long)total_bases);
    c->n_contigs = n_contigs;
    c->total_bases = total_bases;
    MS_CUDA(c, c->contigs.ensure(sizeof(Contig) * (size_t)n_contigs));
    MS_CUDA(c, c->headers.ensure((size_t)hdr_off[n_contigs] + 16));
    MS_CUDA(c, c->names.ensure((size_t)name_off[n_contigs] + 16));
    MS_CUDA(c, cudaMemcpyAsync(c->contigs.p, c->h_contigs.data(), sizeof(Contig) * (size_t)n_contigs, cudaMemcpyHostToDevice, c->stream));
    MS_CUDA(c, cudaMemcpyAsync(c->headers.p, headers, (size_t)hdr_off[n_contigs], cudaMemcpyHostToDevice, c->stream));
    MS_CUDA(c, cudaMemcpyAsync(c->names.p, names, (size_t)name_off[n_contigs], cudaMemcpyHostToDevice, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));  // h_contigs / caller buffers may be pageable
    c->n_recs = 0; c->lit_bytes = 0; c->n_ranges = 0;
    chain_invalidate(c);
    genotype_clear(c);
    return MS_OK;
}

int ms_genome_upload(ms_ctx* c, const uint8_t* bases, int64_t total_bases, int32_t n_contigs, const int64_t* contig_len,
                     const int32_t* bpl, const uint32_t* gid, const uint8_t* headers, const int64_t* hdr_off,
                     const uint8_t* names, const int64_t* name_off) {
    if (!c) return MS_ERR_ARG;
    if (!bases && total_bases > 0) MS_FAIL(c, MS_ERR_ARG, "ms_genome_upload: bases is NULL");
    MS_CUDA(c, cudaSetDevice(c->device));
    stage_begin(c, ST_UPLOAD);
    MS_CUDA(c, c->genome.ensure((size_t)total_bases + 64 + (size_t)c->foreign_cap + 64));
    MS_CUDA(c, cudaMemcpyAsync(c->genome.p, bases, (size_t)total_bases, cudaMemcpyHostToDevice, c->stream));
    MS_CUDA(c, cudaMemsetAsync(c->genome.as<uint8_t>() + total_bases, 'N', 64, c->stream));
    if (total_bases > 0) {
        const int64_t n16 = (total_bases + 15) / 16;
        k_upper<<<(unsigned)((n16 + 255) / 256), 256, 0, c->stream>>>(c->genome.as<uint8_t>(), n16);
        MS_LAUNCH_CHECK(c);
    }
    stage_end(c, ST_UPLOAD);
    return set_contig_table(c, total_bases, n_contigs, contig_len, bpl, gid, headers, hdr_off, names, name_off);
}

int ms_genome_adopt(ms_ctx* c, const uint8_t* d_bases, int64_t total_bases, int32_t n_contigs, const int64_t* contig_len,
                    const int32_t* bpl, const uint32_t* gid, const uint8_t* headers, const int64_t* hdr_off,
                    const uint8_t* names, const int64_t* name_off) {
    if (!c) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    if (d_bases != c->genome.p) {
        MS_CUDA(c, c->genome.ensure((size_t)total_bases + 64));
        MS_CUDA(c, cudaMemcpyAsync(c->genome.p, d_bases, (size_t)total_bases, cudaMemcpyDeviceToDevice, c->stream));
    }
    MS_CUDA(c, cudaMemsetAsync(c->genome.as<uint8_t>() + total_bases, 'N', 64, c->stream));
    return set_contig_table(c, total_bases, n_contigs, contig_len, bpl, gid, headers, hdr_off, names, name_off);
}

int ms_genome_declare(ms_ctx* c, int64_t total_bases, int32_t n_contigs, const int64_t* contig_len, const int32_t* bpl,
                      const uint32_t* gid, const uint8_t* headers, const int64_t* hdr_off, const uint8_t* names,
                      const int64_t* name_off) {
    if (!c || total_bases < 0) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    MS_CUDA(c, c->genome.ensure((size_t)total_bases + 64 + (size_t)c->foreign_cap + 64));
    MS_CUDA(c, cudaMemsetAsync(c->genome.as<uint8_t>() + total_bases, 'N', 64, c->stream));
    return set_contig_table(c, total_bases, n_contigs, contig_len, bpl, gid, headers, hdr_off, names, name_off);
}

int ms_mutate_streamed(ms_ctx* c, uint64_t seed, const uint8_t* bases, uint8_t* fasta, int64_t fasta_cap, uint8_t* vcf,
                       int64_t vcf_cap, int64_t* fasta_bytes, int64_t* vcf_bytes, int64_t group_min_bases) {
    if (!c || !bases || !fasta || !vcf) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    genotype_clear(c);
    const int rc = mutate_streamed(c, seed, bases, fasta, fasta_cap, vcf, vcf_cap, fasta_bytes, vcf_bytes, group_min_bases);
    if (rc != MS_OK) {   // nothing may still be copying from / into the caller's buffers when the error is reported
        cudaStreamSynchronize(c->stream);
        if (c->s_up) { cudaStreamSynchronize(c->s_up); cudaStreamSynchronize(c->s_down); cudaStreamSynchronize(c->s_vcf); }
    }
    return rc;
}

int ms_fasta_ingest_fd(ms_ctx* c, int fd, int64_t nbytes, int32_t* n_records, int32_t* regular) {
    if (!c || fd < 0 || nbytes < 0 || !n_records || !regular) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    const int64_t off = 0;
    return fasta_ingest(c, fd, 1, &off, &nbytes, n_records, regular);
}

int ms_fasta_ingest_ranges(ms_ctx* c, int fd, int32_t n_ranges, const int64_t* off, const int64_t* len, int32_t* n_records,
                           int32_t* regular) {
    if (!c || fd < 0 || n_ranges < 0 || (n_ranges > 0 && (!off || !len)) || !n_records || !regular) return MS_ERR_ARG;
    for (int32_t r = 0; r < n_ranges; ++r)
        if (off[r] < 0 || len[r] < 0) MS_FAIL(c, MS_ERR_ARG, "ms_fasta_ingest_ranges: range %d is negative", r);
    MS_CUDA(c, cudaSetDevice(c->device));
    return fasta_ingest(c, fd, n_ranges, off, len, n_records, regular);
}

int ms_fasta_index(ms_ctx* c, int64_t* hdr_off, int64_t* seq_off, int64_t* length, int32_t* lenc, int32_t* lenb, uint8_t* hdr_blob,
                   int64_t blob_cap) {
    if (!c || !hdr_off) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return fasta_index(c, hdr_off, seq_off, length, lenc, lenb, hdr_blob, blob_cap);
}

int ms_fasta_commit(ms_ctx* c, const uint32_t* gid, const uint8_t* headers, const int64_t* hdr_off, const uint8_t* names,
                    const int64_t* name_off, int32_t* regular) {
    if (!c || !regular) return MS_ERR_ARG;
    const int32_t n = (int32_t)c->fa_recs.size();
    if (n == 0) MS_FAIL(c, MS_ERR_STATE, "ms_fasta_commit: no ingested file");
    MS_CUDA(c, cudaSetDevice(c->device));
    int64_t total = 0;
    std::vector<int64_t> len((size_t)n);
    std::vector<int32_t> bpl((size_t)n);
    for (int i = 0; i < n; ++i) { len[i] = c->fa_recs[i].len; bpl[i] = c->fa_recs[i].lenc; total += len[i]; }
    MS_CUDA(c, c->genome.ensure((size_t)total + 64 + (size_t)c->foreign_cap + 64));
    int rc = fasta_strip(c, total, regular);
    if (rc) return rc;
    c->fa_recs.clear();                       // the image is consumed either way
    if (!*regular) return MS_OK;
    MS_CUDA(c, cudaMemsetAsync(c->genome.as<uint8_t>() + total, 'N', 64, c->stream));
    return set_contig_table(c, total, n, len.data(), bpl.data(), gid, headers, hdr_off, names, name_off);
}

int ms_genome_subset(ms_ctx* c, const int32_t* ids, int32_t n) {
    if (!c || !ids || n <= 0) return MS_ERR_ARG;
    if (c->n_contigs <= 0 || !c->genome.p) MS_FAIL(c, MS_ERR_STATE, "ms_genome_subset: no genome resident");
    MS_CUDA(c, cudaSetDevice(c->device));
    std::vector<Contig> keep((size_t)n);
    int64_t total = 0;
    for (int i = 0; i < n; ++i) {
        if (ids[i] < 0 || ids[i] >= c->n_contigs) MS_FAIL(c, MS_ERR_ARG, "ms_genome_subset: contig %d out of range", ids[i]);
        keep[i] = c->h_contigs[ids[i]];
        total += keep[i].len;
    }
    DevBuf fresh;
    MS_CUDA(c, fresh.ensure((size_t)total + 64 + (size_t)c->foreign_cap + 64));
    int64_t off = 0;
    for (int i = 0; i < n; ++i) {
        if (keep[i].len > 0)
            MS_CUDA(c, cudaMemcpyAsync(fresh.as<uint8_t>() + off, c->genome.as<uint8_t>() + keep[i].goff, (size_t)keep[i].len,
                                       cudaMemcpyDeviceToDevice, c->stream));
        keep[i].goff = off; keep[i].out_len = keep[i].len; keep[i].rec_lo = keep[i].rec_hi = 0;
        off += keep[i].len;
    }
    MS_CUDA(c, cudaMemsetAsync(fresh.as<uint8_t>() + total, 'N', 64, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    c->genome.release();
    c->genome = fresh;
    c->h_contigs = keep;              // header / name blobs stay as they are: the kept entries still point into them
    c->n_contigs = n;
    c->total_bases = total;
    MS_CUDA(c, cudaMemcpyAsync(c->contigs.p, c->h_contigs.data(), sizeof(Contig) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    c->n_recs = 0; c->lit_bytes = 0; c->n_ranges = 0; c->sizes_valid = false; c->counts_valid = false;
    c->fasta_bytes = 0; c->vcf_bytes = 0;
    chain_invalidate(c);
    genotype_clear(c);
    return MS_OK;
}

int ms_genome_read(ms_ctx* c, int64_t off, int64_t n, uint8_t* dst) {
    if (!c || off < 0 || n < 0 || (n > 0 && !dst)) return MS_ERR_ARG;
    if (off + n > c->total_bases) MS_FAIL(c, MS_ERR_ARG, "ms_genome_read: range outside the genome");
    MS_CUDA(c, cudaSetDevice(c->device));
    if (n > 0) MS_CUDA(c, cudaMemcpyAsync(dst, c->genome.as<uint8_t>() + off, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    return MS_OK;
}

int ms_genome_reserve(ms_ctx* c, int64_t extra_bytes) {
    if (!c || extra_bytes < 0) return MS_ERR_ARG;
    c->foreign_cap = extra_bytes;
    // a genome that is already resident (ingested straight from the file) moves into a buffer with the staging space
    const size_t need = (size_t)c->total_bases + 64 + (size_t)extra_bytes + 64;
    if (c->n_contigs > 0 && c->genome.p && c->genome.cap < need) {
        MS_CUDA(c, cudaSetDevice(c->device));
        DevBuf fresh;
        MS_CUDA(c, fresh.ensure(need));
        MS_CUDA(c, cudaMemcpyAsync(fresh.p, c->genome.p, (size_t)c->total_bases + 64, cudaMemcpyDeviceToDevice, c->stream));
        MS_CUDA(c, cudaStreamSynchronize(c->stream));
        c->genome.release();
        c->genome = fresh;
    }
    return MS_OK;
}

// ---- peer windows: a partner contig that lives on another GPU is read in place over NVLink ------------------------
static void close_peers(ms_ctx* c) {
    for (auto& w : c->peers) cudaIpcCloseMemHandle(w.base);
    c->peers.clear();
}

int ms_genome_export(ms_ctx* c, uint8_t* handle, int64_t* nbytes) {
    if (!c || !handle || !nbytes) return MS_ERR_ARG;
    if (c->n_contigs <= 0 || !c->genome.p) MS_FAIL(c, MS_ERR_STATE, "ms_genome_export: no resident genome");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    MS_CUDA(c, cudaSetDevice(c->device));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));     // peers read what earlier calls on this stream wrote
    cudaIpcMemHandle_t h;
    MS_CUDA(c, cudaIpcGetMemHandle(&h, c->genome.p));
    memcpy(handle, &h, 64);
    *nbytes = c->total_bases + 64;
    return MS_OK;
}

int ms_peer_open(ms_ctx* c, const uint8_t* handle, int64_t nbytes, int64_t* rel_off) {
    if (!c || !handle || !rel_off || nbytes <= 0) return MS_ERR_ARG;
    if (!c->genome.p) MS_FAIL(c, MS_ERR_STATE, "ms_peer_open: upload this rank's genome first (sources are relative to it)");
    MS_CUDA(c, cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    void* base = nullptr;
    MS_CUDA(c, cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
    if (c->peer_anchor != c->genome.p) close_peers(c);   // offsets handed out earlier are void
    c->peer_anchor = c->genome.p;
    c->peers.push_back({base, nbytes});
    *rel_off = (int64_t)((const uint8_t*)base - (const uint8_t*)c->genome.p);
    return MS_OK;
}

int ms_peer_pull(ms_ctx* c, int32_t n, const int64_t* src, const int64_t* dst, const int64_t* nbytes) {
    if (!c || n < 0 || (n > 0 && (!src || !dst || !nbytes))) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    uint8_t* g = (uint8_t*)c->genome.p;
    for (int32_t i = 0; i < n; ++i) {
        if (nbytes[i] < 0 || dst[i] < c->total_bases + 64 || dst[i] + nbytes[i] > c->total_bases + 64 + c->foreign_cap)
            MS_FAIL(c, MS_ERR_ARG, "ms_peer_pull: copy %d lands outside the staging region", i);
        if (!source_in_peer_window(c, src[i], nbytes[i])) MS_FAIL(c, MS_ERR_ARG, "ms_peer_pull: copy %d reads outside every peer window", i);
        if (nbytes[i]) MS_CUDA(c, cudaMemcpyAsync(g + dst[i], g + src[i], (size_t)nbytes[i], cudaMemcpyDefault, c->stream));
    }
    return MS_OK;
}

int ms_peer_close(ms_ctx* c) {
    if (!c) return MS_ERR_ARG;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    close_peers(c);
    return MS_OK;
}

int ms_genome_adopt_output(ms_ctx* c) {
    if (!c) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return adopt_output(c);
}

int ms_genome_download(ms_ctx* c, uint8_t* bases, int64_t cap) {
    if (!c || !bases) return MS_ERR_ARG;
    if (cap < c->total_bases) MS_FAIL(c, MS_ERR_ARG, "buffer too small");
    MS_CUDA(c, cudaMemcpyAsync(bases, c->genome.p, (size_t)c->total_bases, cudaMemcpyDeviceToHost, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    return MS_OK;
}

// ---- replay ---------------------------------------------------------------------------
int ms_load_records(ms_ctx* c, const ms_rec* recs, int64_t n_recs, const uint8_t* lit, int64_t lit_bytes) {
    if (!c || n_recs < 0 || lit_bytes < 0 || (n_recs > 0 && !recs)) return MS_ERR_ARG;
    if (c->n_contigs <= 0) MS_FAIL(c, MS_ERR_STATE, "ms_load_records: upload a genome first");
    static_assert(sizeof(ms_rec) == sizeof(Rec), "ms_rec layout");
    const Rec* r = reinterpret_cast<const Rec*>(recs);
    for (int64_t i = 0; i < n_recs; ++i) {
        int f = rec_fault(r, i, c->n_contigs, lit_bytes, c->total_bases + 64 + c->foreign_cap);
        if (f == RF_SRC && r[i].kind == K_RAW && source_in_peer_window(c, r[i].src, r[i].prod)) f = RF_OK;
        if (f) return record_fault(c, f, i);
    }
    MS_CUDA(c, cudaSetDevice(c->device));
    MS_CUDA(c, c->recs.ensure((size_t)(n_recs + 1) * sizeof(Rec)));
    MS_CUDA(c, c->lit.ensure((size_t)lit_bytes + 64));
    if (n_recs) MS_CUDA(c, cudaMemcpyAsync(c->recs.p, recs, (size_t)n_recs * sizeof(Rec), cudaMemcpyHostToDevice, c->stream));
    if (lit_bytes) MS_CUDA(c, cudaMemcpyAsync(c->lit.p, lit, (size_t)lit_bytes, cudaMemcpyHostToDevice, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    records_loaded(c, n_recs, lit_bytes);
    return MS_OK;
}

int ms_load_vcf(ms_ctx* c, const uint8_t* text, int64_t nbytes, int32_t skip_unknown, int32_t* regular, int64_t* n_recs) {
    if (!c || nbytes < 0 || (nbytes > 0 && !text) || !regular || !n_recs) return MS_ERR_ARG;
    *regular = 0; *n_recs = 0;
    if (c->n_contigs <= 0) MS_FAIL(c, MS_ERR_STATE, "ms_load_vcf: upload a genome first");
    MS_CUDA(c, cudaSetDevice(c->device));
    return vcf_load(c, text, nbytes, skip_unknown, 0, regular, n_recs);
}

int ms_load_vcf_phased(ms_ctx* c, const uint8_t* text, int64_t nbytes, int32_t skip_unknown, int32_t ploidy, int32_t* regular,
                       int64_t* n_recs) {
    if (!c || nbytes < 0 || (nbytes > 0 && !text) || !regular || !n_recs) return MS_ERR_ARG;
    *regular = 0; *n_recs = 0;
    if (ploidy < 2 || ploidy > MAX_PLOIDY) MS_FAIL(c, MS_ERR_ARG, "ms_load_vcf_phased: ploidy %d outside 2..%d", ploidy, MAX_PLOIDY);
    if (c->n_contigs <= 0) MS_FAIL(c, MS_ERR_STATE, "ms_load_vcf_phased: upload a genome first");
    MS_CUDA(c, cudaSetDevice(c->device));
    return vcf_load(c, text, nbytes, skip_unknown, ploidy, regular, n_recs);
}

// ---- polyploid runs -------------------------------------------------------------------
int ms_genotype_draw(ms_ctx* c, uint64_t seed, int32_t ploidy, double hom_fraction) {
    if (!c) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return genotype_draw(c, seed, ploidy, hom_fraction);
}

int ms_genotype_load(ms_ctx* c, const uint8_t* masks, int64_t n, int32_t ploidy) {
    if (!c || n < 0 || (n > 0 && !masks)) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return genotype_load(c, masks, n, ploidy);
}

int ms_select_haplotype(ms_ctx* c, int32_t h) {
    if (!c) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return select_haplotype(c, h);
}

int ms_vcf_phased(ms_ctx* c, int64_t* vcf_off) {
    if (!c || !vcf_off) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return vcf_phased(c, vcf_off);
}

// ---- apply ----------------------------------------------------------------------------
int ms_apply(ms_ctx* c, int64_t* fasta_bytes, int64_t* vcf_bytes) {
    if (!c) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    int rc = apply_pipeline(c);
    if (rc != MS_OK) return rc;
    if (fasta_bytes) *fasta_bytes = c->fasta_bytes;
    if (vcf_bytes) *vcf_bytes = c->vcf_bytes;
    return MS_OK;
}

int ms_apply_window(ms_ctx* c, int32_t part, int32_t n_parts, int64_t* window) {
    if (!c || !window) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return apply_window(c, part, n_parts, window);
}

static int which_buffer(ms_ctx* c, int which, void** p, int64_t* n) {
    switch (which) {
        case 0: *p = c->fasta.p; *n = c->fasta_bytes; return MS_OK;
        case 1: *p = c->vcf.p; *n = c->vcf_bytes; return MS_OK;
        case 2: { int rc = fill_record_out(c); if (rc) return rc; }
                *p = c->recs.p; *n = c->n_recs * (int64_t)sizeof(Rec); return MS_OK;
        case 3: *p = c->lit.p; *n = c->lit_bytes; return MS_OK;
        case 4: *p = c->genome.p; *n = c->total_bases; return MS_OK;
        case 5: *p = c->bgzf.p; *n = c->bgzf_bytes; return MS_OK;
        case 6: *p = c->chain.p; *n = c->chain_bytes; return MS_OK;
        case 7: *p = c->gt_vcf.p; *n = c->gt_vcf_bytes; return MS_OK;
        case 8: *p = c->gt_mask.p; *n = c->gt_ploidy ? (c->gt_selected ? c->gt_n_full : c->n_recs) : 0; return MS_OK;
        case 9: *p = c->reads.p; *n = c->reads_bytes; return MS_OK;
        default: MS_FAIL(c, MS_ERR_ARG, "unknown buffer id %d", which);
    }
}

int ms_download(ms_ctx* c, int which, void* dst, int64_t cap, int64_t* nbytes) {
    if (!c) return MS_ERR_ARG;
    void* p; int64_t n;
    int rc = which_buffer(c, which, &p, &n);
    if (rc) return rc;
    if (nbytes) *nbytes = n;
    if (!dst) return MS_OK;  // size query
    if (cap < n) MS_FAIL(c, MS_ERR_ARG, "ms_download: buffer too small (%lld < %lld)", (long long)cap, (long long)n);
    MS_CUDA(c, cudaSetDevice(c->device));
    stage_begin(c, ST_DOWNLOAD);
    if (n) MS_CUDA(c, cudaMemcpyAsync(dst, p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    stage_end(c, ST_DOWNLOAD);
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    return MS_OK;
}

// returns 0 or errno (called from writer threads: no access to the context)
static int pwrite_all(int fd, const uint8_t* p, int64_t n, int64_t off) {
    while (n > 0) {
        const ssize_t w = pwrite(fd, p, (size_t)n, (off_t)off);
        if (w < 0) {
            if (errno == EINTR) continue;
            return errno ? errno : EIO;
        }
        p += w; n -= w; off += w;
    }
    return 0;
}

int ms_download_to_fd(ms_ctx* c, int which, int64_t src_off, int64_t nbytes, int fd, int64_t file_off) {
    if (!c || fd < 0 || src_off < 0 || nbytes < 0 || file_off < 0) return MS_ERR_ARG;
    void* p; int64_t total;
    int rc = which_buffer(c, which, &p, &total);
    if (rc) return rc;
    if (src_off + nbytes > total) MS_FAIL(c, MS_ERR_ARG, "ms_download_to_fd: range outside the buffer");
    if (nbytes == 0) return MS_OK;
    MS_CUDA(c, cudaSetDevice(c->device));
    if ((rc = ensure_stage_buffers(c))) return rc;
    constexpr int64_t CH = ms_ctx::STAGE_BYTES;
    constexpr int NS = ms_ctx::N_STAGE;
    const uint8_t* src = static_cast<const uint8_t*>(p) + src_off;
    const int64_t nch = (nbytes + CH - 1) / CH;
    // The D2H copies run back to back on the stream (55 GB/s); a page-cache / tmpfs write manages a few GB/s per
    // thread, so every staging buffer gets its own writer thread.  pwrite()s to one file serialise on the inode
    // lock, so the destination range is mapped (the file is grown first if needed) and the writers memcpy into the
    // mapping — page faults and copies then run in parallel; files that cannot be mapped (write-only descriptors,
    // pipes) take the pwrite path.
    uint8_t* map = nullptr;
    int64_t map_lo = 0, map_len = 0;
    {
        struct stat sb;
        const int64_t end = file_off + nbytes;
        // (a store into a mapping of a full file system raises SIGBUS where pwrite returns ENOSPC: the mapping is
        // only used when the file system reports room for the whole range with a margin)
        struct statvfs vfs;
        const bool room = fstatvfs(fd, &vfs) == 0 &&
                          (uint64_t)vfs.f_bavail * (uint64_t)vfs.f_frsize >= (uint64_t)nbytes + (uint64_t)nbytes / 8 + (64ull << 20);
        if (room && fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && (sb.st_size >= end || ftruncate(fd, (off_t)end) == 0)) {
            const int64_t page = sysconf(_SC_PAGESIZE);
            map_lo = file_off & ~(page - 1);
            map_len = end - map_lo;
            void* m = mmap(nullptr, (size_t)map_len, PROT_READ | PROT_WRITE, MAP_SHARED, fd, (off_t)map_lo);
            if (m != MAP_FAILED) map = static_cast<uint8_t*>(m);
        }
    }
    std::future<int> writer[NS];
    int werr = 0;
    const int device = c->device;
    stage_begin(c, ST_DOWNLOAD);
    for (int64_t i = 0; i < nch; ++i) {
        const int s = (int)(i % NS);
        if (writer[s].valid()) { const int e = writer[s].get(); if (e && !werr) werr = e; }   // buffer s is free again
        if (werr) break;
        const int64_t n = (i + 1) * CH <= nbytes ? CH : nbytes - i * CH;
        cudaError_t ce = cudaMemcpyAsync(c->h_stage[s], src + i * CH, (size_t)n, cudaMemcpyDeviceToHost, c->stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(c->h_stage_ev[s], c->stream);
        if (ce != cudaSuccess) { werr = -1; c->err = std::string("ms_download_to_fd: ") + cudaGetErrorString(ce); break; }
        const uint8_t* buf = c->h_stage[s];
        cudaEvent_t ev = c->h_stage_ev[s];
        const int64_t off = file_off + i * CH;
        writer[s] = std::async(std::launch::async, [=]() -> int {
            cudaSetDevice(device);
            if (cudaEventSynchronize(ev) != cudaSuccess) return EIO;
            if (map) { memcpy(map + (off - map_lo), buf, (size_t)n); return 0; }
            return pwrite_all(fd, buf, n, off);
        });
    }
    for (int s = 0; s < NS; ++s)
        if (writer[s].valid()) { const int e = writer[s].get(); if (e && !werr) werr = e; }
    if (map) munmap(map, (size_t)map_len);
    stage_end(c, ST_DOWNLOAD);
    if (werr == -1) return MS_ERR_CUDA;
    if (werr) MS_FAIL(c, MS_ERR_ARG, "pwrite failed: %s", strerror(werr));
    return MS_OK;
}

int ms_device_ptr(ms_ctx* c, int which, void** dptr, int64_t* nbytes) {
    if (!c || !dptr || !nbytes) return MS_ERR_ARG;
    return which_buffer(c, which, dptr, nbytes);
}

int ms_contig_out_len(ms_ctx* c, int64_t* out_len) {
    if (!c || !out_len) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    MS_CUDA(c, cudaMemcpy(c->h_contigs.data(), c->contigs.p, sizeof(Contig) * (size_t)c->n_contigs, cudaMemcpyDeviceToHost));
    for (int i = 0; i < c->n_contigs; ++i) out_len[i] = c->h_contigs[i].out_len;
    return MS_OK;
}

int ms_contig_layout(ms_ctx* c, int64_t* fasta_off, int64_t* vcf_off, uint8_t* sep, uint8_t* partial) {
    if (!c || !fasta_off || !vcf_off) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    MS_CUDA(c, cudaMemcpy(c->h_contigs.data(), c->contigs.p, sizeof(Contig) * (size_t)c->n_contigs, cudaMemcpyDeviceToHost));
    std::vector<int64_t> V;
    for (int i = 0; i < c->n_contigs; ++i) {
        const Contig& k = c->h_contigs[i];
        fasta_off[i] = k.hdr_off;
        if (sep) sep[i] = (uint8_t)k.sep;
        if (partial) partial[i] = (uint8_t)(k.out_len % k.bpl != 0);
        // V[rec_lo] of each contig: one 8-byte copy per contig is fine for genome-scale contig counts; batch for many
        vcf_off[i] = 0;
    }
    fasta_off[c->n_contigs] = c->fasta_bytes;
    if (c->n_recs > 0) {
        // gather V[rec_lo[c]] with a strided 2D copy when contigs are few, else download V once
        if (c->n_contigs <= 4096) {
            for (int i = 0; i < c->n_contigs; ++i)
                MS_CUDA(c, cudaMemcpy(&vcf_off[i], c->vcf_off.as<int64_t>() + c->h_contigs[i].rec_lo, 8, cudaMemcpyDeviceToHost));
        } else {
            V.resize((size_t)c->n_recs + 1);
            MS_CUDA(c, cudaMemcpy(V.data(), c->vcf_off.p, (size_t)(c->n_recs + 1) * 8, cudaMemcpyDeviceToHost));
            for (int i = 0; i < c->n_contigs; ++i) vcf_off[i] = V[(size_t)c->h_contigs[i].rec_lo];
        }
    }
    vcf_off[c->n_contigs] = c->vcf_bytes;
    return MS_OK;
}

int ms_contig_records(ms_ctx* c, int64_t* n_records) {
    if (!c || !n_records) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    MS_CUDA(c, cudaMemcpy(c->h_contigs.data(), c->contigs.p, sizeof(Contig) * (size_t)c->n_contigs, cudaMemcpyDeviceToHost));
    for (int i = 0; i < c->n_contigs; ++i) n_records[i] = c->h_contigs[i].rec_hi - c->h_contigs[i].rec_lo;
    return MS_OK;
}

int ms_hash_ranges(ms_ctx* c, int which, int32_t n, const int64_t* start, const int64_t* end, uint64_t* out) {
    if (!c || n < 0 || (n > 0 && (!start || !end || !out))) return MS_ERR_ARG;
    if (n == 0) return MS_OK;
    void* p; int64_t nb;
    int rc = which_buffer(c, which, &p, &nb);
    if (rc) return rc;
    for (int32_t i = 0; i < n; ++i)
        if (start[i] < 0 || end[i] < start[i] || end[i] > nb || (i && start[i] < end[i - 1]))
            MS_FAIL(c, MS_ERR_ARG, "ms_hash_ranges: range %d is outside the buffer or not in ascending order", i);
    MS_CUDA(c, cudaSetDevice(c->device));
    return hash_ranges(c, static_cast<const uint8_t*>(p), n, start, end, out);
}

int ms_bgzf_compress(ms_ctx* c, int which, int32_t n_seg, const int64_t* src_off, const int64_t* nbytes, const int64_t* file_off,
                     const uint8_t* add_nl, int64_t* seg_zbytes, int64_t* total_zbytes) {
    if (!c || (which != 0 && which != 1 && which != 6 && which != 7 && which != 9) || n_seg < 0 || !total_zbytes ||
        (n_seg > 0 && (!src_off || !nbytes || !file_off || !seg_zbytes)))
        return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return bgzf_compress(c, which, n_seg, src_off, nbytes, file_off, add_nl, seg_zbytes, total_zbytes);
}

int ms_bgzf_compress_host(ms_ctx* c, const uint8_t* src, int64_t n, uint8_t* dst, int64_t cap, int64_t* zbytes) {
    if (n < 0 || (n > 0 && !src) || !zbytes) return MS_ERR_ARG;
    const int64_t need = ((n + bgzf::CELL - 1) / bgzf::CELL) * bgzf::MAX_MEMBER;
    *zbytes = 0;
    if (!dst) { *zbytes = need; return MS_OK; }     // size query: an upper bound
    std::vector<uint8_t> member(bgzf::MAX_MEMBER);
    int64_t o = 0;
    for (int64_t i = 0; i < n; i += bgzf::CELL) {
        const int m = (int)std::min<int64_t>(bgzf::CELL, n - i);
        const int z = bgzf::encode_member(src + i, m, member.data());
        if (o + z > cap) {
            if (c) MS_FAIL(c, MS_ERR_ARG, "ms_bgzf_compress_host: output buffer too small");
            return MS_ERR_ARG;
        }
        memcpy(dst + o, member.data(), (size_t)z);
        o += z;
    }
    *zbytes = o;
    return MS_OK;
}

int ms_chain_count(ms_ctx* c, int64_t* n_chains) {
    if (!c || !n_chains) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return chain_count(c, n_chains);
}

int ms_chain_write(ms_ctx* c, const int64_t* first_id, int64_t* chain_off) {
    if (!c || !first_id || !chain_off) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return chain_write(c, first_id, chain_off);
}

int ms_reads_size(ms_ctx* c, const ms_reads_cfg* cfg, const int64_t* n_pairs, int64_t first, int64_t count, int64_t* bytes) {
    if (!c || !cfg || (c->n_contigs > 0 && (!n_pairs || !bytes))) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return reads_size(c, cfg, n_pairs, first, count, bytes);
}

int ms_reads_write(ms_ctx* c, const ms_reads_cfg* cfg, const int64_t* n_pairs, int64_t first, int64_t count, int64_t* nbytes) {
    if (!c || !cfg || !nbytes || (c->n_contigs > 0 && !n_pairs)) return MS_ERR_ARG;
    MS_CUDA(c, cudaSetDevice(c->device));
    return reads_write(c, cfg, n_pairs, first, count, nbytes);
}

int ms_get_stats(ms_ctx* c, ms_stats* out) {
    if (!c || !out) return MS_ERR_ARG;
    memset(out, 0, sizeof(*out));
    cudaStreamSynchronize(c->stream);
    if (c->n_recs >= 0 && c->recs.p) { int rc = count_types(c); if (rc) return rc; }
    for (int s = 0; s < ST_COUNT; ++s) {
        if (c->ev_used[s]) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, c->ev[s][0], c->ev[s][1]) == cudaSuccess) c->stage_ms[s] = ms;
        }
        out->stage_ms[s] = c->stage_ms[s];
    }
    out->n_candidates = c->last_totals.n_candidates;
    out->n_accepted = c->last_totals.n_accepted;
    out->n_records = c->n_recs;
    out->lit_bytes = c->lit_bytes;
    out->fasta_bytes = c->fasta_bytes;
    out->vcf_bytes = c->vcf_bytes;
    out->kernel_launches = c->kernel_launches;
    for (int t = 0; t < 8; ++t) out->counts[t] = c->last_totals.counts[t];
    return MS_OK;
}

}  // extern "C"
