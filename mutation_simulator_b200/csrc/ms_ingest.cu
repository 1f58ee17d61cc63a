// ms_ingest.cu — FASTA ingest on the device (SURVEY.md §8 f1).
//
// Replaces util.py:77-91 (load_fasta -> pyfaidx.Fasta: index the file, then serve upper-cased bases) for regularly
// wrapped files: the raw file bytes go to the GPU through a ring of pinned staging buffers, records and their line layout
// are found there, and the bases are stripped of line breaks, upper-cased and checked against that layout in one
// pass.  The host only ever sees the per-record index (what pyfaidx writes to the .fai) and the deflines.
// Anything irregular (CRLF, ragged or blank lines, lines longer than 1 MiB) is reported as "not regular" and the
// caller falls back to the host parser, which owns pyfaidx's error messages.
#include <unistd.h>
#include <string.h>
#include <errno.h>
#include <algorithm>
#include <future>
#include "ms_common.cuh"

namespace ms {

// '>' at offset 0 or right after a line break starts a record.  pos == nullptr: count only.
__global__ void __launch_bounds__(256)
k_fa_headers(const uint8_t* raw, int64_t n, unsigned long long* count, int64_t* pos, int64_t cap) {
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (i0 >= n) return;
    const uint4 v = *reinterpret_cast<const uint4*>(raw + i0);      // the image is padded to a multiple of 16
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    // SWAR: any byte equal to '>' in this group?
    bool any = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) { const uint32_t x = w[k] ^ 0x3E3E3E3Eu; any |= ((x - 0x01010101u) & ~x & 0x80808080u) != 0u; }
    if (!any) return;
    uint8_t prev = i0 > 0 ? raw[i0 - 1] : (uint8_t)'\n';
    for (int t = 0; t < 16 && i0 + t < n; ++t) {
        const uint8_t ch = (uint8_t)(w[t >> 2] >> (8 * (t & 3)));
        if (ch == '>' && prev == '\n') {
            const unsigned long long slot = atomicAdd(count, 1ull);
            if (pos && (int64_t)slot < cap) pos[slot] = i0 + t;
        }
        prev = ch;
    }
}

constexpr int64_t FA_SCAN_CAP = 1 << 20;   // longest defline / sequence line the device indexer follows

// One thread per record: defline end, first-line width, number of full lines, bases of the partial last line.
__global__ void __launch_bounds__(128)
k_fa_index(const uint8_t* raw, int64_t n, const int64_t* hdr, int32_t n_rec, FaRec* out, int* irregular) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_rec) return;
    FaRec r{};
    r.hdr_lo = hdr[c];
    const int64_t next = c + 1 < n_rec ? hdr[c + 1] : n;
    int64_t he = r.hdr_lo + 1;
    while (he < next && raw[he] != '\n' && he - r.hdr_lo < FA_SCAN_CAP) ++he;
    if (he < next && raw[he] != '\n') { *irregular = 1; return; }
    r.hdr_hi = he;
    if (he > r.hdr_lo + 1 && raw[he - 1] == '\r') { *irregular = 1; return; }     // CRLF: host parser
    const int64_t lo = he + 1 < next ? he + 1 : next, hi = next;
    r.seq_lo = lo;
    const int64_t R = hi - lo;
    if (R > 0) {
        int64_t nl = lo;
        while (nl < hi && raw[nl] != '\n' && nl - lo < FA_SCAN_CAP) ++nl;
        if (nl < hi && raw[nl] != '\n') { *irregular = 1; return; }
        if (nl == lo) { *irregular = 1; return; }                                 // blank first line
        if (nl == hi) {                      // a single line without a line break at the end of the file
            r.lenc = (int32_t)R; r.lenb = (int32_t)R; r.nfull = 0; r.len = R;
        } else {
            const int64_t b = nl - lo + 1;
            r.lenc = (int32_t)(b - 1); r.lenb = (int32_t)b;
            r.nfull = R / b;
            int64_t tail = R - r.nfull * b;
            while (tail > 0 && raw[lo + r.nfull * b + tail - 1] == '\n') --tail;     // blank lines at the end are tolerated
            r.len = r.nfull * (b - 1) + tail;
        }
    }
    out[c] = r;
}

// Deflines (without '>' and the line break) packed back to back.
__global__ void k_fa_pack_headers(const uint8_t* raw, const FaRec* recs, int32_t n_rec, const int64_t* off, uint8_t* blob) {
    const int c = blockIdx.x;
    if (c >= n_rec) return;
    const int64_t lo = recs[c].hdr_lo + 1, len = recs[c].hdr_hi - lo;
    for (int64_t i = threadIdx.x; i < len; i += blockDim.x) blob[off[c] + i] = raw[lo + i];
}

// Bases of every record, line breaks removed, upper-cased (util.py:87 sequence_always_upper); 16 bases per thread.
// Every byte taken as a base must not be a line break and every full line must end in '\n' where the layout says
// so: a file that passes is exactly what the index describes.
__global__ void __launch_bounds__(256)
k_fa_strip(const uint8_t* raw, const FaRec* recs, int32_t n_rec, int64_t total, uint8_t* genome, int* irregular) {
    const int64_t g0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (g0 >= total) return;
    int lo = 0, hi = n_rec;   // last record with goff <= g0
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (recs[mid].goff <= g0) lo = mid; else hi = mid; }
    int c = lo;
    while (c + 1 < n_rec && recs[c + 1].goff <= g0) ++c;   // (records of length 0 share an offset)
    FaRec r = recs[c];
    int64_t b = g0 - r.goff;
    int64_t line = b / r.lenc;
    int64_t col = b - line * r.lenc;
    const uint8_t* src = raw + r.seq_lo + line * r.lenb + col;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    bool bad = false;
    for (int t = 0; t < 16 && g0 + t < total; ++t) {
        while (b >= r.len) {                 // next record
            ++c; r = recs[c]; b = 0; line = 0; col = 0; src = raw + r.seq_lo;
        }
        uint8_t ch = *src;
        bad |= ch == '\n' || ch == '\r';
        if (ch >= 'a' && ch <= 'z') ch -= 32;
        w[t >> 2] |= (uint32_t)ch << (8 * (t & 3));
        ++b; ++col; ++src;
        if (col == r.lenc) {                 // end of a full line
            if (line < r.nfull) { bad |= *src != '\n'; }
            src += r.lenb - r.lenc; col = 0; ++line;
        }
    }
    if (bad) *irregular = 1;
    if (g0 + 16 <= total) *reinterpret_cast<uint4*>(genome + g0) = make_uint4(w[0], w[1], w[2], w[3]);
    else for (int t = 0; g0 + t < total; ++t) genome[g0 + t] = (uint8_t)(w[t >> 2] >> (8 * (t & 3)));
}

// pinned staging buffers shared by ms_fasta_ingest_fd and ms_download_to_fd
int ensure_stage_buffers(ms_ctx* c) {
    for (int i = 0; i < ms_ctx::N_STAGE; ++i) {
        if (!c->h_stage[i]) MS_CUDA(c, cudaMallocHost((void**)&c->h_stage[i], (size_t)ms_ctx::STAGE_BYTES));
        if (!c->h_stage_ev[i]) MS_CUDA(c, cudaEventCreateWithFlags(&c->h_stage_ev[i], cudaEventDisableTiming));
    }
    return MS_OK;
}

// returns 0 or errno (called from reader threads)
static int pread_all(int fd, uint8_t* dst, int64_t n, int64_t off) {
    while (n > 0) {
        const ssize_t k = pread(fd, dst, (size_t)n, (off_t)off);
        if (k < 0 && errno == EINTR) continue;
        if (k <= 0) return k < 0 && errno ? errno : EIO;
        dst += k; off += k; n -= k;
    }
    return 0;
}

// file -> device image -> record index.  The image lives in the FASTA output buffer (dead until the next ms_apply).
// The image is the concatenation of the file's byte ranges [off[r], off[r] + len[r]) (whole records each: one process per
// GPU reads only the records of its own contigs); a single range [0, nbytes) is the whole file.
int fasta_ingest(ms_ctx* c, int fd, int32_t n_ranges, const int64_t* off, const int64_t* len, int32_t* n_records, int32_t* regular) {
    cudaStream_t st = c->stream;
    *n_records = 0; *regular = 0;
    c->fa_recs.clear(); c->fa_bytes = 0;
    c->fasta_bytes = 0; c->vcf_bytes = 0;      // the image takes over the FASTA output buffer: earlier outputs are gone
    reads_invalidate(c);
    constexpr int64_t CH = ms_ctx::STAGE_BYTES;
    constexpr int NS = ms_ctx::N_STAGE;
    struct Chunk { int64_t foff, doff, n; };
    std::vector<Chunk> chunks;
    int64_t nbytes = 0;
    for (int32_t r = 0; r < n_ranges; ++r) {
        for (int64_t done = 0; done < len[r]; done += CH) {
            const int64_t n = len[r] - done < CH ? len[r] - done : CH;
            chunks.push_back(Chunk{off[r] + done, nbytes + done, n});
        }
        nbytes += len[r] > 0 ? len[r] : 0;
    }
    if (nbytes <= 0) return MS_OK;
    int rc = ensure_stage_buffers(c);
    if (rc) return rc;
    MS_CUDA(c, c->fasta.ensure((size_t)nbytes + 64));
    uint8_t* d_raw = c->fasta.as<uint8_t>();
    stage_begin(c, ST_UPLOAD);
    // page-cache reads manage a few GB/s per thread: NS reads are kept in flight, each into its own pinned buffer;
    // the H2D copies are issued in image order as the reads complete
    const int64_t nch = (int64_t)chunks.size();
    std::future<int> reader[NS];
    auto start_read = [&](int64_t i) {
        const int s = (int)(i % NS);
        const Chunk ck = chunks[(size_t)i];
        uint8_t* buf = c->h_stage[s];
        cudaEvent_t ev = c->h_stage_ev[s];
        const bool reuse = i >= NS;
        const int device = c->device;
        reader[s] = std::async(std::launch::async, [=]() -> int {
            if (reuse) { cudaSetDevice(device); if (cudaEventSynchronize(ev) != cudaSuccess) return EIO; }   // previous H2D out of this buffer
            return pread_all(fd, buf, ck.n, ck.foff);
        });
    };
    for (int64_t i = 0; i < nch && i < NS; ++i) start_read(i);
    int rerr = 0;
    for (int64_t i = 0; i < nch; ++i) {
        const int s = (int)(i % NS);
        const int e = reader[s].get();
        if (e && !rerr) rerr = e;
        if (!rerr) {
            const Chunk ck = chunks[(size_t)i];
            cudaError_t ce = cudaMemcpyAsync(d_raw + ck.doff, c->h_stage[s], (size_t)ck.n, cudaMemcpyHostToDevice, st);
            if (ce == cudaSuccess) ce = cudaEventRecord(c->h_stage_ev[s], st);
            if (ce != cudaSuccess) rerr = EIO;
        }
        if (!rerr && i + NS < nch) start_read(i + NS);
    }
    for (int s = 0; s < NS; ++s) if (reader[s].valid()) reader[s].get();
    if (rerr) MS_FAIL(c, MS_ERR_ARG, "ms_fasta_ingest_fd: read failed: %s", strerror(rerr));
    MS_CUDA(c, cudaMemsetAsync(d_raw + nbytes, '\n', 64, st));
    stage_end(c, ST_UPLOAD);

    // records
    MS_CUDA(c, c->scan_tmp2.ensure(64));
    unsigned long long* d_cnt = c->scan_tmp2.as<unsigned long long>();
    int* d_irr = reinterpret_cast<int*>(d_cnt + 1);
    MS_CUDA(c, cudaMemsetAsync(d_cnt, 0, 16, st));
    const unsigned grid = (unsigned)ceil_div(ceil_div(nbytes, 16), 256);
    k_fa_headers<<<grid, 256, 0, st>>>(d_raw, nbytes, d_cnt, nullptr, 0);
    MS_LAUNCH_CHECK(c);
    unsigned long long h_cnt = 0;
    MS_CUDA(c, cudaMemcpyAsync(&h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    if (h_cnt == 0 || h_cnt >= 0x7FFFFFF0ull) return MS_OK;          // no record (or absurdly many): host parser decides
    const int32_t n = (int32_t)h_cnt;
    MS_CUDA(c, c->svec.ensure((size_t)(n + 1) * 8));
    int64_t* d_hdr = c->svec.as<int64_t>();
    MS_CUDA(c, cudaMemsetAsync(d_cnt, 0, 8, st));
    k_fa_headers<<<grid, 256, 0, st>>>(d_raw, nbytes, d_cnt, d_hdr, n);
    MS_LAUNCH_CHECK(c);
    std::vector<int64_t> hdr((size_t)n);
    MS_CUDA(c, cudaMemcpyAsync(hdr.data(), d_hdr, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    std::sort(hdr.begin(), hdr.end());                                // slots were handed out in arrival order
    if (hdr[0] != 0) return MS_OK;                                    // text before the first record: host parser
    MS_CUDA(c, cudaMemcpyAsync(d_hdr, hdr.data(), (size_t)n * 8, cudaMemcpyHostToDevice, st));
    MS_CUDA(c, c->fa_index.ensure(sizeof(FaRec) * (size_t)n));
    k_fa_index<<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(d_raw, nbytes, d_hdr, n, c->fa_index.as<FaRec>(), d_irr);
    MS_LAUNCH_CHECK(c);
    c->fa_recs.resize((size_t)n);
    int h_irr = 0;
    MS_CUDA(c, cudaMemcpyAsync(c->fa_recs.data(), c->fa_index.p, sizeof(FaRec) * (size_t)n, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaMemcpyAsync(&h_irr, d_irr, 4, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    if (h_irr) { c->fa_recs.clear(); return MS_OK; }
    int64_t total = 0;
    for (FaRec& r : c->fa_recs) {
        if (r.len >= (int64_t)0x7FFFFFF0) { c->fa_recs.clear(); MS_FAIL(c, MS_ERR_LIMIT, "a record has %lld bases; this build supports < 2^31", (long long)r.len); }
        r.goff = total; total += r.len;
    }
    MS_CUDA(c, cudaMemcpyAsync(c->fa_index.p, c->fa_recs.data(), sizeof(FaRec) * (size_t)n, cudaMemcpyHostToDevice, st));
    c->fa_bytes = nbytes;
    *n_records = n; *regular = 1;
    return MS_OK;
}

int fasta_index(ms_ctx* c, int64_t* hdr_off, int64_t* seq_off, int64_t* length, int32_t* lenc, int32_t* lenb, uint8_t* hdr_blob,
                int64_t blob_cap) {
    const int32_t n = (int32_t)c->fa_recs.size();
    if (n == 0) MS_FAIL(c, MS_ERR_STATE, "ms_fasta_index: no ingested file");
    cudaStream_t st = c->stream;
    std::vector<int64_t> off((size_t)n + 1);
    off[0] = 0;
    for (int i = 0; i < n; ++i) {
        const FaRec& r = c->fa_recs[i];
        off[i + 1] = off[i] + (r.hdr_hi - r.hdr_lo - 1);
        hdr_off[i] = off[i];
        if (seq_off) seq_off[i] = r.seq_lo;
        if (length) length[i] = r.len;
        if (lenc) lenc[i] = r.lenc;
        if (lenb) lenb[i] = r.lenb;
    }
    hdr_off[n] = off[n];
    if (!hdr_blob) return MS_OK;                                      // sizes only
    if (off[n] > blob_cap) MS_FAIL(c, MS_ERR_ARG, "ms_fasta_index: defline buffer too small (need %lld bytes)", (long long)off[n]);
    MS_CUDA(c, c->scan_tmp.ensure((size_t)(n + 1) * 8));
    MS_CUDA(c, c->vvec.ensure((size_t)off[n] + 16));
    MS_CUDA(c, cudaMemcpyAsync(c->scan_tmp.p, off.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, st));
    k_fa_pack_headers<<<(unsigned)n, 64, 0, st>>>(c->fasta.as<uint8_t>(), c->fa_index.as<FaRec>(), n, c->scan_tmp.as<int64_t>(),
                                                   c->vvec.as<uint8_t>());
    MS_LAUNCH_CHECK(c);
    MS_CUDA(c, cudaMemcpyAsync(hdr_blob, c->vvec.p, (size_t)off[n], cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    return MS_OK;
}

// image -> resident bases; *regular = 0 if the bytes do not match the indexed layout (genome contents then undefined)
int fasta_strip(ms_ctx* c, int64_t total, int32_t* regular) {
    cudaStream_t st = c->stream;
    const int32_t n = (int32_t)c->fa_recs.size();
    int* d_irr = reinterpret_cast<int*>(c->scan_tmp2.as<unsigned long long>() + 1);
    MS_CUDA(c, cudaMemsetAsync(d_irr, 0, 4, st));
    if (total > 0) {
        k_fa_strip<<<(unsigned)ceil_div(ceil_div(total, 16), 256), 256, 0, st>>>(c->fasta.as<uint8_t>(), c->fa_index.as<FaRec>(), n, total,
                                                                                 c->genome.as<uint8_t>(), d_irr);
        MS_LAUNCH_CHECK(c);
    }
    int h_irr = 0;
    MS_CUDA(c, cudaMemcpyAsync(&h_irr, d_irr, 4, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    *regular = h_irr ? 0 : 1;
    return MS_OK;
}

}  // namespace ms
