// ms_reads.cu — paired-end reads from the mutated genome of the last full ms_apply (ms_reads_size / ms_reads_write).
// Reads buffer 0 (the FASTA image), the active record table with its out positions and the contig table.
//   size   one thread per pair draws (s, f, strand, attempt) with the A/C/G/T check of its two template ends, lifts
//          x1 and x2 by a binary search over its contig's records and sizes the record (PairInfo, kept for the write);
//          one scan places the records, one thread per contig sums its bytes in the range
//   write  one warp per pair: lane 0 writes the two name lines, the lanes copy (and complement) the template bases
//          four at a time, one Philox block per four error words, and fill the quality lines; R1 records go to
//          [0, n) of buffer 9 and R2 records to [n, 2n)
#include "ms_common.cuh"
#include "ms_scan.cuh"
#include "ms_reads_core.h"

namespace ms {

namespace {

constexpr int SIZE_THREADS = 256;
constexpr int WRITE_THREADS = 256;

// contig of global pair j: the last c with pre[c] <= j (empty contigs share their pre with the next one)
__device__ __forceinline__ int32_t pair_contig(const int64_t* pre, int32_t n_contigs, int64_t j) {
    int32_t lo = 0, hi = n_contigs;
    while (hi - lo > 1) { const int32_t mid = (lo + hi) >> 1; if (pre[mid] <= j) lo = mid; else hi = mid; }
    return lo;
}

__global__ void __launch_bounds__(SIZE_THREADS)
k_reads_size(ReadsCfg g, const uint8_t* __restrict__ img, const Rec* __restrict__ recs, const Contig* __restrict__ contigs,
             const int64_t* __restrict__ pre, int32_t n_contigs, int64_t first, int64_t count, PairInfo* __restrict__ info) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const int64_t j = first + t;
    const int32_t c = pair_contig(pre, n_contigs, j);
    const Contig& k = contigs[c];
    const uint32_t i = (uint32_t)(j - pre[c]);
    PairInfo p = pair_info(g, img, recs, k, i);
    p.size = read_record_size(k, g.hap, i, p, g.L);
    info[t] = p;
}

__global__ void k_reads_total(const int64_t* total, int64_t count, int64_t* off) { off[count] = *total; }

// bytes of the range's records in each contig
__global__ void __launch_bounds__(128)
k_reads_ctg_bytes(const int64_t* pre, int32_t n_contigs, int64_t first, int64_t count, const int64_t* off, int64_t* bytes) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_contigs) return;
    const int64_t lo = min(max(pre[c] - first, (int64_t)0), count), hi = min(max(pre[c + 1] - first, (int64_t)0), count);
    bytes[c] = off[hi] - off[lo];
}

__global__ void __launch_bounds__(WRITE_THREADS)
k_reads_write(ReadsCfg g, const uint8_t* __restrict__ img, const uint8_t* __restrict__ comp, const uint8_t* __restrict__ names,
              const Contig* __restrict__ contigs, const int64_t* __restrict__ pre, int32_t n_contigs, int64_t first, int64_t count,
              const PairInfo* __restrict__ info, const int64_t* __restrict__ off, uint8_t* __restrict__ out) {
    const int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (t >= count) return;
    const int64_t j = first + t;
    const int32_t c = pair_contig(pre, n_contigs, j);
    const Contig& k = contigs[c];
    const uint32_t i = (uint32_t)(j - pre[c]);
    const PairInfo p = info[t];
    const int32_t L = g.L;
    const uint32_t hdr = p.size - 2u * (uint32_t)L - 4u;
    uint8_t* r1 = out + off[t];
    uint8_t* r2 = r1 + off[count];
    if (lane == 0) {
        WriteSink s1{r1}, s2{r2};
        read_header(s1, names, k, g.hap, i, p, '1');
        read_header(s2, names, k, g.hap, i, p, '2');
    }
    // the 2L bases of R1 then R2 as one sequence: base x uses error word 16 + x = component x % 4 of block 4 + x / 4
    const uint32_t a = (p.meta >> 1) & 7u;
    for (int32_t q = lane; 4 * q < 2 * L; q += 32) {
        const U4 blk = reads_block(g, k.gid, i, a, 4u + (uint32_t)q);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int32_t x = 4 * q + u;
            if (x >= 2 * L) break;
            const int mate = x < L ? 1 : 2;
            const int32_t b = x < L ? x : x - L;
            const uint8_t base = read_error(read_template_base(img, comp, k, p, L, mate, b), u4_word(blk, (uint32_t)u), g.err_thr);
            (mate == 1 ? r1 : r2)[hdr + b] = base;
        }
    }
    for (int32_t b = lane; b < L + 4; b += 32) {
        // "\n+\n" after the bases, then L quality characters and '\n'
        const uint8_t ch = b < 3 ? (uint8_t)"\n+\n"[b] : b < L + 3 ? g.qual : (uint8_t)'\n';
        r1[hdr + L + b] = ch;
        r2[hdr + L + b] = ch;
    }
}

// the checks both entry points share; fills *g and uploads the prefix of n_pairs
int reads_prepare(ms_ctx* c, const ms_reads_cfg* cfg, const int64_t* n_pairs, int64_t first, int64_t count, ReadsCfg* g,
                  const char* who) {
    if (!c->apply_full) MS_FAIL(c, MS_ERR_STATE, "%s: no full ms_apply output is current", who);
    if (cfg->hap < 1 || cfg->hap > 8 || cfg->read_len < 1 || cfg->read_len > READS_MAX_LEN || cfg->frag_mean < cfg->read_len ||
        cfg->frag_mean > READS_MAX_FRAG_MEAN || cfg->frag_sd < 0 || cfg->frag_sd > READS_MAX_FRAG_SD ||
        !(cfg->error_rate >= 0.0 && cfg->error_rate < 1.0) || cfg->qual < 33 || cfg->qual > 126)
        MS_FAIL(c, MS_ERR_ARG, "%s: configuration outside its ranges (hap 1..8, read_len 1..%d, frag_mean read_len..%d, "
                "frag_sd 0..%d, 0 <= error_rate < 1, qual 33..126)", who, READS_MAX_LEN, READS_MAX_FRAG_MEAN, READS_MAX_FRAG_SD);
    const int32_t n = c->n_contigs;
    MS_CUDA(c, cudaMemcpy(c->h_contigs.data(), c->contigs.p, sizeof(Contig) * (size_t)n, cudaMemcpyDeviceToHost));
    c->h_reads_pre.assign((size_t)n + 1, 0);
    for (int32_t i = 0; i < n; ++i) {
        if (n_pairs[i] < 0) MS_FAIL(c, MS_ERR_ARG, "%s: n_pairs[%d] is negative", who, i);
        if (n_pairs[i] > 0 && c->h_contigs[i].out_len < cfg->read_len)
            MS_FAIL(c, MS_ERR_ARG, "%s: contig %d has %lld mutated bases, fewer than one read", who, i,
                    (long long)c->h_contigs[i].out_len);
        if (n_pairs[i] > (int64_t)0xFFFFFFFFll) MS_FAIL(c, MS_ERR_LIMIT, "%s: contig %d has 2^32 pairs or more", who, i);
        c->h_reads_pre[i + 1] = c->h_reads_pre[i] + n_pairs[i];
    }
    if (first < 0 || count < 0 || first + count > c->h_reads_pre[n])
        MS_FAIL(c, MS_ERR_ARG, "%s: pairs [%lld, %lld) outside the %lld pairs", who, (long long)first, (long long)(first + count),
                (long long)c->h_reads_pre[n]);
    *g = ReadsCfg{make_seed(cfg->seed), (uint32_t)cfg->hap, cfg->read_len, cfg->frag_mean, cfg->frag_sd,
                  read_error_threshold(cfg->error_rate), cfg->qual};
    MS_CUDA(c, c->reads_pre.ensure(sizeof(int64_t) * ((size_t)n + 1)));
    MS_CUDA(c, cudaMemcpyAsync(c->reads_pre.p, c->h_reads_pre.data(), sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice,
                               c->stream));
    return fill_record_out(c);
}

// the size pass into reads_info / reads_off (count + 1 offsets); *total = bytes of one file
int reads_size_pass(ms_ctx* c, const ReadsCfg& g, int64_t first, int64_t count, int64_t* total) {
    cudaStream_t st = c->stream;
    const int32_t n = c->n_contigs;
    MS_CUDA(c, c->reads_info.ensure(sizeof(PairInfo) * ((size_t)count + 1)));
    MS_CUDA(c, c->reads_off.ensure(sizeof(int64_t) * ((size_t)count + 1)));
    PairInfo* info = c->reads_info.as<PairInfo>();
    int64_t* off = c->reads_off.as<int64_t>();
    if (count > 0) {
        k_reads_size<<<(unsigned)ceil_div(count, SIZE_THREADS), SIZE_THREADS, 0, st>>>(
            g, c->fasta.as<uint8_t>(), c->recs.as<Rec>(), c->contigs.as<Contig>(), c->reads_pre.as<int64_t>(), n, first, count, info);
        MS_LAUNCH_CHECK(c);
        auto in = [=] __device__(int64_t x) -> int64_t { return (int64_t)info[x].size; };
        auto out = [=] __device__(int64_t x, int64_t ex, int64_t) { off[x] = ex; };
        int64_t* d_total = nullptr;
        MS_CUDA(c, (device_scan<int64_t>(c, in, out, count, (int64_t)0, SumOp(), c->scan_tmp, &d_total)));
        k_reads_total<<<1, 1, 0, st>>>(d_total, count, off);
        MS_LAUNCH_CHECK(c);
    } else {
        MS_CUDA(c, cudaMemsetAsync(off, 0, sizeof(int64_t), st));
    }
    MS_CUDA(c, cudaMemcpyAsync(total, off + count, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    return MS_OK;
}

// reads_info / reads_off now hold the draws of this range
void remember_range(ms_ctx* c, const ReadsCfg& g, int64_t first, int64_t count, int64_t total) {
    c->reads_cfg = g; c->reads_first = first; c->reads_count = count; c->reads_sized_pre = c->h_reads_pre;
    c->reads_sized = true; c->reads_sized_total = total;
}

bool same_range(const ms_ctx* c, const ReadsCfg& g, int64_t first, int64_t count) {
    const ReadsCfg& s = c->reads_cfg;
    return c->reads_sized && s.seed.k0 == g.seed.k0 && s.seed.k1 == g.seed.k1 && s.hap == g.hap && s.L == g.L && s.M == g.M &&
           s.S == g.S && s.err_thr == g.err_thr && s.qual == g.qual && c->reads_first == first && c->reads_count == count &&
           c->reads_sized_pre == c->h_reads_pre;
}

}  // namespace

void reads_invalidate(ms_ctx* c) { c->apply_full = false; c->reads_sized = false; c->reads_bytes = 0; }

int reads_size(ms_ctx* c, const ms_reads_cfg* cfg, const int64_t* n_pairs, int64_t first, int64_t count, int64_t* bytes) {
    ReadsCfg g;
    int rc = reads_prepare(c, cfg, n_pairs, first, count, &g, "ms_reads_size");
    if (rc) return rc;
    const int32_t n = c->n_contigs;
    stage_begin(c, ST_READS);
    int64_t total = 0;
    if ((rc = reads_size_pass(c, g, first, count, &total))) return rc;
    MS_CUDA(c, c->reads_ctg.ensure(sizeof(int64_t) * (size_t)n));
    k_reads_ctg_bytes<<<(unsigned)ceil_div(n, 128), 128, 0, c->stream>>>(c->reads_pre.as<int64_t>(), n, first, count,
                                                                        c->reads_off.as<int64_t>(), c->reads_ctg.as<int64_t>());
    MS_LAUNCH_CHECK(c);
    MS_CUDA(c, cudaMemcpyAsync(bytes, c->reads_ctg.p, sizeof(int64_t) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    stage_end(c, ST_READS);
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    remember_range(c, g, first, count, total);
    return MS_OK;
}

int reads_write(ms_ctx* c, const ms_reads_cfg* cfg, const int64_t* n_pairs, int64_t first, int64_t count, int64_t* nbytes) {
    ReadsCfg g;
    int rc = reads_prepare(c, cfg, n_pairs, first, count, &g, "ms_reads_write");
    if (rc) return rc;
    cudaStream_t st = c->stream;
    stage_begin(c, ST_READS);
    int64_t total = c->reads_sized_total;
    if (!same_range(c, g, first, count)) {      // not the range of the last ms_reads_size: draw and size it here
        c->reads_sized = false;
        if ((rc = reads_size_pass(c, g, first, count, &total))) return rc;
        MS_CUDA(c, cudaStreamSynchronize(st));
        remember_range(c, g, first, count, total);
    }
    c->reads_bytes = 0;
    MS_CUDA(c, c->reads.ensure(2 * (size_t)total + 64));
    if (count > 0) {
        const Tables* d_tab = c->tables.as<Tables>();
        k_reads_write<<<(unsigned)ceil_div(count * 32, WRITE_THREADS), WRITE_THREADS, 0, st>>>(
            g, c->fasta.as<uint8_t>(), d_tab->comp, c->names.as<uint8_t>(), c->contigs.as<Contig>(), c->reads_pre.as<int64_t>(),
            c->n_contigs, first, count, c->reads_info.as<PairInfo>(), c->reads_off.as<int64_t>(), c->reads.as<uint8_t>());
        MS_LAUNCH_CHECK(c);
    }
    stage_end(c, ST_READS);
    MS_CUDA(c, cudaStreamSynchronize(st));
    c->reads_bytes = 2 * total;
    *nbytes = total;
    return MS_OK;
}

}  // namespace ms
