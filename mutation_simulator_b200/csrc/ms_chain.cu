// ms_chain.cu — K8: the UCSC chain file from the input genome to the mutated genome of the last apply
// (ms_chain_count / ms_chain_write).  Reads the SvRec stream, the contig table and the names blob; no genome bytes.
//   count  one thread per contig finds its first and last block; one scan over the SvRecs sums cons (the score) and
//          numbers the copy records (their chain ids); one thread per contig collects both
//   write  work items (ms_chain_core.h) are sized by the emitter with a counting sink, one scan places them, and the
//          down-sweep writes them with the same emitter into buffer 6
#include "ms_common.cuh"
#include "ms_scan.cuh"
#include "ms_chain_core.h"

namespace ms {

namespace {

__global__ void __launch_bounds__(128)
k_chain_contigs(const Contig* contigs, int32_t n_contigs, const uint32_t* N, const SvRec* sv, ChainCtg* cc) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_contigs) return;
    const Contig k = contigs[c];
    ChainCtg x{};
    x.n_lo = (int64_t)N[k.rec_lo];
    x.n_hi = (int64_t)N[k.rec_hi];
    x.item_lo = 2 * x.n_lo + 2 * (int64_t)c;
    chain_bounds(sv, k, x);
    cc[c] = x;
}

__global__ void __launch_bounds__(128)
k_chain_finish(const Contig* contigs, int32_t n_contigs, const int64_t* cons_pre, const uint32_t* copy_pre, ChainCtg* cc) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_contigs) return;
    ChainCtg& x = cc[c];
    x.score = (uint32_t)(contigs[c].len - (cons_pre[x.n_hi] - cons_pre[x.n_lo]));
    x.n_copies = copy_pre[x.n_hi] - copy_pre[x.n_lo];
}

// A copy chain's source must lie inside its own contig: the first copy record whose source leaves it goes to
// err = {MS_ERR_ARG, its SvRec slot}.
__global__ void __launch_bounds__(256)
k_chain_check(const Contig* contigs, int32_t n_contigs, const ChainCtg* cc, const SvRec* sv, int64_t n_sv, unsigned long long* err) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_sv) return;
    const SvRec r = sv[i];
    if (!chain_copy(r)) return;
    int32_t lo = 0, hi = n_contigs;              // the last contig with n_lo <= i holds slot i
    while (hi - lo > 1) { const int32_t mid = (lo + hi) >> 1; if (cc[mid].n_lo <= i) lo = mid; else hi = mid; }
    const int64_t s = r.src - contigs[lo].goff;
    if (s < 0 || s + (int64_t)r.prod > contigs[lo].len)
        if (atomicCAS(&err[0], 0ull, (unsigned long long)MS_ERR_ARG) == 0ull) err[1] = (unsigned long long)i;
}

__global__ void k_chain_totals(const I64x2* total, int64_t n, int64_t* cons_pre, uint32_t* copy_pre) {
    cons_pre[n] = total->a;
    copy_pre[n] = (uint32_t)total->b;
}

// Down-sweep of the write scan, written for its type: a thread owns SCAN_ITEMS consecutive items, sizes them again
// with the counting sink, and writes each at its offset with the writing sink.  A contig's first item records where
// the contig's slice starts.
__global__ void __launch_bounds__(SCAN_THREADS)
k_chain_down(ChainView v, int64_t n_items, const int64_t* __restrict__ tile_prefix, uint8_t* __restrict__ out,
             int64_t* __restrict__ ctg_off) {
    __shared__ int64_t sm[2 * SCAN_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int32_t c0 = base < n_items ? chain_item_contig(v.cc, v.n_contigs, base) : 0;
    uint32_t sz[SCAN_ITEMS];
    int64_t acc = 0;
    {
        int32_t c = c0;
#pragma unroll
        for (int j = 0; j < SCAN_ITEMS; ++j) {
            const int64_t x = base + j;
            sz[j] = 0u;
            if (x < n_items) {
                while (c + 1 < v.n_contigs && v.cc[c + 1].item_lo <= x) ++c;
                sz[j] = chain_item_size(v, c, x);
            }
            acc += sz[j];
        }
    }
    int64_t total;
    const int64_t ex = block_excl_scan(acc, (int64_t)0, SumOp(), total, sm);
    int64_t run = tile_prefix[blockIdx.x] + ex;
    int32_t c = c0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        const int64_t x = base + j;
        if (x < n_items) {
            while (c + 1 < v.n_contigs && v.cc[c + 1].item_lo <= x) ++c;
            if (x == v.cc[c].item_lo) ctg_off[c] = run;
            if (sz[j]) {
                WriteSink s{out + run};
                chain_item(s, v, c, x);
            }
        }
        run += sz[j];
    }
}

}  // namespace

// (an apply output stops being current here, so the reads of a full apply go too)
void chain_invalidate(ms_ctx* c) { c->chain_ready = false; c->chain_counted = false; c->chain_bytes = 0; reads_invalidate(c); }

int chain_count(ms_ctx* c, int64_t* n_chains) {
    if (!c->chain_ready) MS_FAIL(c, MS_ERR_STATE, "ms_chain_count: no ms_apply / ms_apply_window output to describe");
    const int32_t n = c->n_contigs;
    const int64_t n_sv = c->n_sv;
    cudaStream_t st = c->stream;
    stage_begin(c, ST_CHAIN);
    MS_CUDA(c, c->chain_cc.ensure(sizeof(ChainCtg) * (size_t)n));
    MS_CUDA(c, c->chain_cons.ensure((size_t)(n_sv + 1) * sizeof(int64_t)));
    MS_CUDA(c, c->chain_copy.ensure((size_t)(n_sv + 1) * sizeof(uint32_t)));
    MS_CUDA(c, c->chain_err.ensure(16));
    MS_CUDA(c, cudaMemsetAsync(c->chain_err.p, 0, 16, st));
    ChainCtg* d_cc = c->chain_cc.as<ChainCtg>();
    const Contig* d_contigs = c->contigs.as<Contig>();
    const SvRec* sv = c->sv_stream.as<SvRec>();
    int64_t* cons_pre = c->chain_cons.as<int64_t>();
    uint32_t* copy_pre = c->chain_copy.as<uint32_t>();
    unsigned long long* err = c->chain_err.as<unsigned long long>();
    k_chain_contigs<<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(d_contigs, n, c->nvec.as<uint32_t>(), sv, d_cc);
    MS_LAUNCH_CHECK(c);
    {
        auto in = [=] __device__(int64_t i) -> I64x2 {
            const SvRec r = sv[i];
            return I64x2{(int64_t)(r.run_in - r.pos), chain_copy(r) ? 1 : 0};
        };
        auto out = [=] __device__(int64_t i, I64x2 ex, I64x2) { cons_pre[i] = ex.a; copy_pre[i] = (uint32_t)ex.b; };
        I64x2* d_total = nullptr;
        MS_CUDA(c, (device_scan<I64x2>(c, in, out, n_sv, I64x2{0, 0}, SumOp(), c->scan_tmp, &d_total)));
        k_chain_totals<<<1, 1, 0, st>>>(d_total, n_sv, cons_pre, copy_pre);
        MS_LAUNCH_CHECK(c);
    }
    k_chain_finish<<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(d_contigs, n, cons_pre, copy_pre, d_cc);
    MS_LAUNCH_CHECK(c);
    if (n_sv > 0) {
        k_chain_check<<<(unsigned)ceil_div(n_sv, 256), 256, 0, st>>>(d_contigs, n, d_cc, sv, n_sv, err);
        MS_LAUNCH_CHECK(c);
    }
    c->h_chain_cc.resize((size_t)n);
    int64_t h_err[2];
    MS_CUDA(c, cudaMemcpyAsync(c->h_chain_cc.data(), d_cc, sizeof(ChainCtg) * (size_t)n, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaMemcpyAsync(h_err, err, 16, cudaMemcpyDeviceToHost, st));
    stage_end(c, ST_CHAIN);
    MS_CUDA(c, cudaStreamSynchronize(st));
    if (h_err[0]) {
        const int64_t slot = h_err[1];
        int32_t ctg = 0;
        while (ctg + 1 < n && c->h_chain_cc[ctg + 1].n_lo <= slot) ++ctg;
        SvRec r;
        MS_CUDA(c, cudaMemcpy(&r, sv + slot, sizeof(SvRec), cudaMemcpyDeviceToHost));
        MS_FAIL(c, MS_ERR_ARG, "ms_chain_count: the record at position %u of contig %d copies bases from outside its contig "
                "(source %lld, %u bases)", r.pos, ctg, (long long)r.src, r.prod);
    }
    for (int32_t i = 0; i < n; ++i) {
        const ChainCtg& x = c->h_chain_cc[i];
        n_chains[i] = (int64_t)x.primary + (int64_t)x.n_copies;
    }
    c->chain_counted = true;
    return MS_OK;
}

int chain_write(ms_ctx* c, const int64_t* first_id, int64_t* chain_off) {
    if (!c->chain_ready) MS_FAIL(c, MS_ERR_STATE, "ms_chain_write: no ms_apply / ms_apply_window output to describe");
    const int32_t n = c->n_contigs;
    if (!c->chain_counted) {
        std::vector<int64_t> tmp((size_t)n);
        const int rc = chain_count(c, tmp.data());
        if (rc) return rc;
    }
    for (int32_t i = 0; i < n; ++i) {
        ChainCtg& x = c->h_chain_cc[i];
        const int64_t chains = (int64_t)x.primary + (int64_t)x.n_copies;
        if (first_id[i] < 1) MS_FAIL(c, MS_ERR_ARG, "ms_chain_write: first_id[%d] = %lld; chain ids start at 1", i, (long long)first_id[i]);
        if (chains && first_id[i] + chains - 1 >= (int64_t)0x80000000ll)
            MS_FAIL(c, MS_ERR_LIMIT, "ms_chain_write: chain ids of contig %d reach %lld; ids must stay below 2^31", i,
                    (long long)(first_id[i] + chains - 1));
        x.first_id = first_id[i];
    }
    cudaStream_t st = c->stream;
    ChainCtg* d_cc = c->chain_cc.as<ChainCtg>();
    stage_begin(c, ST_CHAIN);
    MS_CUDA(c, cudaMemcpyAsync(d_cc, c->h_chain_cc.data(), sizeof(ChainCtg) * (size_t)n, cudaMemcpyHostToDevice, st));
    const ChainView v{c->sv_stream.as<SvRec>(), c->contigs.as<Contig>(), c->names.as<uint8_t>(), d_cc,
                      c->chain_copy.as<uint32_t>(), n};
    const int64_t n_items = 2 * c->n_sv + 2 * (int64_t)n;
    auto in = [=] __device__(int64_t x) -> int64_t { return (int64_t)chain_item_size(v, chain_item_contig(v.cc, v.n_contigs, x), x); };
    int64_t* tile_prefix = nullptr;
    int64_t nt = 0;
    MS_CUDA(c, (scan_tile_sums<int64_t>(c, in, n_items, (int64_t)0, SumOp(), c->scan_tmp, &tile_prefix, &nt)));
    int64_t total = 0;
    MS_CUDA(c, cudaMemcpyAsync(&total, tile_prefix + nt, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    MS_CUDA(c, c->chain.ensure((size_t)total + 64));
    MS_CUDA(c, c->chain_off.ensure((size_t)(n + 1) * sizeof(int64_t)));
    if (nt > 0) {
        k_chain_down<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(v, n_items, tile_prefix, c->chain.as<uint8_t>(), c->chain_off.as<int64_t>());
        MS_LAUNCH_CHECK(c);
    }
    MS_CUDA(c, cudaMemcpyAsync(chain_off, c->chain_off.p, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    stage_end(c, ST_CHAIN);
    MS_CUDA(c, cudaStreamSynchronize(st));
    chain_off[n] = total;
    c->chain_bytes = total;
    return MS_OK;
}

}  // namespace ms
