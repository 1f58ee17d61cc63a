// ms_genotype.cu — polyploid runs (--ploidy): genotypes of the record table, haplotype selection and the phased VCF.
//   k_genotype   one thread per record of the full table draws its haplotype mask (ms_genotype_core.h) into buffer 8
//   select h     a scan over the flags "bit h-1 of the mask" compacts the full table into the active table (the second
//                record buffer); the literal pool is shared.  The plan pass reads the active table, so K5 / K6 / K8
//                see an ordinary table.  h = 0 swaps the full table back.
//   K7p          the phased VCF body of the full table into buffer 7: line sizes in closed form (K7's + 2 (P - 1)),
//                one scan for the offsets, then one thread per record writes its line with vcf_emit and a PhasedGt tail.
//                Reads genome, records, contigs and masks only, so it works the same in tile mode.
#include "ms_common.cuh"
#include "ms_scan.cuh"
#include "ms_genotype_core.h"

namespace ms {

namespace {

__global__ void __launch_bounds__(256)
k_genotype(const Rec* recs, int64_t n, const Contig* contigs, Seed seed, int ploidy, uint64_t thr, uint8_t* mask) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Rec r = recs[i];
    const Contig& c = contigs[r.contig];
    mask[i] = genotype_mask(seed, c.gid, genotype_key(c, r), ploidy, thr);
}

// off[c] = V[first record of contig c] (records sorted by contig), off[n_contigs] = V[n]
__global__ void __launch_bounds__(128)
k_phased_contig_off(const Rec* recs, int64_t n, int32_t n_contigs, const int64_t* V, int64_t* off) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > n_contigs) return;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (recs[mid].contig < (uint32_t)c) lo = mid + 1; else hi = mid;
    }
    off[c] = V[lo];
}

__global__ void k_store_i64(int64_t* dst, const int64_t* src) { *dst = *src; }

// K7p write pass: one thread per record writes its line at V[i] (V[i + 1] - V[i] bytes, none when omitted)
__global__ void __launch_bounds__(256)
k_vcf_phased_write(VcfView v, const Rec* recs, int64_t n, const Contig* contigs, const uint8_t* mask, int ploidy,
                   const int64_t* V, uint8_t* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || V[i + 1] == V[i]) return;
    const Rec r = recs[i];
    WriteSink s{out + V[i]};
    vcf_emit(s, v, contigs[r.contig], r, PhasedGt{mask[i], ploidy});
}

}  // namespace

void genotype_clear(ms_ctx* c) {
    c->gt_ploidy = 0;
    c->gt_selected = 0;
    c->gt_vcf_bytes = 0;
}

// make the full table the active one again
static void restore_full(ms_ctx* c) {
    if (!c->gt_selected) return;
    std::swap(c->recs, c->recs_full);
    c->n_recs = c->gt_n_full;
    c->gt_selected = 0;
    c->sizes_valid = c->gt_sizes_valid_full;
    c->counts_valid = false;
    c->rec_out_valid = true;
    chain_invalidate(c);
}

int genotype_draw(ms_ctx* c, uint64_t seed, int32_t ploidy, double hom_fraction) {
    if (ploidy < 2 || ploidy > MAX_PLOIDY) MS_FAIL(c, MS_ERR_ARG, "ms_genotype_draw: ploidy %d outside 2..%d", ploidy, MAX_PLOIDY);
    if (!(hom_fraction >= 0.0 && hom_fraction <= 1.0)) MS_FAIL(c, MS_ERR_ARG, "ms_genotype_draw: hom_fraction %g outside [0, 1]", hom_fraction);
    if (c->n_contigs <= 0) MS_FAIL(c, MS_ERR_STATE, "ms_genotype_draw: no genome resident");
    restore_full(c);
    const int64_t n = c->n_recs;
    MS_CUDA(c, c->gt_mask.ensure((size_t)n + 16));
    stage_begin(c, ST_GENOTYPE);
    if (n > 0) {
        k_genotype<<<(unsigned)ceil_div(n, 256), 256, 0, c->stream>>>(c->recs.as<Rec>(), n, c->contigs.as<Contig>(), make_seed(seed),
                                                                    ploidy, hom_threshold(hom_fraction), c->gt_mask.as<uint8_t>());
        MS_LAUNCH_CHECK(c);
    }
    stage_end(c, ST_GENOTYPE);
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    c->gt_ploidy = ploidy;
    c->gt_vcf_bytes = 0;
    return MS_OK;
}

int genotype_load(ms_ctx* c, const uint8_t* masks, int64_t n, int32_t ploidy) {
    if (ploidy < 2 || ploidy > MAX_PLOIDY) MS_FAIL(c, MS_ERR_ARG, "ms_genotype_load: ploidy %d outside 2..%d", ploidy, MAX_PLOIDY);
    restore_full(c);
    if (n != c->n_recs) MS_FAIL(c, MS_ERR_ARG, "ms_genotype_load: %lld masks for %lld records", (long long)n, (long long)c->n_recs);
    for (int64_t i = 0; i < n; ++i)
        if (masks[i] >> ploidy) MS_FAIL(c, MS_ERR_ARG, "ms_genotype_load: mask %lld (0x%x) has bits above ploidy %d", (long long)i, masks[i], ploidy);
    MS_CUDA(c, c->gt_mask.ensure((size_t)n + 16));
    if (n) MS_CUDA(c, cudaMemcpyAsync(c->gt_mask.p, masks, (size_t)n, cudaMemcpyHostToDevice, c->stream));
    MS_CUDA(c, cudaStreamSynchronize(c->stream));
    c->gt_ploidy = ploidy;
    c->gt_vcf_bytes = 0;
    return MS_OK;
}

int select_haplotype(ms_ctx* c, int32_t h) {
    if (!c->gt_ploidy) MS_FAIL(c, MS_ERR_STATE, "ms_select_haplotype: the record table has no genotypes (ms_genotype_draw / _load)");
    if (h < 0 || h > c->gt_ploidy) MS_FAIL(c, MS_ERR_ARG, "ms_select_haplotype: haplotype %d outside 0..%d", h, c->gt_ploidy);
    if (h == 0) { restore_full(c); return MS_OK; }
    cudaStream_t st = c->stream;
    if (!c->gt_selected) {
        int rc = fill_record_out(c);        // the full table keeps the Rec.out of its last apply
        if (rc) return rc;
        std::swap(c->recs, c->recs_full);
        c->gt_n_full = c->n_recs;
        c->gt_sizes_valid_full = c->sizes_valid;
    }
    const int64_t n = c->gt_n_full;
    MS_CUDA(c, c->recs.ensure((size_t)(n + 1) * sizeof(Rec)));
    const Rec* full = c->recs_full.as<Rec>();
    Rec* act = c->recs.as<Rec>();
    const uint8_t* mask = c->gt_mask.as<uint8_t>();
    const uint32_t bit = 1u << (h - 1);
    int64_t m = 0;
    stage_begin(c, ST_SELECT);
    if (n > 0) {
        auto in = [=] __device__(int64_t i) -> int64_t { return (mask[i] & bit) ? 1 : 0; };
        auto out = [=] __device__(int64_t i, int64_t ex, int64_t v) {
            if (!v) return;
            Rec r = full[i];
            r.out = 0;                   // the haplotype's own output positions come with its next apply
            act[ex] = r;
        };
        int64_t* d_total = nullptr;
        MS_CUDA(c, (device_scan<int64_t>(c, in, out, n, (int64_t)0, SumOp(), c->scan_tmp, &d_total)));
        MS_CUDA(c, cudaMemcpyAsync(&m, d_total, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    }
    stage_end(c, ST_SELECT);
    MS_CUDA(c, cudaStreamSynchronize(st));
    c->n_recs = m;
    c->gt_selected = h;
    c->sizes_valid = false;
    c->counts_valid = false;
    c->rec_out_valid = true;
    chain_invalidate(c);
    return MS_OK;
}

int vcf_phased(ms_ctx* c, int64_t* vcf_off) {
    if (!c->gt_ploidy) MS_FAIL(c, MS_ERR_STATE, "ms_vcf_phased: the record table has no genotypes (ms_genotype_draw / _load)");
    const int P = c->gt_ploidy;
    const int64_t n = c->gt_selected ? c->gt_n_full : c->n_recs;
    const Rec* recs = (c->gt_selected ? c->recs_full : c->recs).as<Rec>();
    const uint8_t* mask = c->gt_mask.as<uint8_t>();
    const Contig* contigs = c->contigs.as<Contig>();
    const int32_t nc = c->n_contigs;
    cudaStream_t st = c->stream;
    const Tables* d_tab = c->tables.as<Tables>();
    const VcfView vv{c->genome.as<uint8_t>(), c->lit.as<uint8_t>(), c->names.as<uint8_t>(), d_tab->conv, d_tab->comp, c->seed_last};
    MS_CUDA(c, c->gt_voff.ensure((size_t)(n + 1) * sizeof(int64_t)));
    MS_CUDA(c, c->gt_ctg_off.ensure((size_t)(nc + 1) * sizeof(int64_t)));
    int64_t* V = c->gt_voff.as<int64_t>();
    stage_begin(c, ST_VCF_PHASED);
    {
        auto in = [=] __device__(int64_t i) -> int64_t {
            const Rec r = recs[i];
            return (int64_t)phased_line_size(vv, contigs[r.contig], r, P);
        };
        auto out = [=] __device__(int64_t i, int64_t ex, int64_t) { V[i] = ex; };
        int64_t* d_total = nullptr;
        MS_CUDA(c, (device_scan<int64_t>(c, in, out, n, (int64_t)0, SumOp(), c->scan_tmp, &d_total)));
        k_store_i64<<<1, 1, 0, st>>>(V + n, d_total);
        MS_LAUNCH_CHECK(c);
    }
    int64_t total = 0;
    MS_CUDA(c, cudaMemcpyAsync(&total, V + n, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    MS_CUDA(c, c->gt_vcf.ensure((size_t)total + 64));
    if (n > 0) {
        k_vcf_phased_write<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(vv, recs, n, contigs, mask, P, V, c->gt_vcf.as<uint8_t>());
        MS_LAUNCH_CHECK(c);
    }
    k_phased_contig_off<<<(unsigned)ceil_div(nc + 1, 128), 128, 0, st>>>(recs, n, nc, V, c->gt_ctg_off.as<int64_t>());
    MS_LAUNCH_CHECK(c);
    MS_CUDA(c, cudaMemcpyAsync(vcf_off, c->gt_ctg_off.p, (size_t)(nc + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    stage_end(c, ST_VCF_PHASED);
    MS_CUDA(c, cudaStreamSynchronize(st));
    c->gt_vcf_bytes = total;
    return MS_OK;
}

}  // namespace ms
