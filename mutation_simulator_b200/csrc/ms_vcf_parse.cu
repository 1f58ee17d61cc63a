// ms_vcf_parse.cu — VCF replay input parsed on the device (ms_load_vcf): what records.py:119-191 records_from_vcf +
// ms_load_records do, for the regular shape of ms_vcf_parse_core.h (every VCF the reference or this package writes).
//
// text -> device (chunked copies) -> line starts (one scan over 16-byte groups, which also flags the bytes that
// str.splitlines() would break at) -> one thread per line parses it into a Rec (ms_vcf_parse_core.h) -> one scan over
// the lines compacts the records in file order and lays the inserted bytes out as the literal pool, in file order too
// -> every contig must form one block of lines with increasing POS; a scan over the blocks' lengths in contig order
// places them, which is what the host's stable sort by (contig, pos) gives for such files -> the checks of
// ms_load_records (rec_fault) on the finished table.  Anything irregular ends the call with *regular = 0 and the
// context untouched; the caller then runs the host parser, which owns the error messages.
#include <algorithm>
#include <utility>
#include "ms_common.cuh"
#include "ms_scan.cuh"
#include "ms_vcf_parse_core.h"

namespace ms {
using namespace vcfp;

constexpr int64_t VCF_COPY_CHUNK = 64 << 20;

// line starts in bytes [16 g, 16 g + 16): offset 0, and each byte after a '\n' that is not past the end.
// dst == nullptr: count only; else write them from dst on and raise *irregular on a byte splitlines() breaks at.
__device__ __forceinline__ int64_t group_line_starts(const uint8_t* t, int64_t n, int64_t g, int64_t* dst, int* irregular) {
    const int64_t i0 = g * 16;
    const uint4 v = *reinterpret_cast<const uint4*>(t + i0);   // the text is padded with zeros to a multiple of 16
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    int64_t cnt = 0;
    if (g == 0) { if (dst) dst[cnt] = 0; ++cnt; }
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const uint8_t b = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
        if (b == '\n' && i0 + k + 1 < n) { if (dst) dst[cnt] = i0 + k + 1; ++cnt; }
        bad |= irregular_byte(b);
    }
    if (dst && bad) *irregular = 1;
    return cnt;
}

// one thread per line; lines[k] .. lines[k + 1] - 1 is line k without its '\n'.  Skipped lines become T_DEAD.
__global__ void __launch_bounds__(256)
k_vcf_parse_lines(const uint8_t* t, const int64_t* lines, int64_t n_lines, NameTable names, int skip_unknown, Rec* lrec,
                  int* irregular) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_lines) return;
    Rec r{};
    const int kind = parse_line(t, lines[k], lines[k + 1] - 1, names, skip_unknown, &r);
    if (kind == VL_IRREGULAR) *irregular = 1;
    if (kind != VL_REC) r.type = T_DEAD;
    lrec[k] = r;
}

// every contig's records form one block (first[c], last[c]) of increasing POS (held in Rec.out)
__global__ void __launch_bounds__(256)
k_vcf_blocks(const Rec* krec, int64_t m, int64_t* first, int64_t* last, int32_t* nblk, int* irregular) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t c = krec[j].contig;
    if (j == 0 || krec[j - 1].contig != c) {
        if (atomicAdd(&nblk[c], 1) != 0) *irregular = 1;   // the contig's lines are split over two blocks
        first[c] = j;
    } else if (krec[j].out <= krec[j - 1].out) {
        *irregular = 1;
    }
    if (j == m - 1 || krec[j + 1].contig != c) last[c] = j + 1;
}

// record j of block c goes to slot base[c] + j (base[c] = records of the contigs before c - first[c])
__global__ void __launch_bounds__(256) k_vcf_place(const Rec* krec, int64_t m, const int64_t* base, Rec* recs) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    Rec r = krec[j];
    r.out = 0;
    recs[base[r.contig] + j] = r;
}

// ms_load_vcf_phased: the haplotype mask of every record line from its GT field (other lines keep 0)
__global__ void __launch_bounds__(256)
k_vcf_parse_gt(const uint8_t* t, const int64_t* lines, int64_t n_lines, const Rec* lrec, int ploidy, uint8_t* lmask, int* irregular) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_lines) return;
    uint8_t m = 0;
    if (lrec[k].type != T_DEAD && !parse_gt(t, lines[k], lines[k + 1] - 1, ploidy, &m)) *irregular = 1;
    lmask[k] = m;
}

// the masks follow their records to the table order of k_vcf_place
__global__ void __launch_bounds__(256) k_vcf_place_mask(const Rec* krec, const uint8_t* kmask, int64_t m, const int64_t* base, uint8_t* mask) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    mask[base[krec[j].contig] + j] = kmask[j];
}

// the first record that fails a check of ms_load_records: (index << 3) | RecFault
__global__ void __launch_bounds__(256)
k_vcf_faults(const Rec* recs, int64_t m, int32_t n_contigs, int64_t lit_bytes, int64_t src_end, unsigned long long* first) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const int f = rec_fault(recs, j, n_contigs, lit_bytes, src_end);
    if (f) atomicMin(first, ((unsigned long long)j << 3) | (unsigned long long)f);
}

int vcf_load(ms_ctx* c, const uint8_t* text, int64_t n, int32_t skip_unknown, int32_t ploidy, int32_t* regular, int64_t* n_recs) {
    cudaStream_t st = c->stream;
    const int32_t nc = c->n_contigs;

    // CHROM -> contig: the names k_vcf_write writes (the device blob), hashed on the host
    int64_t blob = 0;
    std::vector<VcfContig> vc((size_t)nc);
    for (int32_t i = 0; i < nc; ++i) {
        const Contig& k = c->h_contigs[i];
        vc[i] = VcfContig{k.name_src, k.goff, k.name_len, (int32_t)k.len};
        blob = std::max(blob, k.name_src + k.name_len);
    }
    std::vector<uint8_t> h_names((size_t)blob + 1);
    if (blob) MS_CUDA(c, cudaMemcpyAsync(h_names.data(), c->names.p, (size_t)blob, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    const uint32_t tsize = table_size(nc);
    std::vector<int32_t> slot(tsize);
    build_table(h_names.data(), vc.data(), nc, slot.data(), tsize);
    const size_t slot_bytes = ((size_t)tsize * 4 + 15) & ~(size_t)15;
    MS_CUDA(c, c->vp_names.ensure(slot_bytes + sizeof(VcfContig) * (size_t)nc));
    int32_t* d_slot = c->vp_names.as<int32_t>();
    VcfContig* d_vc = reinterpret_cast<VcfContig*>(c->vp_names.as<uint8_t>() + slot_bytes);
    MS_CUDA(c, cudaMemcpyAsync(d_slot, slot.data(), (size_t)tsize * 4, cudaMemcpyHostToDevice, st));
    MS_CUDA(c, cudaMemcpyAsync(d_vc, vc.data(), sizeof(VcfContig) * (size_t)nc, cudaMemcpyHostToDevice, st));
    const NameTable names{d_slot, tsize - 1, c->names.as<uint8_t>(), d_vc};

    // scalars (irregular flag, first fault) and per-contig block bounds
    MS_CUDA(c, c->vp_contig.ensure(64 + (size_t)nc * (3 * 8 + 4)));
    int* d_irr = c->vp_contig.as<int>();
    unsigned long long* d_fault = reinterpret_cast<unsigned long long*>(c->vp_contig.as<uint8_t>() + 8);
    int64_t* d_first = reinterpret_cast<int64_t*>(c->vp_contig.as<uint8_t>() + 64);
    int64_t* d_last = d_first + nc;
    int64_t* d_base = d_last + nc;
    int32_t* d_nblk = reinterpret_cast<int32_t*>(d_base + nc);
    MS_CUDA(c, cudaMemsetAsync(d_irr, 0, 8, st));
    MS_CUDA(c, cudaMemsetAsync(d_fault, 0xFF, 8, st));
    MS_CUDA(c, cudaMemsetAsync(d_first, 0, (size_t)nc * (3 * 8 + 4), st));

    // the text, zero padded
    MS_CUDA(c, c->vp_text.ensure((size_t)n + 64));
    uint8_t* t = c->vp_text.as<uint8_t>();
    for (int64_t off = 0; off < n; off += VCF_COPY_CHUNK)
        MS_CUDA(c, cudaMemcpyAsync(t + off, text + off, (size_t)std::min(VCF_COPY_CHUNK, n - off), cudaMemcpyHostToDevice, st));
    MS_CUDA(c, cudaMemsetAsync(t + n, 0, 64, st));

    // line starts
    const int64_t ng = ceil_div(n, 16);
    int64_t n_lines = 0;
    if (ng > 0) {
        // counted first: the array of line starts is sized by the count, not by the text
        auto in = [=] __device__(int64_t g) -> int64_t { return group_line_starts(t, n, g, nullptr, nullptr); };
        int64_t* ts = nullptr;
        int64_t nt = 0;
        MS_CUDA(c, scan_tile_sums<int64_t>(c, in, ng, (int64_t)0, SumOp(), c->scan_tmp, &ts, &nt));
        MS_CUDA(c, cudaMemcpyAsync(&n_lines, ts + nt, 8, cudaMemcpyDeviceToHost, st));
        MS_CUDA(c, cudaStreamSynchronize(st));
        MS_CUDA(c, c->vp_lines.ensure((size_t)(n_lines + 1) * 8));
        int64_t* lines = c->vp_lines.as<int64_t>();
        auto out = [=] __device__(int64_t g, int64_t ex, int64_t) { group_line_starts(t, n, g, lines + ex, d_irr); };
        k_scan_down<int64_t, SumOp, decltype(in), decltype(out)><<<(unsigned)nt, SCAN_THREADS, 0, st>>>(in, out, ng, (int64_t)0, SumOp(), ts);
        MS_LAUNCH_CHECK(c);
        const int64_t end = text[n - 1] == '\n' ? n : n + 1;       // line k ends at lines[k + 1] - 1
        MS_CUDA(c, cudaMemcpyAsync(lines + n_lines, &end, 8, cudaMemcpyHostToDevice, st));
    }

    // one record per line, then the records and their literals compacted in file order
    MS_CUDA(c, c->vp_lrec.ensure((size_t)(n_lines + 1) * sizeof(Rec)));
    MS_CUDA(c, c->vp_krec.ensure((size_t)(n_lines + 1) * sizeof(Rec)));
    MS_CUDA(c, c->vp_lit.ensure((size_t)n + 64));
    Rec* lrec = c->vp_lrec.as<Rec>();
    Rec* krec = c->vp_krec.as<Rec>();
    uint8_t* pool = c->vp_lit.as<uint8_t>();
    uint8_t* lmask = nullptr;    // ploidy > 0: masks per line, then per compacted record
    uint8_t* kmask = nullptr;
    if (ploidy > 0) {
        MS_CUDA(c, c->vp_lmask.ensure((size_t)n_lines + 16));
        MS_CUDA(c, c->vp_kmask.ensure((size_t)n_lines + 16));
        lmask = c->vp_lmask.as<uint8_t>();
        kmask = c->vp_kmask.as<uint8_t>();
    }
    I64x2 tot{0, 0};
    int h_irr = 0;
    if (n_lines > 0) {
        const int64_t* lines = c->vp_lines.as<int64_t>();
        k_vcf_parse_lines<<<(unsigned)ceil_div(n_lines, 256), 256, 0, st>>>(t, lines, n_lines, names, skip_unknown, lrec, d_irr);
        MS_LAUNCH_CHECK(c);
        if (lmask) {
            k_vcf_parse_gt<<<(unsigned)ceil_div(n_lines, 256), 256, 0, st>>>(t, lines, n_lines, lrec, ploidy, lmask, d_irr);
            MS_LAUNCH_CHECK(c);
        }
        auto in = [=] __device__(int64_t k) -> I64x2 {
            const Rec& r = lrec[k];
            return r.type == T_DEAD ? I64x2{0, 0} : I64x2{1, r.kind == K_LIT ? (int64_t)r.prod : 0};
        };
        auto out = [=] __device__(int64_t k, I64x2 ex, I64x2 v) {
            if (!v.a) return;
            Rec r = lrec[k];
            if (r.kind == K_LIT) {
                for (int64_t i = 0; i < v.b; ++i) pool[ex.b + i] = t[r.src + i];
                r.src = ex.b;
            }
            krec[ex.a] = r;
            if (lmask) kmask[ex.a] = lmask[k];
        };
        I64x2* d_tot = nullptr;
        MS_CUDA(c, device_scan<I64x2>(c, in, out, n_lines, I64x2{0, 0}, SumOp(), c->scan_tmp, &d_tot));
        MS_CUDA(c, cudaMemcpyAsync(&tot, d_tot, sizeof(I64x2), cudaMemcpyDeviceToHost, st));
    }
    MS_CUDA(c, cudaMemcpyAsync(&h_irr, d_irr, 4, cudaMemcpyDeviceToHost, st));
    MS_CUDA(c, cudaStreamSynchronize(st));
    if (h_irr) return MS_OK;
    const int64_t m = tot.a, lit_bytes = tot.b;

    // blocks in contig order
    if (m > 0) {
        const unsigned grid = (unsigned)ceil_div(m, 256);
        k_vcf_blocks<<<grid, 256, 0, st>>>(krec, m, d_first, d_last, d_nblk, d_irr);
        MS_LAUNCH_CHECK(c);
        std::vector<int64_t> bounds((size_t)nc * 2);
        MS_CUDA(c, cudaMemcpyAsync(&h_irr, d_irr, 4, cudaMemcpyDeviceToHost, st));
        MS_CUDA(c, cudaMemcpyAsync(bounds.data(), d_first, (size_t)nc * 16, cudaMemcpyDeviceToHost, st));
        MS_CUDA(c, cudaStreamSynchronize(st));
        if (h_irr) return MS_OK;
        std::vector<int64_t> base((size_t)nc);
        for (int64_t ci = 0, run = 0; ci < nc; ++ci) {       // blocks in contig order
            base[ci] = run - bounds[ci];
            run += bounds[nc + ci] - bounds[ci];
        }
        MS_CUDA(c, cudaMemcpyAsync(d_base, base.data(), (size_t)nc * 8, cudaMemcpyHostToDevice, st));
        k_vcf_place<<<grid, 256, 0, st>>>(krec, m, d_base, lrec);
        MS_LAUNCH_CHECK(c);
        if (lmask) {
            k_vcf_place_mask<<<grid, 256, 0, st>>>(krec, kmask, m, d_base, lmask);
            MS_LAUNCH_CHECK(c);
        }
        k_vcf_faults<<<grid, 256, 0, st>>>(lrec, m, nc, lit_bytes, c->total_bases + 64 + c->foreign_cap, d_fault);
        MS_LAUNCH_CHECK(c);
        // (a K_RAW source in a peer window, which ms_load_records accepts, cannot come from a VCF line: its sources
        // lie inside its own contig)
        unsigned long long h_fault = 0;
        MS_CUDA(c, cudaMemcpyAsync(&h_fault, d_fault, 8, cudaMemcpyDeviceToHost, st));
        MS_CUDA(c, cudaStreamSynchronize(st));
        if (h_fault != ~0ull) return record_fault(c, (int)(h_fault & 7), (int64_t)(h_fault >> 3));
    }
    std::swap(c->recs, c->vp_lrec);
    std::swap(c->lit, c->vp_lit);
    records_loaded(c, m, lit_bytes);
    if (ploidy > 0) {
        std::swap(c->gt_mask, c->vp_lmask);
        c->gt_ploidy = ploidy;
    }
    *regular = 1;
    *n_recs = m;
    return MS_OK;
}

}  // namespace ms
