// api.cu -- the C ABI of include/elprep_b200.h: context lifecycle, batch ingest, phase entry points, fetch.
#include <algorithm>
#include <map>
#include <thread>
#include "../../include/elprep_b200.h"
#include "ctx.h"

int run_apply_kernel(elp_ctx* c, bool with_lut);
#ifdef RS_TIMING
void rs_dump_timing();
#endif

namespace {

thread_local std::string g_create_error;

inline unsigned nblk(uint64_t n, int t) { return (unsigned)((n + t - 1) / t); }

__global__ void __launch_bounds__(256) rebase_kernel(uint64_t n, const uint64_t* __restrict__ rel, uint64_t base, uint64_t* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rel[i] + base;
}
__global__ void __launch_bounds__(256) lens_kernel(uint64_t n, const int32_t* __restrict__ lseq, uint32_t* __restrict__ qlen, uint32_t* __restrict__ slen) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const uint32_t l = (uint32_t)lseq[i]; qlen[i] = l; slen[i] = (l + 1) >> 1; }
}
__global__ void __launch_bounds__(256) add_base_kernel(uint64_t n, uint64_t* __restrict__ v, uint64_t base) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] += base;
}
__global__ void __launch_bounds__(256) widen_kernel(uint64_t n, const uint32_t* __restrict__ in, uint64_t* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}
__global__ void __launch_bounds__(256) rel_off_kernel(uint64_t n, const uint64_t* __restrict__ off, uint64_t first, uint64_t* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) out[i] = off[first + i] - off[first];
}

// which QUAL values occur (bit q of a 128-bit map): the BQSR count kernel classifies QUAL bytes through an 8-entry table and is only
// selected when that table separates every value that is present.  Runs at ingest over the bytes just appended.
__global__ void __launch_bounds__(256) qual_presence_kernel(const uint8_t* __restrict__ q, uint64_t n, uint32_t* __restrict__ present) {
    unsigned long long lo = 0, hi = 0;
    uint32_t other = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t head = (16 - (reinterpret_cast<uintptr_t>(q) & 15)) & 15;             // bytes before the first aligned 16-byte chunk
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    auto one = [&](uint32_t v) { lo |= 1ull << v; hi |= 1ull << (v - 64u); other |= v & 0x80u; };   // shifts >= 64 give 0
    if (t < head && t < n) one(q[t]);
    const uint64_t n16 = n > head ? (n - head) >> 4 : 0;
    const uint4* q4 = reinterpret_cast<const uint4*>(q + head);
    for (uint64_t i = t; i < n16; i += stride) {
        const uint4 v = ld_stream_u4(q4 + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; k++) { one(w[k] & 255u); one((w[k] >> 8) & 255u); one((w[k] >> 16) & 255u); one(w[k] >> 24); }
    }
    const uint64_t tail0 = head + (n16 << 4);
    if (tail0 + t < n && t < 16) one(q[tail0 + t]);
    for (int o = 16; o; o >>= 1) { lo |= __shfl_xor_sync(FULL_MASK, lo, o); hi |= __shfl_xor_sync(FULL_MASK, hi, o); other |= __shfl_xor_sync(FULL_MASK, other, o); }
    if ((threadIdx.x & 31) == 0) {
        if ((uint32_t)lo) atomicOr(present, (uint32_t)lo);
        if ((uint32_t)(lo >> 32)) atomicOr(present + 1, (uint32_t)(lo >> 32));
        if ((uint32_t)hi) atomicOr(present + 2, (uint32_t)hi);
        if ((uint32_t)(hi >> 32) || other) atomicOr(present + 3, (uint32_t)(hi >> 32) | (other ? 0x80000000u : 0u));   // bit 127: some byte >= 128
    }
}

template <class T> int grow(elp_ctx* c, DBuf<T>& b, size_t need, size_t keep) {
    cudaError_t e = b.reserve(need, c->stream, keep);
    if (e != cudaSuccess) return c->fail(e == cudaErrorMemoryAllocation ? E_NOMEM : E_CUDA, "device allocation of %zu bytes failed: %s", need * sizeof(T), cudaGetErrorString(e));
    return E_OK;
}
#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

}  // namespace

// Small host->device uploads INSIDE the phases (value ranges, look-up tables, ...) do not go through the copy engine: it serves its queue in
// order, so behind the multi-gigabyte upload of another context of a pipelined caller they would wait for all of it.  The bytes are staged in
// page-locked host memory that the GPU can address, and a kernel pulls them across.
__global__ void __launch_bounds__(256) pull_kernel(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, size_t n) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (i + 16 <= n) *reinterpret_cast<uint4*>(dst + i) = *reinterpret_cast<const uint4*>(src + i);
    else for (size_t k = i; k < n; k++) dst[k] = src[k];
}
int upload_small(elp_ctx* c, void* dst, const void* src, size_t bytes) {
    constexpr size_t CAP = 8u << 20;
    if (!bytes) return E_OK;
    if (bytes > CAP || (reinterpret_cast<uintptr_t>(dst) & 15)) { CUDA_TRY(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream)); return E_OK; }
    if (!c->h_stage) CUDA_TRY(c, cudaHostAlloc(&c->h_stage, CAP, cudaHostAllocPortable | cudaHostAllocMapped));
    if (c->stage_off + bytes > CAP) { CUDA_TRY(c, cudaStreamSynchronize(c->stream)); c->stage_off = 0; }
    uint8_t* st = reinterpret_cast<uint8_t*>(c->h_stage) + c->stage_off;
    memcpy(st, src, bytes);
    void* dev_src = st;
    CUDA_TRY(c, cudaHostGetDevicePointer(&dev_src, st, 0));
    c->launches++;
    pull_kernel<<<(unsigned)((bytes + 16 * 256 - 1) / (16 * 256)), 256, 0, c->stream>>>(reinterpret_cast<uint8_t*>(dst), reinterpret_cast<const uint8_t*>(dev_src), bytes);
    LAUNCH_CHECK(c);
    c->stage_off += (bytes + 255) & ~(size_t)255;
    return E_OK;
}

int qual_presence_update(elp_ctx* c, uint64_t first_byte, uint64_t n_bytes) {
    if (!n_bytes) return E_OK;
    const unsigned grid = (unsigned)std::min<uint64_t>((n_bytes / 16 + 255) / 256 + 1, 148 * 16);
    c->launches++;
    qual_presence_kernel<<<grid, 256, 0, c->stream>>>(c->qual.p + first_byte, n_bytes, c->d_qpresent);
    LAUNCH_CHECK(c);
    return E_OK;
}

int upload_side_inputs(elp_ctx* c) {
    if (!c->side_dirty) return E_OK;
    const int nc = c->n_contigs;
    std::vector<const uint8_t*> hp(nc); std::vector<const int32_t*> sp(nc);
    for (int i = 0; i < nc; i++) { hp[i] = c->d_refhot_raw[i] ? c->d_refhot_raw[i] + REFHOT_PAD : nullptr; sp[i] = c->d_sites[i]; }
    if (nc) {
        CUDA_TRY(c, cudaMemcpyAsync(c->d_refhot_ptrs, hp.data(), nc * sizeof(void*), cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_ref_len, c->ref_len.data(), nc * 8, cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_site_ptrs, sp.data(), nc * sizeof(void*), cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_n_sites, c->n_sites.data(), nc * 8, cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    c->side_dirty = false;
    return E_OK;
}

extern "C" {

const char* elp_last_error(const elp_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int elp_create(const elp_config* cfg, elp_ctx** out) {
    if (!cfg || !out) { g_create_error = "elp_create: null argument"; return ELP_EINVAL; }
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0 || cfg->device < 0 || cfg->device >= ndev) {
        g_create_error = std::string("elp_create: no usable CUDA device (") + (e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range") + "); this library has no CPU fallback";
        return ELP_ENODEVICE;
    }
    if ((e = cudaSetDevice(cfg->device)) != cudaSuccess) { g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e); return ELP_ENODEVICE; }
    elp_ctx* c = new elp_ctx();
    c->device = cfg->device;
    c->profile = cfg->profile != 0;
    auto bail = [&](int code) { g_create_error = c->err; elp_destroy(c); return code; };
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { c->err = "cudaStreamCreate failed"; return bail(ELP_ECUDA); }
    c->n_contigs = cfg->n_contigs;
    for (int i = 0; i < cfg->n_contigs; i++) { c->contig_len.push_back(cfg->contig_lengths[i]); c->contig_names.push_back(cfg->contig_names && cfg->contig_names[i] ? cfg->contig_names[i] : ""); }
    // library ids: equal LB strings share an id (lbTable, mark-duplicates.go:413-423); covariates: PU if present else ID (bqsr.go:35-51)
    c->n_rg = cfg->n_read_groups;
    std::map<std::string, int> libs, covs;
    for (int i = 0; i < c->n_rg; i++) {
        if (!cfg->rg_id || !cfg->rg_id[i]) { c->err = "Missing mandatory ID entry in an @RG line in a SAM file header."; return bail(ELP_EINVAL); }
        c->rg_ids.push_back(cfg->rg_id[i]);
        const char* lb = cfg->rg_lb ? cfg->rg_lb[i] : nullptr;
        if (lb) { auto it = libs.find(lb); if (it == libs.end()) { it = libs.emplace(lb, (int)libs.size()).first; c->lib_names.push_back(lb); } c->rg_lib.push_back(it->second); } else c->rg_lib.push_back(-1);
        const char* pu = cfg->rg_pu ? cfg->rg_pu[i] : nullptr;
        std::string name = pu ? pu : cfg->rg_id[i];
        auto it = covs.find(name);
        if (it == covs.end()) { it = covs.emplace(name, (int)c->cov_names.size()).first; c->cov_names.push_back(name); }
        c->rg_cov.push_back(it->second);
    }
    c->n_lib = (int)libs.size();
    c->max_cycle = cfg->max_cycle > 0 ? cfg->max_cycle : 500;
    c->quantize_levels = cfg->quantize_levels;
    if (cfg->sqq && cfg->n_sqq > 0) c->sqq.assign(cfg->sqq, cfg->sqq + cfg->n_sqq);
    if (cfg->tablename_prefix) c->prefix = cfg->tablename_prefix;
    c->optical_pixel_distance = cfg->optical_pixel_distance > 0 ? cfg->optical_pixel_distance : 100;
    c->geom.n_cov = (int)c->cov_names.size(); c->geom.max_cycle = c->max_cycle;
    const int nc = std::max(1, c->n_contigs), nr = std::max(1, c->n_rg);
    bool ok = cudaMalloc(&c->d_rg_lib, nr * 4) == cudaSuccess && cudaMalloc(&c->d_rg_cov, nr * 4) == cudaSuccess && cudaMalloc(&c->d_contig_len, nc * 4) == cudaSuccess &&
              cudaMalloc(&c->d_ranges, sizeof(DeviceRanges)) == cudaSuccess && cudaMalloc(&c->d_err, 4) == cudaSuccess &&
              cudaMalloc(&c->d_refhot_ptrs, nc * sizeof(void*)) == cudaSuccess &&
              cudaMalloc(&c->d_bq_small, 512 * 4) == cudaSuccess && cudaMalloc(&c->d_qpresent, 16) == cudaSuccess && cudaMalloc(&c->d_ref_len, nc * 8) == cudaSuccess &&
              cudaMalloc(&c->d_site_ptrs, nc * sizeof(void*)) == cudaSuccess && cudaMalloc(&c->d_n_sites, nc * 8) == cudaSuccess &&
              cudaMalloc(&c->d_tables, std::max<size_t>(16, c->geom.cells() * 2 * sizeof(int64_t))) == cudaSuccess;
    if (!ok) { c->err = "device allocation failed in elp_create"; return bail(ELP_ENOMEM); }
    if (c->n_rg) { cudaMemcpy(c->d_rg_lib, c->rg_lib.data(), c->n_rg * 4, cudaMemcpyHostToDevice); cudaMemcpy(c->d_rg_cov, c->rg_cov.data(), c->n_rg * 4, cudaMemcpyHostToDevice); }
    if (c->n_contigs) cudaMemcpy(c->d_contig_len, c->contig_len.data(), c->n_contigs * 4, cudaMemcpyHostToDevice);
    cudaMemset(c->d_err, 0, 4);
    cudaMemset(c->d_qpresent, 0, 16);
    c->n_qual = c->n_seq = ARENA_FRONT_PAD;
    cudaMemset(c->d_tables, 0, std::max<size_t>(16, c->geom.cells() * 2 * sizeof(int64_t)));
    c->d_refhot_raw.assign(c->n_contigs, nullptr); c->ref_len.assign(c->n_contigs, 0);
    c->d_sites.assign(c->n_contigs, nullptr); c->n_sites.assign(c->n_contigs, 0);
    if ((e = cudaGetLastError()) != cudaSuccess) { c->err = std::string("elp_create: ") + cudaGetErrorString(e); return bail(ELP_ECUDA); }
    *out = c;
    return ELP_OK;
}

void elp_destroy(elp_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (auto p : c->d_refhot_raw) if (p) cudaFree(p);
    for (auto p : c->d_sites) if (p) cudaFree(p);
    for (auto p : c->d_regions) if (p) cudaFree(p);
    if (c->d_region_ptrs) cudaFree((void*)c->d_region_ptrs);
    if (c->d_n_regions) cudaFree(c->d_n_regions);
    void* singles[] = {c->d_rg_lib, c->d_rg_cov, c->d_contig_len, c->d_ranges, c->d_err, (void*)c->d_refhot_ptrs, c->d_bq_small, c->d_qpresent, c->d_ref_len, (void*)c->d_site_ptrs, c->d_n_sites, c->d_tables,
                       c->d_lut, c->d_clut, c->d_rowtab, c->d_cov_exists, c->d_opt_ctr, c->d_opt_hist, c->d_opt_ovf, c->d_opt_small, c->d_rg_names, c->d_rg_name_off, c->ws.ghist, c->ws.gofs, c->ws.counters, c->ws.status};
    for (void* p : singles) if (p) cudaFree(p);
    c->refid.release(); c->pos.release(); c->nref.release(); c->pnext.release(); c->tlen.release(); c->rg.release(); c->flag.release(); c->mapq.release(); c->optf.release(); c->s_optf.release();
    c->qname_off.release(); c->cigar_off.release(); c->qual_off.release(); c->seq_off.release(); c->qname.release(); c->seq.release(); c->qual.release(); c->cigar.release();
    c->bam_raw.release(); c->bam_off.release(); c->bam_all.release(); c->bam_all_off.release(); c->bam_start.release(); c->lseq_stage.release(); c->off_stage.release(); c->upos.release(); c->score.release(); c->qhash.release(); c->keys_a.release(); c->keys_b.release();
    c->bq_recs.release(); c->bq_segs.release(); c->vals_a.release(); c->vals_b.release(); c->mate.release(); c->pair_a.release(); c->pair_b.release(); c->scan_tmp.release(); c->scan_blk.release(); c->bytes_tmp.release();
    c->perm.release(); c->s_refid.release(); c->s_pos.release(); c->s_nref.release(); c->s_pnext.release(); c->s_tlen.release(); c->s_rg.release(); c->s_lseq.release();
    c->s_flag.release(); c->s_mapq.release(); c->s_qual_off.release(); c->s_seq_off.release(); c->s_cigar_off.release(); c->s_out_off.release(); c->s_ncigar.release(); c->qual_out.release();
    for (auto& pe : c->pending) { cudaEventDestroy(pe.a); cudaEventDestroy(pe.b); }
    for (auto e : c->event_pool) cudaEventDestroy(e);
    if (c->timer_a) { cudaEventDestroy(c->timer_a); cudaEventDestroy(c->timer_b); }
    elp_comm_destroy(c);
    if (c->d_owner) cudaFree(c->d_owner);
    c->sp_sendbuf.release(); c->sp_recvbuf.release(); c->sp_sent_idx.release();
    if (c->h_stage) cudaFreeHost(c->h_stage);
    if (c->copy_in) { cudaStreamDestroy(c->copy_in); cudaEventDestroy(c->ev_in); cudaEventDestroy(c->ev_staged); }
    if (c->copy_out) { cudaStreamDestroy(c->copy_out); cudaEventDestroy(c->ev_out); }
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int elp_reset(elp_ctx* c) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (c->copy_in) CUDA_TRY(c, cudaStreamSynchronize(c->copy_in));
    if (c->copy_out) CUDA_TRY(c, cudaStreamSynchronize(c->copy_out));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    c->n = c->n_qname = c->n_cigar = 0; c->n_qual = c->n_seq = ARENA_FRONT_PAD; c->n_bam = c->bam_reads = 0; c->n_filtered = 0; c->n_cleaned = 0;
    CUDA_TRY(c, cudaMemsetAsync(c->d_qpresent, 0, 16, c->stream));
    c->adapted = c->sorted = c->qual_out_valid = c->gathered = c->finalized = c->opt_valid = false;
    c->launches = 0;
    CUDA_TRY(c, cudaMemsetAsync(c->d_err, 0, 4, c->stream));
    return ELP_OK;
}

int elp_reserve(elp_ctx* c, uint64_t n_reads, uint64_t n_bases, uint64_t n_cigar_ops, uint64_t n_qname_bytes) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    std::lock_guard<std::mutex> lk(c->append_mu);
    const size_t n = n_reads + 1;
    TRY(grow(c, c->refid, n, c->n)); TRY(grow(c, c->pos, n, c->n)); TRY(grow(c, c->nref, n, c->n)); TRY(grow(c, c->pnext, n, c->n)); TRY(grow(c, c->tlen, n, c->n));
    TRY(grow(c, c->rg, n, c->n)); TRY(grow(c, c->flag, n + 1, c->n)); TRY(grow(c, c->mapq, n, c->n)); TRY(grow(c, c->optf, n, c->n));
    TRY(grow(c, c->qname_off, n + 1, c->n + 1)); TRY(grow(c, c->cigar_off, n + 1, c->n + 1)); TRY(grow(c, c->qual_off, n + 1, c->n + 1)); TRY(grow(c, c->seq_off, n + 1, c->n + 1));
    TRY(grow(c, c->qname, n_qname_bytes + 64, c->n_qname)); TRY(grow(c, c->cigar, n_cigar_ops + 16, c->n_cigar));
    TRY(grow(c, c->qual, n_bases + 64 + ARENA_FRONT_PAD, c->n_qual)); TRY(grow(c, c->seq, n_bases / 2 + n_reads + 64 + ARENA_FRONT_PAD, c->n_seq));
    return ELP_OK;
}

int elp_set_reference(elp_ctx* c, int32_t contig, const uint8_t* bases, uint64_t n) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (contig < 0 || contig >= c->n_contigs) return c->fail(E_INVAL, "elp_set_reference: contig %d out of range", contig);
    return pack_reference(c, contig, bases, n);
}

int elp_set_known_sites(elp_ctx* c, int32_t contig, const int32_t* se, uint64_t n_intervals, int already_flat) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (contig < 0 || contig >= c->n_contigs) return c->fail(E_INVAL, "elp_set_known_sites: contig %d out of range", contig);
    std::vector<int32_t> v(se, se + 2 * n_intervals);
    uint64_t n = n_intervals;
    if (!already_flat && n > 1) {
        // stable sort by start (intervals.ParallelSortByStart) then Flatten (intervals/intervals.go:88-117): merge while next.Start <= cur.End
        std::vector<std::pair<int32_t, int32_t>> iv(n);
        for (uint64_t i = 0; i < n; i++) iv[i] = {v[2 * i], v[2 * i + 1]};
        std::stable_sort(iv.begin(), iv.end(), [](const std::pair<int32_t, int32_t>& a, const std::pair<int32_t, int32_t>& b) { return a.first < b.first; });
        uint64_t m = 0;
        for (uint64_t i = 0; i < n; i++) {
            if (m > 0 && iv[i].first <= iv[m - 1].second) { if (iv[i].second > iv[m - 1].second) iv[m - 1].second = iv[i].second; }
            else iv[m++] = iv[i];
        }
        n = m;
        for (uint64_t i = 0; i < n; i++) { v[2 * i] = iv[i].first; v[2 * i + 1] = iv[i].second; }
    }
    if (c->d_sites[contig]) { cudaFree(c->d_sites[contig]); c->d_sites[contig] = nullptr; }
    if (n) {
        CUDA_TRY(c, cudaMalloc(&c->d_sites[contig], n * 8));
        CUDA_TRY(c, cudaMemcpy(c->d_sites[contig], v.data(), n * 8, cudaMemcpyHostToDevice));
    }
    c->n_sites[contig] = n; c->side_dirty = true;
    return ELP_OK;
}

uint64_t elp_n_reads(const elp_ctx* c) { return c ? c->n : 0; }

// elp_append_batch and its asynchronous form.  All host->device copies go to the context's ingest stream (`copy_in`), the small kernels
// that turn batch-relative offsets into arena offsets follow on the compute stream behind an event, so a pipelined caller can overlap
// the upload of one context with the kernels and the download of another (bench.py's e2e loop does exactly that with two contexts).
static uint64_t sum_lengths(const int32_t* l, uint64_t n, uint64_t* seq_bytes) {
    const unsigned nt = n > (1u << 20) ? std::min(8u, std::max(1u, std::thread::hardware_concurrency())) : 1u;
    std::vector<uint64_t> a(nt, 0), b(nt, 0);
    auto work = [&](unsigned t) { uint64_t x = 0, y = 0; for (uint64_t i = n * t / nt, e = n * (t + 1) / nt; i < e; i++) { const uint64_t v = (uint64_t)(uint32_t)l[i]; x += v; y += (v + 1) >> 1; } a[t] = x; b[t] = y; };
    if (nt == 1) work(0); else { std::vector<std::thread> th; for (unsigned t = 0; t < nt; t++) th.emplace_back(work, t); for (auto& x : th) x.join(); }
    uint64_t x = 0, y = 0; for (unsigned t = 0; t < nt; t++) { x += a[t]; y += b[t]; }
    *seq_bytes = y; return x;
}

// Large host<->device copies go out whole by default.  (A copy engine serves its queue in order, so cutting a copy into pieces that are all
// enqueued at once does not let another context's small copies overtake it -- measured with tools/e2e_probe.py: 32 MB pieces cost 5 % of the
// duplex upload rate and the small copies waited just the same.  The phases therefore avoid the copy engines for their small uploads
// (upload_small), and a pipelined caller orders its downloads so that none is in flight while another context's phases read back.)
// ELPREP_B200_COPY_CHUNK_MB > 0 restores the pieces for experiments.
static cudaError_t copy_chunked(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s) {
    static const size_t CH = [] { const char* e = getenv("ELPREP_B200_COPY_CHUNK_MB"); const long v = e ? atol(e) : 0; return v <= 0 ? ~(size_t)0 : (size_t)v << 20; }();
    for (size_t o = 0; o < bytes; o += CH) {
        cudaError_t e = cudaMemcpyAsync((char*)dst + o, (const char*)src + o, std::min(CH, bytes - o), kind, s);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

static int append_impl(elp_ctx* c, const elp_batch* b, bool wait) {
    cudaSetDevice(c->device);
    std::lock_guard<std::mutex> lk(c->append_mu);
    const uint64_t bn = b->n;
    if (bn == 0) return ELP_OK;
    if (c->sorted) return c->fail(E_STATE, "elp_append_batch after elp_sort_markdup (call elp_reset first)");
    const uint64_t n0 = c->n, n1 = n0 + bn;
    if (n1 >= (1ull << 32)) return c->fail(E_LIMIT, "more than 2^32-1 reads in one context");
    const uint64_t bq = b->qname_off[bn] - b->qname_off[0], bc = b->cigar_off[bn] - b->cigar_off[0];
    uint64_t bseq = 0;
    const uint64_t bbases = sum_lengths(b->l_seq, bn, &bseq);
    // growing a buffer moves it: uploads of an earlier asynchronous append that are still in flight must land first
    if (c->copy_in && (n1 + 2 > c->flag.cap || n1 + 2 > c->qname_off.cap || c->n_qname + bq + 64 > c->qname.cap || c->n_cigar + bc + 16 > c->cigar.cap ||
                       c->n_qual + bbases + 64 > c->qual.cap || c->n_seq + bseq + 64 > c->seq.cap)) CUDA_TRY(c, cudaStreamSynchronize(c->copy_in));
    TRY(grow(c, c->refid, n1 + 1, n0)); TRY(grow(c, c->pos, n1 + 1, n0)); TRY(grow(c, c->nref, n1 + 1, n0)); TRY(grow(c, c->pnext, n1 + 1, n0)); TRY(grow(c, c->tlen, n1 + 1, n0));
    TRY(grow(c, c->rg, n1 + 1, n0)); TRY(grow(c, c->flag, n1 + 2, n0)); TRY(grow(c, c->mapq, n1 + 1, n0)); TRY(grow(c, c->optf, n1 + 1, n0));
    TRY(grow(c, c->qname_off, n1 + 2, n0 + 1)); TRY(grow(c, c->cigar_off, n1 + 2, n0 + 1)); TRY(grow(c, c->qual_off, n1 + 2, n0 + 1)); TRY(grow(c, c->seq_off, n1 + 2, n0 + 1));
    TRY(grow(c, c->qname, c->n_qname + bq + 64, c->n_qname)); TRY(grow(c, c->cigar, c->n_cigar + bc + 16, c->n_cigar));
    TRY(grow(c, c->qual, c->n_qual + bbases + 64, c->n_qual)); TRY(grow(c, c->seq, c->n_seq + bseq + 64, c->n_seq));
    if (!c->copy_in) { CUDA_TRY(c, cudaStreamCreateWithFlags(&c->copy_in, cudaStreamNonBlocking)); CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming)); CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_staged, cudaEventDisableTiming)); }
    cudaStream_t s = c->stream, ci = c->copy_in;
    // the staging buffers of the previous append must have been consumed by its kernels; growth (above) may also have used the compute stream
    CUDA_TRY(c, cudaEventRecord(c->ev_staged, s)); CUDA_TRY(c, cudaStreamWaitEvent(ci, c->ev_staged, 0));
    TRY(grow(c, c->off_stage, 2 * (bn + 2), 0)); TRY(grow(c, c->lseq_stage, bn + 2, 0)); TRY(grow(c, c->scan_tmp, 2 * bn + 8, 0));
    const cudaMemcpyKind H2D = cudaMemcpyHostToDevice;
    CUDA_TRY(c, copy_chunked(c->refid.p + n0, b->refid, bn * 4, H2D, ci)); CUDA_TRY(c, copy_chunked(c->pos.p + n0, b->pos, bn * 4, H2D, ci));
    CUDA_TRY(c, copy_chunked(c->nref.p + n0, b->nref, bn * 4, H2D, ci)); CUDA_TRY(c, copy_chunked(c->pnext.p + n0, b->pnext, bn * 4, H2D, ci));
    CUDA_TRY(c, copy_chunked(c->tlen.p + n0, b->tlen, bn * 4, H2D, ci)); CUDA_TRY(c, copy_chunked(c->rg.p + n0, b->rg, bn * 4, H2D, ci));
    CUDA_TRY(c, copy_chunked(c->flag.p + n0, b->flag, bn * 2, H2D, ci)); CUDA_TRY(c, copy_chunked(c->mapq.p + n0, b->mapq, bn, H2D, ci));
    if (b->opt_flags) CUDA_TRY(c, copy_chunked(c->optf.p + n0, b->opt_flags, bn, H2D, ci)); else CUDA_TRY(c, cudaMemsetAsync(c->optf.p + n0, 0, bn, ci));
    uint64_t* st_q = c->off_stage.p; uint64_t* st_c = c->off_stage.p + (bn + 2);
    CUDA_TRY(c, copy_chunked(st_q, b->qname_off, (bn + 1) * 8, H2D, ci));
    CUDA_TRY(c, copy_chunked(st_c, b->cigar_off, (bn + 1) * 8, H2D, ci));
    CUDA_TRY(c, copy_chunked(c->lseq_stage.p, b->l_seq, bn * 4, H2D, ci));
    if (bq) CUDA_TRY(c, copy_chunked(c->qname.p + c->n_qname, b->qname + b->qname_off[0], bq, H2D, ci));
    if (bc) CUDA_TRY(c, copy_chunked(c->cigar.p + c->n_cigar, b->cigar + b->cigar_off[0], bc * 4, H2D, ci));
    if (bseq) CUDA_TRY(c, copy_chunked(c->seq.p + c->n_seq, b->seq, bseq, H2D, ci));
    if (bbases) CUDA_TRY(c, copy_chunked(c->qual.p + c->n_qual, b->qual, bbases, H2D, ci));
    CUDA_TRY(c, cudaEventRecord(c->ev_in, ci));
    CUDA_TRY(c, cudaStreamWaitEvent(s, c->ev_in, 0));
    // offsets: batch-relative -> arena-global
    rebase_kernel<<<nblk(bn + 1, 256), 256, 0, s>>>(bn + 1, st_q, c->n_qname - b->qname_off[0], c->qname_off.p + n0); c->launches++;
    rebase_kernel<<<nblk(bn + 1, 256), 256, 0, s>>>(bn + 1, st_c, c->n_cigar - b->cigar_off[0], c->cigar_off.p + n0); c->launches++;
    uint32_t* qlen = c->scan_tmp.p; uint32_t* slen = c->scan_tmp.p + bn + 4;
    lens_kernel<<<nblk(bn, 256), 256, 0, s>>>(bn, c->lseq_stage.p, qlen, slen); c->launches++;
    LAUNCH_CHECK(c);
    TRY(exclusive_scan_u32_to_u64(c, qlen, c->qual_off.p + n0, bn));
    add_base_kernel<<<nblk(bn + 1, 256), 256, 0, s>>>(bn + 1, c->qual_off.p + n0, c->n_qual); c->launches++;
    TRY(exclusive_scan_u32_to_u64(c, slen, c->seq_off.p + n0, bn));
    add_base_kernel<<<nblk(bn + 1, 256), 256, 0, s>>>(bn + 1, c->seq_off.p + n0, c->n_seq); c->launches++;
    LAUNCH_CHECK(c);
    TRY(qual_presence_update(c, c->n_qual, bbases));
    c->n = n1; c->n_qname += bq; c->n_cigar += bc; c->n_qual += bbases; c->n_seq += bseq;
    c->adapted = false;
    if (wait) { CUDA_TRY(c, cudaStreamSynchronize(ci)); CUDA_TRY(c, cudaStreamSynchronize(s)); }   // the caller's buffers may be released after return (cgo pointer rules)
    return ELP_OK;
}

int elp_append_batch(elp_ctx* c, const elp_batch* b) { if (!c || !b) return ELP_EINVAL; return append_impl(c, b, true); }
int elp_append_batch_async(elp_ctx* c, const elp_batch* b) { if (!c || !b) return ELP_EINVAL; return append_impl(c, b, false); }
int elp_append_wait(elp_ctx* c) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (c->copy_in) CUDA_TRY(c, cudaStreamSynchronize(c->copy_in));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ELP_OK;
}

int elp_sort_markdup(elp_ctx* c, int sorting_order, int mark_duplicates) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (c->sorted) return c->fail(E_STATE, "elp_sort_markdup called twice (call elp_reset first)");
    if (mark_duplicates != 0 && mark_duplicates != ELP_MARKDUP && mark_duplicates != ELP_MARKDUP_OPTICAL) return c->fail(E_INVAL, "elp_sort_markdup: mark_duplicates must be 0, ELP_MARKDUP or ELP_MARKDUP_OPTICAL");
    if (mark_duplicates) TRY(phase_markdup(c, mark_duplicates == ELP_MARKDUP_OPTICAL));
    TRY(phase_coordinate_sort(c, sorting_order == ELP_SO_COORDINATE ? 1 : (sorting_order == ELP_SO_QUERYNAME ? 2 : 0)));
    return ELP_OK;
}

int elp_bqsr_gather(elp_ctx* c) { if (!c) return ELP_EINVAL; cudaSetDevice(c->device); return phase_bqsr_gather(c); }
int elp_bqsr_finalize(elp_ctx* c, const char* report_path) { if (!c) return ELP_EINVAL; cudaSetDevice(c->device); return phase_bqsr_finalize(c, report_path); }
int elp_bqsr_apply(elp_ctx* c) { if (!c) return ELP_EINVAL; cudaSetDevice(c->device); return phase_bqsr_apply(c); }

uint64_t elp_bqsr_tables_len(const elp_ctx* c) { return c ? (uint64_t)c->geom.cells() * 2 : 0; }
int32_t elp_bqsr_n_cov(const elp_ctx* c) { return c ? c->geom.n_cov : 0; }
const char* elp_bqsr_cov_name(const elp_ctx* c, int32_t cov) { return (c && cov >= 0 && cov < (int)c->cov_names.size()) ? c->cov_names[cov].c_str() : nullptr; }
int elp_bqsr_tables_get(elp_ctx* c, int64_t* dense, uint64_t n) {
    if (!c || !dense) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (n != elp_bqsr_tables_len(c)) return c->fail(E_INVAL, "elp_bqsr_tables_get: expected %llu values", (unsigned long long)elp_bqsr_tables_len(c));
    CUDA_TRY(c, cudaMemcpyAsync(dense, c->d_tables, n * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ELP_OK;
}
int elp_bqsr_tables_put(elp_ctx* c, const int64_t* dense, uint64_t n) {
    if (!c || !dense) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (n != elp_bqsr_tables_len(c)) return c->fail(E_INVAL, "elp_bqsr_tables_put: expected %llu values", (unsigned long long)elp_bqsr_tables_len(c));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_tables, dense, n * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    c->gathered = true; c->finalized = false;
    return ELP_OK;
}
int elp_bqsr_tables_device(elp_ctx* c, void** p, uint64_t* n) {
    if (!c || !p || !n) return ELP_EINVAL;
    cudaSetDevice(c->device);
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    *p = c->d_tables; *n = elp_bqsr_tables_len(c);
    c->finalized = false;
    return ELP_OK;
}
int elp_bqsr_empirical_get(elp_ctx* c, uint8_t* emp, uint64_t n) {
    if (!c || !emp) return ELP_EINVAL;
    if (!c->finalized) return c->fail(E_STATE, "elp_bqsr_empirical_get before elp_bqsr_finalize");
    if (n != c->geom.cells()) return c->fail(E_INVAL, "elp_bqsr_empirical_get: expected %zu values", c->geom.cells());
    std::copy(c->h_emp.begin(), c->h_emp.end(), emp);
    return ELP_OK;
}

uint64_t elp_fetch_qual_bytes(elp_ctx* c, uint64_t first, uint64_t n) {
    if (!c || !c->sorted || first + n > c->n) return 0;
    cudaSetDevice(c->device);
    uint64_t v[2] = {0, 0};
    cudaMemcpyAsync(&v[0], c->s_out_off.p + first, 8, cudaMemcpyDeviceToHost, c->stream);
    cudaMemcpyAsync(&v[1], c->s_out_off.p + first + n, 8, cudaMemcpyDeviceToHost, c->stream);
    cudaStreamSynchronize(c->stream);
    return v[1] - v[0];
}

static int fetch_impl(elp_ctx* c, uint64_t first, uint64_t n, uint64_t* record_index, uint32_t* record_index32, uint16_t* flag, uint64_t* qual_off, uint8_t* qual, uint64_t qual_capacity, bool wait) {
    cudaSetDevice(c->device);
    if (!c->sorted) return c->fail(E_STATE, "elp_fetch before elp_sort_markdup");
    if (first + n > c->n) return c->fail(E_INVAL, "elp_fetch: range [%llu,%llu) exceeds %llu reads", (unsigned long long)first, (unsigned long long)(first + n), (unsigned long long)c->n);
    if (n == 0) { if (qual_off) qual_off[0] = 0; return ELP_OK; }
    cudaStream_t s = c->stream;
    if (!c->copy_out) { CUDA_TRY(c, cudaStreamCreateWithFlags(&c->copy_out, cudaStreamNonBlocking)); CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming)); }
    cudaStream_t co = c->copy_out;
    uint64_t v[2] = {0, 0};
    if (qual) {
        if (!c->qual_out_valid) TRY(run_apply_kernel(c, false));   // no BQSR: just the QUAL bytes in output order
        if (first == 0 && n == c->n) { v[0] = 0; v[1] = c->qual_out_total; }
        else {
            CUDA_TRY(c, cudaMemcpyAsync(&v[0], c->s_out_off.p + first, 8, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(c, cudaMemcpyAsync(&v[1], c->s_out_off.p + first + n, 8, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(c, cudaStreamSynchronize(s));
        }
        if (v[1] - v[0] > qual_capacity) return c->fail(E_INVAL, "elp_fetch: qual buffer too small (%llu > %llu)", (unsigned long long)(v[1] - v[0]), (unsigned long long)qual_capacity);
    }
    if (record_index || qual_off) TRY(grow(c, c->off_stage, 2 * (n + 2), 0));
    if (record_index) { widen_kernel<<<nblk(n, 256), 256, 0, s>>>(n, c->perm.p + first, c->off_stage.p); c->launches++; }
    if (qual_off) { rel_off_kernel<<<nblk(n + 1, 256), 256, 0, s>>>(n, c->s_out_off.p, first, c->off_stage.p + (n + 2)); c->launches++; }
    LAUNCH_CHECK(c);
    // everything the compute stream produced so far (apply, the two small kernels above) -> the download stream
    CUDA_TRY(c, cudaEventRecord(c->ev_out, s)); CUDA_TRY(c, cudaStreamWaitEvent(co, c->ev_out, 0));
    if (qual) CUDA_TRY(c, copy_chunked(qual, c->qual_out.p + v[0], v[1] - v[0], cudaMemcpyDeviceToHost, co));
    if (record_index) CUDA_TRY(c, copy_chunked(record_index, c->off_stage.p, n * 8, cudaMemcpyDeviceToHost, co));
    if (record_index32) CUDA_TRY(c, copy_chunked(record_index32, c->perm.p + first, n * 4, cudaMemcpyDeviceToHost, co));
    if (flag) CUDA_TRY(c, copy_chunked(flag, c->s_flag.p + first, n * 2, cudaMemcpyDeviceToHost, co));
    if (qual_off) CUDA_TRY(c, copy_chunked(qual_off, c->off_stage.p + (n + 2), (n + 1) * 8, cudaMemcpyDeviceToHost, co));
    if (wait) CUDA_TRY(c, cudaStreamSynchronize(co));
    return ELP_OK;
}
int elp_fetch(elp_ctx* c, uint64_t first, uint64_t n, uint64_t* record_index, uint16_t* flag, uint64_t* qual_off, uint8_t* qual, uint64_t qual_capacity) {
    if (!c) return ELP_EINVAL;
    return fetch_impl(c, first, n, record_index, nullptr, flag, qual_off, qual, qual_capacity, true);
}
int elp_fetch_async(elp_ctx* c, uint64_t first, uint64_t n, uint32_t* record_index32, uint16_t* flag, uint64_t* qual_off, uint8_t* qual, uint64_t qual_capacity) {
    if (!c) return ELP_EINVAL;
    return fetch_impl(c, first, n, nullptr, record_index32, flag, qual_off, qual, qual_capacity, false);
}
int elp_fetch_wait(elp_ctx* c) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (c->copy_out) CUDA_TRY(c, cudaStreamSynchronize(c->copy_out));
    return ELP_OK;
}

int elp_fetch_opt_flags(elp_ctx* c, uint64_t first, uint64_t n, uint8_t* opt_flags) {
    if (!c || (!opt_flags && n)) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (!c->sorted) return c->fail(E_STATE, "elp_fetch_opt_flags before elp_sort_markdup");
    if (first + n > c->n) return c->fail(E_INVAL, "elp_fetch_opt_flags: range exceeds %llu reads", (unsigned long long)c->n);
    if (n) { CUDA_TRY(c, cudaMemcpyAsync(opt_flags, c->s_optf.p + first, n, cudaMemcpyDeviceToHost, c->stream)); CUDA_TRY(c, cudaStreamSynchronize(c->stream)); }
    return ELP_OK;
}

int elp_debug_adapt(elp_ctx* c, int32_t* upos, int32_t* score) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    TRY(phase_adapt(c));
    if (upos) CUDA_TRY(c, cudaMemcpyAsync(upos, c->upos.p, c->n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (score) CUDA_TRY(c, cudaMemcpyAsync(score, c->score.p, c->n * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ELP_OK;
}

uint64_t elp_launch_count(const elp_ctx* c) { return c ? c->launches : 0; }
int elp_synchronize(elp_ctx* c) { if (!c) return ELP_EINVAL; cudaSetDevice(c->device); CUDA_TRY(c, cudaStreamSynchronize(c->stream)); return ELP_OK; }
int elp_reset_stats(elp_ctx* c) { if (!c) return ELP_EINVAL; cudaSetDevice(c->device); c->resolve_events(); c->stats.clear(); c->launches = 0; return ELP_OK; }
int elp_timer_start(elp_ctx* c) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    if (!c->timer_a) { CUDA_TRY(c, cudaEventCreate(&c->timer_a)); CUDA_TRY(c, cudaEventCreate(&c->timer_b)); }
    CUDA_TRY(c, cudaEventRecord(c->timer_a, c->stream));
    return ELP_OK;
}
int elp_timer_stop(elp_ctx* c, double* ms) {
    if (!c || !ms || !c->timer_a) return ELP_EINVAL;
    cudaSetDevice(c->device);
    CUDA_TRY(c, cudaEventRecord(c->timer_b, c->stream));
    CUDA_TRY(c, cudaEventSynchronize(c->timer_b));
    float f = 0; CUDA_TRY(c, cudaEventElapsedTime(&f, c->timer_a, c->timer_b));
    *ms = f;
    return ELP_OK;
}
int elp_kernel_stats(elp_ctx* c, elp_kernel_stat* out, int cap) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    c->resolve_events();
    int k = 0;
    for (auto& kv : c->stats) {
        if (k >= cap) break;
        std::snprintf(out[k].name, sizeof out[k].name, "%s", kv.first.c_str());
        out[k].launches = kv.second.launches; out[k].ms = kv.second.ms; out[k].alg_bytes = kv.second.alg_bytes;
        k++;
    }
    return k;
}

int elp_debug_sort_u64(elp_ctx* c, uint64_t* keys, uint32_t* vals, uint64_t n, int key_bits) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    TRY(grow(c, c->keys_a, n + 4, 0)); TRY(grow(c, c->keys_b, n + 4, 0)); TRY(grow(c, c->vals_a, n + 4, 0)); TRY(grow(c, c->vals_b, n + 4, 0));
    CUDA_TRY(c, cudaMemcpyAsync(c->keys_a.p, keys, n * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(c->vals_a.p, vals, n * 4, cudaMemcpyHostToDevice, c->stream));
    bool in_b = false;
    TRY(radix_sort_u64(c, c->keys_a.p, c->keys_b.p, c->vals_a.p, c->vals_b.p, n, key_bits, &in_b, "u64"));
    CUDA_TRY(c, cudaMemcpyAsync(keys, in_b ? c->keys_b.p : c->keys_a.p, n * 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(vals, in_b ? c->vals_b.p : c->vals_a.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
#ifdef RS_TIMING
    rs_dump_timing();
#endif
    return ELP_OK;
}

int elp_debug_sort_u128(elp_ctx* c, uint64_t* keys_hi, uint64_t* keys_lo, uint32_t* vals, uint64_t n, int key_bits) {
    if (!c) return ELP_EINVAL;
    cudaSetDevice(c->device);
    TRY(grow(c, c->keys_a, 2 * n + 4, 0)); TRY(grow(c, c->keys_b, 2 * n + 4, 0)); TRY(grow(c, c->vals_a, n + 4, 0)); TRY(grow(c, c->vals_b, n + 4, 0));
    std::vector<uint64_t> inter(2 * n);
    for (uint64_t i = 0; i < n; i++) { inter[2 * i] = keys_lo[i]; inter[2 * i + 1] = keys_hi[i]; }
    CUDA_TRY(c, cudaMemcpyAsync(c->keys_a.p, inter.data(), n * 16, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(c->vals_a.p, vals, n * 4, cudaMemcpyHostToDevice, c->stream));
    bool in_b = false;
    TRY(radix_sort_u128(c, c->keys_a.p, c->keys_b.p, c->vals_a.p, c->vals_b.p, n, key_bits, &in_b, "u128"));
    CUDA_TRY(c, cudaMemcpyAsync(inter.data(), in_b ? c->keys_b.p : c->keys_a.p, n * 16, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(vals, in_b ? c->vals_b.p : c->vals_a.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    for (uint64_t i = 0; i < n; i++) { keys_lo[i] = inter[2 * i]; keys_hi[i] = inter[2 * i + 1]; }
    return ELP_OK;
}

}  // extern "C"
