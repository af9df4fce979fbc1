// ctx.h -- the device context behind the C ABI (include/elprep_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include "common.cuh"
#include "radix_sort.cuh"

// simple growable device buffer
template <class T> struct DBuf {
    T* p = nullptr;
    size_t cap = 0;   // elements
    cudaError_t reserve(size_t n, cudaStream_t s, size_t keep = 0) {   // keeps the first `keep` elements
        if (n <= cap) return cudaSuccess;
        size_t ncap = n + n / 8 + 64;
        T* q = nullptr;
        cudaError_t e = cudaMalloc(&q, ncap * sizeof(T));
        if (e != cudaSuccess) return e;
        if (p && keep) { e = cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, s); if (e != cudaSuccess) return e; }
        if (p) { cudaStreamSynchronize(s); cudaFree(p); }
        p = q; cap = ncap;
        return cudaSuccess;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// duplication metrics of one library (filters.DuplicatesCtr, mark-optical-duplicates.go:95-110): the seven counters in the
// reference's field order and the three count histograms (all, non-optical, optical)
struct DupCounters { int64_t ctr[7] = {0, 0, 0, 0, 0, 0, 0}; std::map<int64_t, int64_t> hist[3]; };
#define REFHOT_PAD 512
#define ARENA_FRONT_PAD 64   // QUAL / SEQ arenas start at this offset: kernels read aligned windows that may begin before a read
#define OPT_NCTR 8
#define OPT_HBINS 1024
#define OPT_OVF_CAP (1 << 16)

struct KernelStat { uint64_t launches = 0; double ms = 0, alg_bytes = 0; };
struct PendingEvent { std::string name; cudaEvent_t a, b; double alg_bytes; };

// dense BQSR table geometry: [n_cov][94][1 + (2*max_cycle+1) + 16][2]
struct TableGeom {
    int n_cov = 0, max_cycle = 500;
    __host__ __device__ int ncols() const { return 1 + (2 * max_cycle + 1) + 16; }
    __host__ __device__ size_t cells() const { return (size_t)n_cov * 94 * ncols(); }
    __host__ __device__ size_t idx(int cov, int q, int col) const { return ((size_t)cov * 94 + q) * ncols() + col; }
    __host__ __device__ int col_cycle(int cyc) const { return 1 + cyc + max_cycle; }
    __host__ __device__ int col_ctx(int ctx) const { return 1 + (2 * max_cycle + 1) + ctx; }
};

struct elp_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;   // upload / download streams of the asynchronous append / fetch
    cudaEvent_t ev_in = nullptr, ev_staged = nullptr, ev_out = nullptr;
    void* h_stage = nullptr; size_t stage_off = 0;        // page-locked staging of upload_small
    std::string err;
    std::mutex append_mu;
    bool profile = false;

    // ---- header-derived ----
    int n_contigs = 0;
    std::vector<int32_t> contig_len;
    std::vector<std::string> contig_names;
    int n_rg = 0;
    std::vector<int32_t> rg_lib, rg_cov;       // per @RG
    int n_lib = 0;
    std::vector<std::string> cov_names;
    std::vector<std::string> lib_names;       // [n_lib]
    int max_cycle = 500, quantize_levels = 0, optical_pixel_distance = 100;
    std::vector<uint8_t> sqq;
    std::string prefix = "GATK";
    int32_t* d_rg_lib = nullptr;     // [n_rg]
    int32_t* d_rg_cov = nullptr;     // [n_rg]
    int32_t* d_contig_len = nullptr; // [n_contigs]

    // ---- reference genome + known sites (device) ----
    std::vector<uint64_t> ref_len;
    std::vector<uint8_t*> d_refhot_raw;   // per contig: one-hot reference nibbles (bqsr_gather.cu pack_reference), payload at +REFHOT_PAD
    const uint8_t** d_refhot_ptrs = nullptr; // [n_contigs] device array of the payload pointers
    uint64_t* d_ref_len = nullptr;
    std::vector<int32_t*> d_sites;        // per contig, (start,end) pairs
    std::vector<uint64_t> n_sites;
    const int32_t** d_site_ptrs = nullptr;
    uint64_t* d_n_sites = nullptr;
    bool side_dirty = true;

    // ---- reads, arrival order (SoA columns) ----
    uint64_t n = 0, n_qname = 0, n_cigar = 0, n_qual = 0, n_seq = 0;
    DBuf<int32_t> refid, pos, nref, pnext, tlen, rg;
    DBuf<uint16_t> flag;
    DBuf<uint8_t> mapq;
    DBuf<uint8_t> optf;                       // elp_batch.opt_flags (ELP_OPT_SR ...)
    DBuf<uint64_t> qname_off, cigar_off, qual_off, seq_off;   // [n+1]
    DBuf<uint8_t> qname, seq, qual;
    DBuf<uint32_t> cigar;
    DBuf<uint8_t> bam_raw; DBuf<uint64_t> bam_off;   // staging of elp_append_bam: raw records and their offsets
    DBuf<uint8_t> bam_all; DBuf<uint64_t> bam_all_off; uint64_t n_bam = 0, bam_reads = 0;   // all raw records (for elp_fetch_bam) and the start of every read's record
    DBuf<uint64_t> bam_start;                 // starts of the records that pass the ingest filters
    uint32_t filter_mask = 0; int32_t filter_min_mapq = 0; uint64_t n_filtered = 0;   // elp_set_ingest_filter
    std::vector<int32_t*> d_regions; std::vector<uint64_t> n_regions; const int32_t** d_region_ptrs = nullptr; uint64_t* d_n_regions = nullptr; bool regions_dirty = true;   // target regions (BED) of RemoveNonOverlappingReads
    uint64_t n_cleaned = 0;                  // reads whose CIGAR elp_clean_sam rewrote
    uint8_t* d_rg_names = nullptr; uint32_t* d_rg_name_off = nullptr; std::vector<std::string> rg_ids;   // @RG IDs for the RG:Z match
    DBuf<int32_t> lseq_stage;       // staging for l_seq of the batch being appended
    DBuf<uint64_t> off_stage;       // staging for batch-relative offsets

    // ---- per-read temps (arrival order) ----
    DBuf<int32_t> upos, score;
    DBuf<uint64_t> qhash;
    DeviceRanges* d_ranges = nullptr;
    DeviceRanges h_ranges{};
    uint32_t* d_err = nullptr;       // device error word
    bool adapted = false;

    // ---- sort scratch ----
    DBuf<uint64_t> keys_a, keys_b;           // u64 keys, or u128 keys as pairs (2 words per key)
    DBuf<uint32_t> vals_a, vals_b;
    rs::Workspace ws;
    DBuf<uint32_t> mate;                      // [n] mate index or 0xffffffff
    DBuf<uint32_t> pair_a, pair_b, scan_tmp, scan_blk;
    DBuf<uint8_t> bytes_tmp;
    DBuf<uint4> bq_recs, bq_segs;             // BQSR count kernel: work records of the eligible reads, segment table
    uint32_t* d_bq_small = nullptr;           // class histogram, region bases, list counters, segment counts, work-queue heads
    uint32_t* d_qpresent = nullptr;           // [4] bit q set iff QUAL value q (0..127) occurs in the arena (maintained at ingest)

    // ---- output order ----
    bool sorted = false;                      // columns below valid
    DBuf<uint32_t> perm;                      // [n] arrival index of k-th output record
    DBuf<int32_t> s_refid, s_pos, s_nref, s_pnext, s_tlen, s_rg, s_lseq;
    DBuf<uint16_t> s_flag;
    DBuf<uint8_t> s_mapq, s_optf;
    DBuf<uint64_t> s_qual_off, s_seq_off, s_cigar_off, s_out_off;   // s_out_off[n+1]: offsets of the output qual stream
    DBuf<uint32_t> s_ncigar;
    DBuf<uint8_t> qual_out;                   // recalibrated QUAL in output order
    bool qual_out_valid = false;
    uint64_t qual_out_total = 0;              // bytes of the output QUAL stream

    // ---- BQSR ----
    TableGeom geom;
    int64_t* d_tables = nullptr;              // dense [cells][2]
    std::vector<int64_t> h_tables;
    std::vector<uint8_t> h_emp;               // [cells]
    bool gathered = false, finalized = false;
    uint64_t gather_eligible = 0;             // reads the last elp_bqsr_gather recalibrated (what the roofline line charges)
    uint8_t* d_lut = nullptr;                 // [n_cov][94][2*lut_maxcyc+1][17]
    int lut_maxcyc = 0;
    size_t lut_cap = 0;
    uint8_t* d_cov_exists = nullptr;          // [n_cov]
    uint8_t* d_clut = nullptr; uint16_t* d_rowtab = nullptr;   // compact apply table for the shared-memory kernel: [cycle][covariate][slot][17], QUAL -> slot offset
    uint32_t clut_bytes = 0, clut_blk = 0, clut_S17 = 0; int clut_Lc = 0; size_t clut_cap = 0; uint32_t clut_present[4] = {0, 0, 0, 0};
    std::vector<uint8_t> h_lut;               // the full apply table [n_cov][94][2*lut_maxcyc+1][17] on the host

    // ---- duplication metrics (optical.cu) ----
    void* d_opt_ctr = nullptr; void* d_opt_hist = nullptr; void* d_opt_ovf = nullptr; uint32_t* d_opt_small = nullptr;
    std::vector<DupCounters> opt;             // [n_lib + 1], slot 0 = "Unknown Library"
    bool opt_valid = false;

    // ---- several GPUs (comm.cu) ----
    void* comm = nullptr;                     // ncclComm_t
    int rank = 0, world = 1;
    int32_t* d_owner = nullptr;               // [n_contigs] rank owning each contig
    uint64_t n_ghost = 0, sp_sent_total = 0;  // visiting mates appended behind the local reads during duplicate marking; records this rank sent
    std::vector<uint32_t> sp_send, sp_recv;   // records to / from every rank
    DBuf<uint4> sp_sendbuf, sp_recvbuf; DBuf<uint32_t> sp_sent_idx;
    bool any_rank_entering = true;

    // ---- measurement ----
    uint64_t launches = 0;
    std::map<std::string, KernelStat> stats;
    std::vector<PendingEvent> pending;
    std::vector<cudaEvent_t> event_pool;
    cudaEvent_t timer_a = nullptr, timer_b = nullptr;

    int fail(int code, const char* fmt, ...) {
        char buf[1024];
        va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
        err = buf;
        return code;
    }
    // bracket one kernel launch: counts it and, when profiling, records a CUDA-event pair on the launching stream
    cudaEvent_t get_event() {
        if (!event_pool.empty()) { cudaEvent_t e = event_pool.back(); event_pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    void begin(const char* name, double alg_bytes) {
        launches++;
        if (!profile) return;
        PendingEvent pe; pe.name = name; pe.alg_bytes = alg_bytes; pe.a = get_event(); pe.b = get_event();
        cudaEventRecord(pe.a, stream);
        pending.push_back(pe);
    }
    void end() {
        if (!profile) return;
        cudaEventRecord(pending.back().b, stream);
    }
    void set_pending_bytes(const char* name, double bytes) { for (auto& pe : pending) if (pe.name == name) pe.alg_bytes = bytes; }
    void resolve_events() {
        if (pending.empty()) return;
        cudaStreamSynchronize(stream);
        for (auto& pe : pending) {
            float ms = 0; cudaEventElapsedTime(&ms, pe.a, pe.b);
            KernelStat& s = stats[pe.name]; s.launches++; s.ms += ms; s.alg_bytes += pe.alg_bytes;
            event_pool.push_back(pe.a); event_pool.push_back(pe.b);
        }
        pending.clear();
    }
};

#define CUDA_TRY(ctx, call)                                                                                   \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess) return (ctx)->fail(E_CUDA, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e__), __FILE__, __LINE__, cudaGetErrorString(e__)); \
    } while (0)

#define LAUNCH_CHECK(ctx) CUDA_TRY(ctx, cudaGetLastError())

// ---- internal phase entry points (implemented in the .cu files) ----
int radix_sort_u64(elp_ctx* c, uint64_t* keys_a, uint64_t* keys_b, uint32_t* vals_a, uint32_t* vals_b, uint64_t n, int key_bits, bool* result_in_b, const char* tag);
int radix_sort_u128(elp_ctx* c, uint64_t* keys_a, uint64_t* keys_b, uint32_t* vals_a, uint32_t* vals_b, uint64_t n, int key_bits, bool* result_in_b, const char* tag);
int exclusive_scan_u32_to_u64(elp_ctx* c, const uint32_t* in, uint64_t* out, uint64_t n);   // out[n+1]
int exclusive_scan_u64(elp_ctx* c, const uint64_t* in, uint64_t* out, uint64_t n, uint64_t base);          // out[n+1], out[0]=base
int phase_adapt(elp_ctx* c);
int phase_markdup(elp_ctx* c, bool optical);
int phase_optical(elp_ctx* c, uint64_t npairs, const uint64_t* sorted_keys, const uint32_t* sorted_vals, int bS);
int phase_coordinate_sort(elp_ctx* c, int order);   // 0 keep, 1 coordinate, 2 queryname
int phase_bqsr_gather(elp_ctx* c);
int phase_bqsr_finalize(elp_ctx* c, const char* report_path);
int phase_bqsr_apply(elp_ctx* c);
int build_apply_lut(elp_ctx* c, int Lc);   // bqsr_finalize.cu
int build_compact_lut(elp_ctx* c);
int upload_side_inputs(elp_ctx* c);
int pack_reference(elp_ctx* c, int contig, const uint8_t* bases, uint64_t n);   // bqsr_gather.cu
int check_device_errors(elp_ctx* c);
int upload_small(elp_ctx* c, void* dst, const void* src, size_t bytes);   // api.cu: host -> device without the copy engine
int comm_allreduce_ranges(elp_ctx* c);   // comm.cu
int spread_exchange_begin(elp_ctx* c);
int spread_exchange_end(elp_ctx* c);
int exclusive_scan_u64_from_u32(elp_ctx* c, const uint32_t* in, uint64_t* out, uint64_t n, uint64_t base);   // out[n+1], out[0] = base
int qual_presence_update(elp_ctx* c, uint64_t first_byte, uint64_t n_bytes);   // api.cu: called by both ingest paths
