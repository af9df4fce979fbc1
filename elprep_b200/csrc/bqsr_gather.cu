// bqsr_gather.cu -- BQSR covariate gather on the device (replaces (*BaseRecalibrator).Recalibrate,
// filters/bqsr.go:467-551, with the read clipping of filters/utils.go:130-534).
//
// The fast path (bqsr_prep2_kernel, bqsr_count_kernel: bqsr_count.inl) takes the reads whose clipping has a closed form when
// the QUAL alphabet is small.  The general kernels below take every read it refuses, or all reads when it does not apply,
// in output (coordinate) order:
//   bqsr_prep_kernel   one THREAD per read: recalibrateAln eligibility (:225-244), hardClipAdaptorSequence and
//                      hardClipSoftClippedBases on a private copy of the CIGAR (utils.go:148-534), the known-sites
//                      intersection and its read coordinates (calculateSkipSlice :389-414).  The serial, branchy CIGAR
//                      surgery runs 32 reads per warp instead of one; the result is a 48-byte descriptor per read.
//   gen_list_kernel    lists the eligible reads that bqsr_chunk_kernel<false> does not take.
//   bqsr_chunk_kernel  16 consecutive bases per lane: mismatch vs reference (computeSnpEvents :254-285), cycle (:376-387) and
//                      2-mer context (:64-146,312-362) covariates, and the table updates.  Observation and mismatch counters
//                      of the frequent QUAL values are privatised in shared memory per CTA (persistent CTAs, flushed once
//                      with 64-bit atomics); infrequent QUAL values go to the global table.  <false> takes the reads whose
//                      clipped CIGAR is one M run inside the contig; <true> the listed ones (insertions / deletions, more
//                      than 4 known-site ranges, cycles beyond --max-cycle, bases past the contig end).
// Kept bases keep their original alignment under hard clipping, so reference positions come from the ORIGINAL CIGAR
// offset by the clip start; only the known-sites mask needs the clipped CIGAR (its coordinate mapping has quirks).
// Table layout: dense int64 [n_cov][94][1 + (2*max_cycle+1) + 16][2] = (observations, mismatches); the
// QualityScores column is derived as the row sum of the Cycles columns (every counted base updates both).
#include <algorithm>
#include <vector>
#include "ctx.h"
#include "bqsr_simd.cuh"
#include "bqsr_lane.cuh"

namespace {

constexpr int MAXC = 64;        // CIGAR operations per read handled by the kernel
constexpr int MAXIT = 16;       // 32*MAXIT = 512 bases per clipped read (cycles beyond max_cycle=500 are an error anyway)

__device__ __forceinline__ int op_of(uint32_t c) { return (int)(c & 15); }
__device__ __forceinline__ int len_of(uint32_t c) { return (int)(c >> 4); }
__device__ __forceinline__ uint32_t mk(int len, int op) { return ((uint32_t)len << 4) | (uint32_t)op; }
// BAM op codes: M0 I1 D2 N3 S4 H5 P6 =7 X8
__device__ __forceinline__ int cons_read(int o) { return o == 0 || o == 1 || o == 4 || o == 7 || o == 8; }
__device__ __forceinline__ int cons_ref(int o) { return o == 0 || o == 2 || o == 3 || o == 7 || o == 8; }

struct Clip {          // working copy of one alignment (lane 0 only)
    int32_t pos; int nc; int s0, slen; int err;
    uint32_t* cg;      // shared memory, MAXC+4 entries
    uint32_t* tmp;     // shared memory, MAXC+4 entries
};

__device__ int32_t aln_end(const Clip& a) { int32_t l = 0; for (int i = 0; i < a.nc; i++) l += cons_ref(op_of(a.cg[i])) * len_of(a.cg[i]); return a.pos + l - 1; }
__device__ int soft_start(const Clip& a) { int32_t s = a.pos; for (int i = 0; i < a.nc; i++) { int o = op_of(a.cg[i]); if (o == 4) s -= len_of(a.cg[i]); else if (o != 5) break; } return s; }
__device__ int read_len(const uint32_t* cg, int nc) { int l = 0; for (int i = 0; i < nc; i++) l += cons_read(op_of(cg[i])) * len_of(cg[i]); return l; }

// computeReadCoordinateForReferenceCoordinate, filters/utils.go:267-326
__device__ int compute_read_coord(const uint32_t* cv, int nc, int softStart, int refIndex, int* falls) {
    const int goal = refIndex - softStart;
    *falls = 0;
    if (goal < 0) return -1;
    int readBases = 0, refBases = 0, fallsInside = 0, endsJustBefore = 0, fob = 0, index = 0;
    while (refBases != goal && index < nc) {
        const uint32_t el = cv[index]; index++;
        const int eo = op_of(el), elen = len_of(el);
        int shift = 0;
        if (cons_ref(eo) || eo == 4) { shift = (refBases + elen < goal) ? elen : goal - refBases; refBases += shift; }
        if (refBases != goal) readBases += cons_read(eo) * elen;
        else {
            if (shift >= elen && index == nc) return -1;
            int no = -1;
            if (shift < elen) fallsInside = (eo == 2 || eo == 3);
            else {
                uint32_t nx = cv[index]; index++;
                if (op_of(nx) == 1) { readBases += len_of(nx); if (index == nc) return -1; nx = cv[index]; index++; }
                no = op_of(nx);
                endsJustBefore = (no == 2 || no == 3);
            }
            fob = endsJustBefore || fallsInside;
            if (!fob) readBases += cons_read(eo) * shift;
            else if (endsJustBefore) readBases += cons_read(eo) * (shift - 1);
            else if (fallsInside || (endsJustBefore && (no == 2 || no == 3))) readBases--;
        }
    }
    if (refBases != goal) return -1;
    *falls = fob;
    return readBases;
}
// getReadCoordinateForReferenceCoordinate, filters/utils.go:335-349 (+ readStartsWithInsertion, bqsr.go:287-299)
__device__ int get_read_coord(const uint32_t* cv, int nc, int softStart, int refIndex, bool tail_right, bool* ok) {
    int falls; int rb = compute_read_coord(cv, nc, softStart, refIndex, &falls);
    if (rb == -1) { *ok = false; return -1; }
    if (tail_right && falls) rb++;
    if (!tail_right && rb == 0) {
        for (int i = 0; i < nc; i++) {
            const int o = op_of(cv[i]);
            if (o == 1) { const int fl = len_of(cv[i]), m = read_len(cv, nc) - 1; rb = fl < m ? fl : m; break; }
            if (o == 5 || o == 4) continue;
            break;
        }
    }
    *ok = true; return rb;
}
__device__ int hard_soft_offset(const uint32_t* c, int nc) {   // utils.go:351-371
    int size = 0, i = 0;
    for (; i < nc; i++) { if (op_of(c[i]) == 5) size += len_of(c[i]); else break; }
    for (; i < nc; i++) { if (op_of(c[i]) == 4) size += len_of(c[i]); else break; }
    return size;
}
__device__ __forceinline__ int clip_shift(uint32_t op, int cigarLength) {   // utils.go:377-386
    const int o = op_of(op);
    if (o == 1) return -cigarLength;
    if (o == 2 || o == 3) return len_of(op);
    return 0;
}
__device__ int clean_hard_clipped(uint32_t* c, int nc) {   // utils.go:473-504
    int total = 0, index = 0;
    for (; index < nc; index++) { const int o = op_of(c[index]); if (o == 5 || o == 2 || o == 3) total += len_of(c[index]); else break; }
    if (index > 0) { c[0] = mk(total, 5); for (int k = index; k < nc; k++) c[1 + k - index] = c[k]; nc = 1 + nc - index; }
    total = 0; index = nc - 1;
    for (; index >= 0; index--) { const int o = op_of(c[index]); if (o == 5 || o == 2 || o == 3) total += len_of(c[index]); else break; }
    if (index < nc - 1) { c[index + 1] = mk(total, 5); nc = index + 2; }
    return nc;
}
// hardClipCigar, utils.go:407-471: writes into a.tmp, returns the new op count
__device__ int hard_clip_cigar(const Clip& a, int start, int stop) {
    const uint32_t* cv = a.cg; const int nc = a.nc; uint32_t* out = a.tmp;
    int index = 0, total = stop - start + 1, ashift = 0, no = 0;
    if (start == 0) {
        int ci = 0;
        for (int k = 0; k < nc; k++) { ci = k; if (op_of(cv[k]) != 5) break; total += len_of(cv[k]); }
        for (; index <= stop && ci < nc; ci++) {
            const uint32_t op = cv[ci]; const int L = len_of(op), shift = cons_read(op_of(op)) * L;
            if (index + shift == stop + 1) { ashift += clip_shift(op, L); out[no++] = mk(total + ashift, 5); }
            else if (index + shift > stop + 1) {
                const int after = L - (stop - index + 1);
                ashift += clip_shift(op, stop - index + 1);
                out[no++] = mk(total + ashift, 5); out[no++] = mk(after, op_of(op));
            }
            index += shift;
            ashift += clip_shift(op, shift);
        }
        for (; ci < nc; ci++) out[no++] = cv[ci];
    } else {
        int ci = 0;
        for (; index < start && ci < nc; ci++) {
            const uint32_t op = cv[ci]; const int L = len_of(op), shift = cons_read(op_of(op)) * L;
            if (index + shift < start) out[no++] = op;
            else {
                const int after = start - index;
                ashift += clip_shift(op, L - (start - index));
                if (op_of(op) == 5) total += after; else out[no++] = mk(after, op_of(op));
            }
            index += shift;
        }
        for (; ci < nc; ci++) { const uint32_t op = cv[ci]; ashift += clip_shift(op, len_of(op)); if (op_of(op) == 5) total += len_of(op); }
        out[no++] = mk(total + ashift, 5);
    }
    return clean_hard_clipped(out, no);
}
// hardClip, utils.go:388-405 (the read is mapped here, so POS always shifts for left clips)
__device__ void hard_clip(Clip& a, int start, int stop) {
    const int ncl = hard_clip_cigar(a, start, stop);
    const int readLength = a.slen, newLength = readLength - (stop - start + 1);
    const int copyStart = (start == 0) ? stop + 1 : 0;
    if (newLength < 0 || copyStart + newLength > readLength) { a.err = 1; a.slen = 0; return; }
    const int shift = hard_soft_offset(a.tmp, ncl) - hard_soft_offset(a.cg, a.nc);
    a.s0 += copyStart; a.slen = newLength;
    for (int k = 0; k < ncl; k++) a.cg[k] = a.tmp[k];
    a.nc = ncl;
    if (start == 0) a.pos += shift;
}

// ---------------------------------------------------------------- per-read descriptor written by the prep kernel
struct __align__(16) ReadDesc {
    uint64_t qloc;            // QUAL arena offset of the first kept base | refid << 40
    uint64_t nloc;            // SEQ nibble index of the first kept base (2 * seq_off + c_s0)
    int32_t c_pos;            // POS after clipping (1-based)
    uint16_t c_s0, c_len;     // kept bases [c_s0, c_s0 + c_len) of the original read; c_len == 0: not recalibrated
    uint8_t flags, cov, n_skip, pad;
    uint32_t ovf;             // slot of the 512-bit skip bitmask when more than 4 known-site ranges hit the read
    uint16_t skip[4][2];      // inclusive [first,last] clipped read coordinates masked by known sites
};                            // 48 bytes = three 16-byte loads: location | scalars | skip ranges
constexpr uint8_t DF_REVERSED = 1, DF_LAST = 2, DF_SINGLE_M = 4, DF_SKIP_OVF = 8, DF_LEAN = 16;
constexpr int OVF_WORDS = 16;   // 512 bits

struct GatherArgs {
    uint64_t n;
    const int32_t *refid, *pos, *nref, *pnext, *tlen, *rg, *lseq; const uint16_t* flag; const uint8_t* mapq; const uint8_t* optf;
    const uint64_t *qual_off, *seq_off, *cigar_off; const uint32_t* ncigar;
    const uint32_t* cigar; const uint8_t *seq, *qual;
    const int32_t* rg_cov; int n_rg;
    const int32_t* contig_len; int n_contigs;
    const uint8_t* const* refhot; const uint64_t* ref_len;   // per contig: one-hot reference nibbles (A/C/G/T -> 1/2/4/8, else 0), low nibble first
    const int32_t* const* sites; const uint64_t* n_sites;
    TableGeom geom; unsigned long long* tables; uint32_t* err;
    ReadDesc* desc; uint32_t* ovf_bits; uint32_t* ovf_count; uint32_t ovf_cap;
    uint32_t* gen_list; uint32_t* gen_count;   // reads for the chunk kernel's GEN variant
    int lanes_per_read;              // chunk kernel: lanes (16-base chunks) reserved per read
    // shared-memory privatisation: observation counters of the frequent QUAL values live in shared memory
    int8_t qslot[94]; uint8_t slot_q[94]; int n_slots, Lc;
    int ncols_s, ctx_col_s;          // chunk kernel rows: skewed cycle cells [0, ctx_col_s), then 16 context cells
    const uint32_t* in_list; uint32_t n_in;   // when set: only these reads (the general path behind bqsr_prep2_kernel); they all go through the per-lane CIGAR walk
};

// ---------------------------------------------------------------- kernel A: one thread per read
__global__ void __launch_bounds__(128) bqsr_prep_kernel(GatherArgs A) {
    const uint64_t tix = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tix >= (A.in_list ? (uint64_t)A.n_in : A.n)) return;
    const uint64_t k = A.in_list ? (uint64_t)A.in_list[tix] : tix;
    ReadDesc d; d.qloc = 0; d.nloc = 0; d.c_pos = 0; d.c_s0 = 0; d.c_len = 0; d.flags = 0; d.cov = 0; d.n_skip = 0; d.pad = 0; d.ovf = 0;
#pragma unroll
    for (int r = 0; r < 4; r++) { d.skip[r][0] = 0; d.skip[r][1] = 0; }
    ReadDesc* out = A.desc + k;
    auto done = [&]() {
        const uint4* src = reinterpret_cast<const uint4*>(&d); uint4* dst = reinterpret_cast<uint4*>(out);
        dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2];
    };
    // ---- recalibrateAln, bqsr.go:225-244 ----
    const uint16_t f = A.flag[k];
    const uint8_t mq = A.mapq[k];
    const int32_t refid = A.refid[k], pos0 = A.pos[k], g = A.rg[k], L0 = A.lseq[k];
    const int nc0 = (int)A.ncigar[k];
    bool elig = !(A.optf[k] & 1u) &&       // the `sr` tag: a group-file copy of a spread read is never recalibrated (bqsr.go:225-229)
                (mq > 0 && mq < 255) && !(f & (F_SECONDARY | F_DUPLICATE | F_QCFAILED)) && !((f & F_UNMAPPED) || refid < 0 || pos0 == 0) && pos0 > 0 && L0 > 0 &&
                g >= 0 && g < A.n_rg && refid < A.n_contigs;
    if (elig && pos0 > A.contig_len[refid]) elig = false;            // alignmentAgreesWithHeader, utils.go:130-138
    if (!elig) { done(); return; }
    if (nc0 > MAXC) { atomicOr(A.err, DERR_CIGAR_LIMIT); done(); return; }
    uint32_t cg[MAXC + 4], tmp[MAXC + 4];
    const uint64_t coff = A.cigar_off[k];
    int bad = 0, rl = 0;
    for (int i = 0; i < nc0; i++) { const uint32_t op = A.cigar[coff + i]; cg[i] = op; const int o = op_of(op); bad |= (o == 3); rl += cons_read(o) * len_of(op); }
    if (bad || rl != L0) { done(); return; }                        // no N operation; SEQ length == read length from the CIGAR
    Clip a; a.pos = pos0; a.nc = nc0; a.s0 = 0; a.slen = L0; a.err = 0; a.cg = cg; a.tmp = tmp;
    {
        const int32_t pnext = A.pnext[k], tlen = A.tlen[k], nref = A.nref[k];
        // hardClipAdaptorSequence, utils.go:148-222
        bool well = false; int alnEnd = -1;
        const bool next_unmapped = (f & F_NEXTUNMAPPED) || nref < 0 || pnext == 0;   // isStrictNextUnmapped, utils.go:144
        if (tlen != 0 && (f & F_MULTIPLE) && !next_unmapped && (((f & F_REVERSED) != 0) != ((f & F_NEXTREVERSED) != 0))) {
            if (f & F_REVERSED) { alnEnd = aln_end(a); well = alnEnd > pnext; }
            else well = pos0 <= pnext + tlen;
        }
        if (well) {
            const int boundary = (f & F_REVERSED) ? (int)pnext - 1 : (int)pos0 + (tlen < 0 ? -tlen : tlen);
            if (boundary >= pos0) {
                if (alnEnd < 0) alnEnd = aln_end(a);
                if (boundary <= alnEnd) {
                    bool ok;
                    if (f & F_REVERSED) { const int stop = get_read_coord(a.cg, a.nc, soft_start(a), boundary, false, &ok); if (!ok) a.err = 2; else hard_clip(a, 0, stop); }
                    else { const int start = get_read_coord(a.cg, a.nc, soft_start(a), boundary, true, &ok); if (!ok) a.err = 2; else hard_clip(a, start, a.slen - 1); }
                }
            }
        }
        // hardClipSoftClippedBases, utils.go:506-534
        if (!a.err && a.slen > 0) {
            int readIndex = 0, cutLeft = -1, cutRight = -1; bool rightTail = false;
            for (int i = 0; i < a.nc; i++) {
                const int o = op_of(a.cg[i]), ln = len_of(a.cg[i]);
                if (o == 4) { if (rightTail) cutRight = readIndex; else cutLeft = readIndex + ln - 1; }
                else if (o != 5) rightTail = true;
                readIndex += cons_read(o) * ln;
            }
            if (cutRight >= 0) hard_clip(a, cutRight, a.slen - 1);
            if (!a.err && a.slen > 0 && cutLeft >= 0) hard_clip(a, 0, cutLeft);
        }
    }
    if (a.err) { atomicOr(A.err, DERR_CLIP); done(); return; }
    if (a.slen <= 0) { done(); return; }
    if (a.slen > 32 * MAXIT) { atomicOr(A.err, DERR_READLEN_LIMIT); done(); return; }
    const int L = a.slen;
    // is the clipped CIGAR a single M-type operation (plus hard clips)?
    int n_m = 0, n_other = 0;
    for (int i = 0; i < a.nc; i++) { const int o = op_of(a.cg[i]); if (o == 0 || o == 7 || o == 8) n_m++; else if (o != 5) n_other++; }
    d.c_pos = a.pos; d.c_s0 = (uint16_t)a.s0; d.c_len = (uint16_t)L; d.cov = (uint8_t)A.rg_cov[g];
    d.qloc = (A.qual_off[k] + (uint64_t)a.s0) | ((uint64_t)(uint32_t)refid << 40);
    d.nloc = A.seq_off[k] * 2 + (uint64_t)a.s0;
    d.flags = ((f & F_REVERSED) ? DF_REVERSED : 0) | ((f & F_LAST) ? DF_LAST : 0) | ((n_m == 1 && n_other == 0) ? DF_SINGLE_M : 0);
    // ---- known sites (calculateSkipSlice, bqsr.go:389-414): the clipped read has no S, so softStart/softEnd = POS / End ----
    const uint64_t ns = A.n_sites[refid];
    if (ns) {
        const int32_t* sv = A.sites[refid];
        int refl = 0;
        for (int i = 0; i < a.nc; i++) refl += cons_ref(op_of(a.cg[i])) * len_of(a.cg[i]);
        const int ss = a.pos, se = a.pos + refl - 1;
        // intervals.Intersect, intervals/intervals.go:166-173
        uint64_t lo = 0, hi = ns;
        while (lo < hi) { const uint64_t m = (lo + hi) >> 1; if (!(sv[2 * m + 1] >= ss)) lo = m + 1; else hi = m; }
        const uint64_t s0 = lo;
        uint64_t s1 = s0;
        while (s1 < ns && sv[2 * s1] <= se) s1++;
        if (s1 - s0 <= 4) {
            for (uint64_t s = s0; s < s1; s++) {
                bool ok; int fs = get_read_coord(a.cg, a.nc, ss, sv[2 * s], false, &ok);
                if (!ok || fs < 0) fs = 0;
                int fe = get_read_coord(a.cg, a.nc, ss, sv[2 * s + 1], false, &ok);
                if (!ok || fe > L - 1) fe = L - 1;
                if (fs <= fe) { d.skip[d.n_skip][0] = (uint16_t)fs; d.skip[d.n_skip][1] = (uint16_t)fe; d.n_skip++; }
            }
        } else {
            const uint32_t slot = atomicAdd(A.ovf_count, 1u);
            if (slot >= A.ovf_cap) { atomicOr(A.err, DERR_READLEN_LIMIT); done(); return; }
            uint32_t bits[OVF_WORDS];
            for (int i = 0; i < OVF_WORDS; i++) bits[i] = 0;
            for (uint64_t s = s0; s < s1; s++) {
                bool ok; int fs = get_read_coord(a.cg, a.nc, ss, sv[2 * s], false, &ok);
                if (!ok || fs < 0) fs = 0;
                int fe = get_read_coord(a.cg, a.nc, ss, sv[2 * s + 1], false, &ok);
                if (!ok || fe > L - 1) fe = L - 1;
                for (int i = fs; i <= fe; i++) bits[i >> 5] |= 1u << (i & 31);
            }
            for (int i = 0; i < OVF_WORDS; i++) A.ovf_bits[(size_t)slot * OVF_WORDS + i] = bits[i];
            d.flags |= DF_SKIP_OVF; d.ovf = slot;
        }
    }
    // chunk kernel without a list: one M run, every cycle inside --max-cycle (|cycle| <= L), inside the contig.  Every read fits
    // the lanes of a read: L <= min(512, lseq_max) <= CHUNK * lanes_per_read.
    if (!A.in_list && (d.flags & DF_SINGLE_M) && !(d.flags & DF_SKIP_OVF) && L <= A.geom.max_cycle &&
        (uint64_t)(a.pos - 1) + (uint64_t)L <= A.ref_len[refid]) d.flags |= DF_LEAN;
    done();
}

// rare per-base events, out of line: QUAL without a shared-memory slot, QUAL > 93, a cycle beyond --max-cycle
// (checkCycleCovariate, bqsr.go:364-369)
__device__ __noinline__ void count_rare(const GatherArgs& A, int cov, int q, int cyc, uint32_t ctx, bool okc, uint32_t snp, uint32_t* errbits) {
    const uint32_t e = (q > 93 ? DERR_QUAL_RANGE : 0u) | (cyc > A.geom.max_cycle || cyc < -A.geom.max_cycle ? DERR_CYCLE : 0u);
    if (e) { *errbits |= e; return; }
    atomicAdd(A.tables + 2 * A.geom.idx(cov, q, A.geom.col_cycle(cyc)), 1ull);
    if (okc) atomicAdd(A.tables + 2 * A.geom.idx(cov, q, A.geom.col_ctx((int)ctx)), 1ull);
    if (snp) {
        atomicAdd(A.tables + 2 * A.geom.idx(cov, q, A.geom.col_cycle(cyc)) + 1, 1ull);
        if (okc) atomicAdd(A.tables + 2 * A.geom.idx(cov, q, A.geom.col_ctx((int)ctx)) + 1, 1ull);
    }
}

// shared memory through explicit 32-bit shared-window addresses (generic pointers cost an address conversion per access)
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void reds_inc(uint32_t a) { asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(a) : "memory"); }
__device__ __forceinline__ void reds_add(uint32_t a, uint32_t v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

// ---------------------------------------------------------------- kernel B: 16 consecutive bases per lane (the common case)
// Reads whose clipped CIGAR is one M run (DF_LEAN, > 90 % of a WGS sample).  A warp takes 32 / lanes_per_read consecutive
// reads per step; lane (r, c) owns bases [16c, 16c+16) of read r.  Everything per base is SIMD inside 32/64-bit words:
//   QUAL    16 bytes  (unaligned 16-byte window out of two aligned 128-bit loads)
//   SEQ     16 BAM nibbles -> base codes 0..3 / 8 by bit arithmetic, 4 bits per base
//   REF     16 one-hot reference nibbles (pack_reference); the read's BAM nibbles are one-hot for A/C/G/T too: mismatch = XOR
//   context previous base in sequencing direction by shifting the code word one nibble (edge nibble from the neighbour lane)
//   masks   counted / context-valid / mismatch / known-site flags as one bit per nibble
// leaving ~14 instructions per base for the two shared-memory increments (cycle, context).  The cycle column of a
// shared-memory row is skewed (cell c lives at c + c/16): the lanes of a read sit 16 cycles apart, which would otherwise
// put them all on two banks.
struct ChunkSmem { uint32_t obs, mis, qslot; };   // shared-window byte addresses

#ifndef CHUNK_MINB
#define CHUNK_MINB 4
#endif
// GEN: every eligible read that is not DF_LEAN, from a list.  The reference window of a lane comes from a walk of the CIGAR
// (insertions / deletions, bases past the contig end); known sites may come as the 512-bit mask (DF_SKIP_OVF); a read longer
// than --max-cycle takes its cycles past the shared-memory rows, so all its counted bases go to the global table.
template <bool GEN>
__global__ void __launch_bounds__(256, CHUNK_MINB) bqsr_chunk_kernel(GatherArgs A, const uint32_t* __restrict__ list, uint32_t n_list) {
    extern __shared__ uint32_t sm_tab[];
    // QUAL -> row of the CTA's tables: bits 0..5 = shared-memory slot, or n_slots = the trash row (updates that must not
    // count land there, which keeps the per-base code free of predicates); bit 6: QUAL < 6 (never counted, bqsr.go:506);
    // bit 7: counted but without a slot (or QUAL > 93) -> the chunk is redone base by base in the slow tail
    __shared__ uint8_t sm_qslot[256];
    __shared__ unsigned long long sm_ge[CHUNK + 1], sm_le[CHUNK + 1];   // nibble flags for index >= k / index <= k - 1
    const unsigned lane = lane_id();
    const int rows = A.n_slots + 1;
    const int cells = A.geom.n_cov * rows * A.ncols_s;
    uint32_t* sm_mis = sm_tab + cells;
    for (int i = threadIdx.x; i < 2 * cells; i += blockDim.x) sm_tab[i] = 0;
    {
        const int b = threadIdx.x;
        uint8_t v = (uint8_t)A.n_slots;
        if (b < 6) v |= 0x40; else if (b < 94 && A.qslot[b] >= 0) v = (uint8_t)A.qslot[b]; else v |= 0x80;
        sm_qslot[b] = v;
        if (b <= CHUNK) { sm_ge[b] = b == CHUNK ? 0ull : (ONES << (4 * b)); sm_le[b] = b == 0 ? 0ull : (ONES >> (4 * (CHUNK - b))); }
    }
    __syncthreads();
    const uint32_t s_ge = (uint32_t)__cvta_generic_to_shared(sm_ge), s_le = (uint32_t)__cvta_generic_to_shared(sm_le);
    // one flag per nibble for the bases lo..hi of a chunk (empty if lo > hi): two shared-memory look-ups
    auto range16 = [&](int lo, int hi) -> unsigned long long {
        unsigned long long ge, le;
        asm volatile("ld.shared.u64 %0, [%1];" : "=l"(ge) : "r"(s_ge + 8u * (uint32_t)min(max(lo, 0), CHUNK)));
        asm volatile("ld.shared.u64 %0, [%1];" : "=l"(le) : "r"(s_le + 8u * (uint32_t)min(max(hi + 1, 0), CHUNK)));
        return ge & le;
    };
    ChunkSmem S;
    S.obs = (uint32_t)__cvta_generic_to_shared(sm_tab); S.mis = (uint32_t)__cvta_generic_to_shared(sm_mis); S.qslot = (uint32_t)__cvta_generic_to_shared(sm_qslot);
    const int Lc = A.Lc, lpr = A.lanes_per_read, rpw = 32 / lpr;
    const uint32_t row_bytes = (uint32_t)A.ncols_s * 4u, ctx_off = (uint32_t)A.ctx_col_s * 4u;
    const int r = (int)lane / lpr, c = (int)lane - r * lpr;                     // read slot inside the warp step, chunk inside the read
    const bool lane_used = r < rpw;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    const uint64_t wid = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint4* dbase = reinterpret_cast<const uint4*>(A.desc);
    uint32_t errbits = 0;
    // descriptors are fetched one step ahead
    const uint64_t n_items = GEN ? (uint64_t)n_list : A.n;
    auto read_of = [&](uint64_t item) -> uint64_t { return GEN ? (uint64_t)__ldg(list + item) : item; };
    uint64_t k = wid * rpw + (uint64_t)r;
    uint4 nloc = make_uint4(0, 0, 0, 0), nsc = make_uint4(0, 0, 0, 0);
    uint64_t nread = 0;
    if (lane_used && k < n_items) { nread = read_of(k); nloc = __ldg(dbase + 3 * nread); nsc = __ldg(dbase + 3 * nread + 1); }
    for (uint64_t k0 = wid * rpw; k0 < n_items; k0 += warps * rpw) {
        const uint4 loc = nloc, sc = nsc;
        const uint64_t item = k0 + (uint64_t)r, inext = item + warps * rpw;
        const uint64_t kcur = nread;
        const bool have = lane_used && item < n_items;
        nloc = make_uint4(0, 0, 0, 0); nsc = nloc;
        if (lane_used && inext < n_items) { nread = read_of(inext); nloc = __ldg(dbase + 3 * nread); nsc = __ldg(dbase + 3 * nread + 1); }
        const uint32_t flags = sc.z & 0xff;
        const int L = (have && (GEN || (flags & DF_LEAN))) ? (int)(sc.y >> 16) : 0;   // 0: nothing to do for this lane group
        const int i0 = c * CHUNK, nb = min(max(L - i0, 0), CHUNK);                      // bases of this chunk
        const bool rev = flags & DF_REVERSED;
        // ---- loads ----
        uint32_t Q[4] = {0, 0, 0, 0};
        unsigned long long C = 0, X = 0, pastf = 0;   // X: read nibbles XOR reference nibbles, non-zero where they differ
        if (nb > 0) {
            const uint64_t qloc = ((uint64_t)loc.y << 32) | loc.x, nl = ((uint64_t)loc.w << 32) | loc.z;
            const uint32_t refid = (uint32_t)(qloc >> 40);
            load16_unaligned(A.qual + (qloc & ((1ull << 40) - 1)) + (uint64_t)i0, Q);
            const unsigned long long nibs = load16_nibbles_bam(A.seq, nl + (uint64_t)i0);
            C = (unsigned long long)codes_of((uint32_t)nibs) | ((unsigned long long)codes_of((uint32_t)(nibs >> 32)) << 32);
            unsigned long long R = 0;
            if (!GEN) R = load16_nibbles_le(A.refhot[refid], (uint64_t)((int64_t)(int32_t)sc.x - 1 + i0));
            else {
                // computeSnpEvents (bqsr.go:254-285) over the ORIGINAL alignment (kept bases keep their positions under hard
                // clipping): find the operation holding the chunk's first base; a chunk inside one M run is one window load,
                // a chunk that touches an insertion / deletion takes its reference codes base by base
                const uint64_t coff = A.cigar_off[kcur]; const int nc = (int)A.ncigar[kcur];
                const int oi0 = (int)(sc.y & 0xffff) + i0;                    // read offset in the stored (unclipped) read
                int ri = 0, ci = 0, oplen = 0, opk = -1; int64_t j = (int64_t)A.pos[kcur] - 1;
                for (; ci < nc; ci++) {
                    const uint32_t op = __ldg(A.cigar + coff + ci); const int o = op_of(op), ln = len_of(op);
                    if (cons_read(o)) { if (oi0 < ri + ln) { opk = o; oplen = ln; break; } ri += ln; }
                    if (o == 0 || o == 7 || o == 8 || o == 2 || o == 3) j += ln;
                }
                const int64_t reflen = (int64_t)A.ref_len[refid];
                const bool mtype = opk == 0 || opk == 7 || opk == 8;
                if (mtype && oi0 + nb <= ri + oplen && j + (oi0 - ri) + nb <= reflen) R = load16_nibbles_le(A.refhot[refid], (uint64_t)(j + (oi0 - ri)));
                else {
                    const uint8_t* rh = A.refhot[refid];
                    int rem = opk < 0 ? 0 : ri + oplen - oi0;                   // bases left in the current operation
                    int64_t jj = j + (mtype ? (oi0 - ri) : 0);
                    bool m = mtype;
                    for (int b = 0; b < nb; b++) {
                        while (rem == 0 && ci + 1 < nc) {                      // next read-consuming operation (deletions move the reference)
                            ci++;
                            const uint32_t op = __ldg(A.cigar + coff + ci); const int o = op_of(op), ln = len_of(op);
                            if (o == 2 || o == 3) { jj += ln; continue; }
                            if (cons_read(o)) { rem = ln; m = (o == 0 || o == 7 || o == 8); }
                        }
                        unsigned long long rc = (nibs >> (4 * b)) & 15ull;      // no reference base (insertion): never a mismatch
                        if (m) {
                            if (jj >= reflen) pastf |= 1ull << (4 * b);
                            else rc = (unsigned long long)((__ldg(rh + (jj >> 1)) >> (4 * (int)(jj & 1))) & 15u);
                            jj++;
                        }
                        R |= rc << (4 * b);
                        rem--;
                    }
                }
            }
            X = nibs ^ R;
        }
        if (nb < CHUNK) { const unsigned long long inlen = range16(0, nb - 1); C = (C & (inlen * 15ull)) | ((ONES & ~inlen) << 3); }   // codes past the read end: 8
        // ---- low-quality tails (computeStrandedClippedSeq, bqsr.go:312-331): first / last base with QUAL > 2 ----
        int first, last;
        qual_gt2_span(Q, nb, i0, first, last);
        // the lanes of one read reduce among themselves (segmented by member mask)
        const unsigned gmask = lane_used ? ((lpr == 32 ? 0xffffffffu : ((1u << lpr) - 1u)) << (r * lpr)) : (1u << lane);
        const int leftPos = __reduce_min_sync(gmask, first), rightPos = __reduce_max_sync(gmask, last);
        // neighbour chunks' edge codes for the context of the first / last base of this chunk
        const uint32_t c_hi = (uint32_t)(C >> 32), c_lo = (uint32_t)C;
        uint32_t edge_prev = __shfl_up_sync(FULL_MASK, c_hi, 1) >> 28, edge_next = __shfl_down_sync(FULL_MASK, c_lo, 1) & 15u;
        if (c == 0) edge_prev = 8; if (c == lpr - 1 || lane == 31) edge_next = 8;
        if (L > 0) {   // (warp-level primitives are above this line)
        // ---- per-base flags, one bit per nibble ----
        const unsigned long long Pn = rev ? ((C >> 4) | ((unsigned long long)edge_next << 60)) : ((C << 4) | edge_prev);   // previous base in sequencing direction
        const unsigned long long M3 = 0x3333333333333333ull, xr = rev ? M3 : 0ull;
        const unsigned long long ctxw = ((Pn ^ xr) & M3) | (((C ^ xr) & M3) << 2);          // key>>4 = prev | cur<<2, complemented for reverse reads (bqsr.go:64-76)
        const int wlo = rev ? leftPos : leftPos + 1, whi = rev ? rightPos - 1 : rightPos;      // bases whose context lies inside [leftPos, rightPos]
        unsigned long long skipf = 0;
        const uint32_t n_skip = (sc.z >> 16) & 0xff;
        if (n_skip) {
            const uint4 sk = __ldg(dbase + 3 * kcur + 2);   // (kcur: read index of this lane group)
            const uint32_t skv[4] = {sk.x, sk.y, sk.z, sk.w};
#pragma unroll
            for (int t = 0; t < 4; t++) if (t < (int)n_skip) skipf |= range16((int)(skv[t] & 0xffff) - i0, (int)(skv[t] >> 16) - i0);
        } else if (GEN && (flags & DF_SKIP_OVF)) {
            // more than 4 ranges: the chunk's 16 bits of the read's 512-bit mask (i0 is a multiple of 16: one word), one flag per nibble
            unsigned long long x = (__ldg(A.ovf_bits + (size_t)sc.w * OVF_WORDS + (i0 >> 5)) >> (i0 & 31)) & 0xffffull;
            x = (x | x << 24) & 0x000000FF000000FFull;
            x = (x | x << 12) & 0x000F000F000F000Full;
            x = (x | x << 6) & 0x0303030303030303ull;
            skipf = (x | x << 3) & ONES;
        }
        const unsigned long long counted = ~(C >> 3) & ONES & ~skipf;                             // ACGT, inside the read, not a known site (QUAL >= 6 via the slot table)
        const unsigned long long okc = counted & ~((Pn | C) >> 3) & range16(wlo - i0, whi - i0);
        const unsigned long long snpf = (X | (X >> 1) | (X >> 2) | (X >> 3)) & counted;         // computeSnpEvents, bqsr.go:254-285
        if (GEN && (pastf & counted)) errbits |= DERR_REFEND;                                   // a counted base beyond the end of its contig
        if (counted) {
        // ---- table updates ----
        const uint32_t cov = (sc.z >> 8) & 0xff;
        const int lastf = (flags & DF_LAST) ? 1 : 0;
        const int rof = 1 - 2 * lastf, inc = rev ? -rof : rof, cf = rof + (rev ? (L - 1) * rof : 0);   // prepareCycleCovariates, bqsr.go:376-383
        const int ci0 = cf + i0 * inc + Lc;                                                          // cycle cell of the chunk's first base
        const uint32_t obs0 = S.obs + cov * (uint32_t)rows * row_bytes;
        const uint32_t cnt_w[2] = {(uint32_t)counted, (uint32_t)(counted >> 32)}, okc_w[2] = {(uint32_t)okc, (uint32_t)(okc >> 32)};
        const uint32_t ctx_w[2] = {(uint32_t)ctxw, (uint32_t)(ctxw >> 32)};
        const uint32_t obs_ctx = obs0 + ctx_off;
        // a read longer than --max-cycle has cycles beyond the shared-memory rows (|cycle| <= Lc): all its counted bases take the slow tail
        const bool global_only = GEN && L > A.geom.max_cycle;
        uint32_t racc = 0;
        if (!global_only) {
            int ci = ci0;
#pragma unroll
            for (int j = 0; j < CHUNK; j++) {
                // no predicates and no branches: a base that is not counted adds 0, a QUAL without a slot adds to the trash row
                const uint32_t q = (Q[j >> 2] >> (8 * (j & 3))) & 0xffu;
                const uint32_t lut = lds_u8(S.qslot + q);
                const uint32_t roff = (lut & 0x3fu) * row_bytes;
                const uint32_t a1 = obs0 + roff + (uint32_t)(ci + (ci >> 4)) * 4u;
                const uint32_t nib4 = (j & 7) == 0 ? ((ctx_w[j >> 3] << 2) & 0x3cu) : ((ctx_w[j >> 3] >> (4 * (j & 7) - 2)) & 0x3cu);
                const uint32_t a2 = obs_ctx + roff + nib4;
                reds_add(a1, (cnt_w[j >> 3] >> (4 * (j & 7))) & 1u);
                reds_add(a2, (okc_w[j >> 3] >> (4 * (j & 7))) & 1u);
                racc |= lut;
                ci += inc;
            }
        }
        // slow tail: mismatches (sparse) and, if some base of the chunk has a QUAL without a shared-memory slot, all counted bases
        unsigned long long later = (global_only || (racc & 0x80u)) ? counted : snpf;
        while (later) {
            const int j = (__ffsll((long long)later) - 1) >> 2;
            later &= ~(15ull << (4 * j));
            const uint32_t qw = j < 4 ? Q[0] : (j < 8 ? Q[1] : (j < 12 ? Q[2] : Q[3]));
            const uint32_t q = (qw >> (8 * (j & 3))) & 0xffu;
            const uint32_t lut = lds_u8(S.qslot + q);
            const int cj = ci0 + j * inc;
            const uint32_t ctx = (uint32_t)((ctxw >> (4 * j)) & 15ull);
            const bool ok = (okc >> (4 * j)) & 1ull, snp = (snpf >> (4 * j)) & 1ull;
            const bool slotted = !global_only && !(lut & 0x80u);
            if ((lut & 0x40u) || (slotted && !snp)) continue;   // QUAL < 6: not counted; slotted match: done in the fast loop
            if (slotted) {     // a mismatch (sparse, ~0.5 % of bases) on the CTA's second table
                const uint32_t mrow = S.mis + (cov * (uint32_t)rows + (lut & 0x3fu)) * row_bytes;
                reds_inc(mrow + (uint32_t)(cj + (cj >> 4)) * 4u);
                if (ok) reds_inc(mrow + ctx_off + ctx * 4u);
            } else count_rare(A, (int)cov, (int)q, cj - Lc, ctx, ok, snp ? 1u : 0u, &errbits);
        }
        }
        }
    }
    errbits = __reduce_or_sync(FULL_MASK, errbits);
    if (errbits && lane == 0) atomicOr(A.err, errbits);
    __syncthreads();
    const int ncols_s = A.ncols_s, ctx_col = A.ctx_col_s;
    for (int i = threadIdx.x; i < cells; i += blockDim.x) {
        const uint32_t v = sm_tab[i], e = sm_mis[i];
        if (!(v | e)) continue;
        const int col_s = i % ncols_s, cs = i / ncols_s, slot = cs % rows, cov = cs / rows;
        if (slot == A.n_slots) continue;   // trash row
        int col_g;
        if (col_s < ctx_col) { const int cyc_cell = 16 * (col_s / 17) + col_s % 17; col_g = A.geom.col_cycle(cyc_cell - Lc); }   // undo the skew
        else col_g = A.geom.col_ctx(col_s - ctx_col);
        if (v) atomicAdd(A.tables + 2 * A.geom.idx(cov, A.slot_q[slot], col_g), (unsigned long long)v);
        if (e) atomicAdd(A.tables + 2 * A.geom.idx(cov, A.slot_q[slot], col_g) + 1, (unsigned long long)e);
    }
}

// work list of the eligible reads that are not DF_LEAN, for the chunk kernel's GEN variant.  One global atomic per block.
__global__ void __launch_bounds__(256) gen_list_kernel(GatherArgs A) {
    __shared__ uint32_t s_cnt, s_base;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const uint64_t tix = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in = tix < (A.in_list ? (uint64_t)A.n_in : A.n);
    const uint64_t k = in ? (A.in_list ? (uint64_t)A.in_list[tix] : tix) : 0;
    bool want = false;
    if (in) { const uint4 sc = __ldg(reinterpret_cast<const uint4*>(A.desc) + 3 * k + 1); want = (sc.y >> 16) != 0 && !(sc.z & DF_LEAN); }
    const unsigned b = __ballot_sync(FULL_MASK, want);
    uint32_t wb = 0;
    if (b && lane_id() == 0) wb = atomicAdd(&s_cnt, (uint32_t)__popc(b));
    wb = __shfl_sync(FULL_MASK, wb, 0);
    __syncthreads();
    if (threadIdx.x == 0 && s_cnt) s_base = atomicAdd(A.gen_count, s_cnt);
    __syncthreads();
    if (want) A.gen_list[s_base + wb + __popc(b & lanemask_lt())] = (uint32_t)k;
}

// QUAL value histogram of a prefix of the QUAL arena: picks which values get shared-memory slots
__global__ void __launch_bounds__(256) qual_sample_kernel(const uint8_t* __restrict__ qual, uint64_t n, uint32_t* __restrict__ hist) {
    __shared__ uint32_t sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) atomicAdd(&sh[qual[i]], 1u);
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

// QualityScores[(rg,q)] = sum over cycles of Cycles[(rg,q,cycle)] (each counted base updates both, bqsr.go:518-529)
__global__ void derive_q_kernel(TableGeom geom, long long* tables) {
    const int row = blockIdx.x;   // cov*94 + q
    long long obs = 0, mis = 0;
    const size_t base = (size_t)row * geom.ncols();
    for (int c = 1 + threadIdx.x; c < 1 + 2 * geom.max_cycle + 1; c += blockDim.x) { obs += tables[2 * (base + c)]; mis += tables[2 * (base + c) + 1]; }
    __shared__ long long so[8], sm[8];
    for (int o = 16; o; o >>= 1) { obs += __shfl_xor_sync(FULL_MASK, obs, o); mis += __shfl_xor_sync(FULL_MASK, mis, o); }
    if ((threadIdx.x & 31) == 0) { so[threadIdx.x >> 5] = obs; sm[threadIdx.x >> 5] = mis; }
    __syncthreads();
    if (threadIdx.x == 0) { long long a = 0, b = 0; for (int i = 0; i < (int)(blockDim.x >> 5); i++) { a += so[i]; b += sm[i]; } tables[2 * base] = a; tables[2 * base + 1] = b; }
}

#include "bqsr_count.inl"

}  // namespace

// the reference bases of one contig -> one-hot nibbles, the only device copy of the genome (read by the chunk and count kernels).
// REFHOT_PAD bytes in front (windows of reads at the start of a contig and the shifted window of an insertion start before
// base 0), 64 behind.  The bases pass through a device buffer that is freed before the call returns.
int pack_reference(elp_ctx* c, int contig, const uint8_t* bases, uint64_t n) {
    const uint64_t n_out = (n + 1) / 2;
    if (c->d_refhot_raw[contig]) { cudaFree(c->d_refhot_raw[contig]); c->d_refhot_raw[contig] = nullptr; }
    c->ref_len[contig] = 0; c->side_dirty = true;
    CUDA_TRY(c, cudaMalloc(&c->d_refhot_raw[contig], n_out + REFHOT_PAD + 64));
    CUDA_TRY(c, cudaMemsetAsync(c->d_refhot_raw[contig], 0, n_out + REFHOT_PAD + 64, c->stream));
    uint8_t* d_bases = nullptr;
    cudaError_t e = cudaSuccess;
    if (n) {
        CUDA_TRY(c, cudaMalloc(&d_bases, n));
        e = cudaMemcpyAsync(d_bases, bases, n, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) {
            c->launches++;
            ref_pack_hot_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, c->stream>>>(d_bases, n, c->d_refhot_raw[contig] + REFHOT_PAD, n_out);
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (d_bases) cudaFree(d_bases);
    CUDA_TRY(c, e);
    c->ref_len[contig] = n;
    return E_OK;
}

namespace {

// the general kernels (prep -> descriptors -> chunk kernels with shared-memory counters) over all reads (in_list == nullptr) or over
// the list bqsr_prep2_kernel left for them
int gather_general(elp_ctx* c, GatherArgs A, const uint32_t* in_list, uint32_t n_in, double bytes) {
    const uint64_t n = c->n;
    const uint64_t n_work = in_list ? (uint64_t)n_in : n;
    if (!n_work) return E_OK;
    const int Lc = std::max(1, std::min(c->max_cycle, c->h_ranges.lseq_max));
    A.Lc = Lc; A.ctx_col_s = 2 * Lc + ((2 * Lc) >> 4) + 1; A.ncols_s = A.ctx_col_s + 16;
    A.lanes_per_read = std::min(32, std::max(1, (c->h_ranges.lseq_max + CHUNK - 1) / CHUNK));
    A.in_list = in_list; A.n_in = n_in;
    for (int q = 0; q < 94; q++) { A.qslot[q] = -1; A.slot_q[q] = 0; }
    {
        // slot map: the most frequent QUAL values >= 6 of a sample get shared-memory counters (<= 48 KB per CTA)
        CUDA_TRY(c, c->scan_tmp.reserve(256 + 4, c->stream));
        CUDA_TRY(c, cudaMemsetAsync(c->scan_tmp.p, 0, 256 * 4, c->stream));
        const uint64_t ns = std::min<uint64_t>(c->n_qual, 8u << 20);
        c->begin("bqsr_g_qual_sample", (double)ns);
        qual_sample_kernel<<<64, 256, 0, c->stream>>>(c->qual.p, ns, c->scan_tmp.p);
        c->end(); LAUNCH_CHECK(c);
        uint32_t h[256];
        CUDA_TRY(c, cudaMemcpyAsync(h, c->scan_tmp.p, sizeof h, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        std::vector<int> qs;
        for (int q = 6; q < 94; q++) if (h[q]) qs.push_back(q);
        std::sort(qs.begin(), qs.end(), [&](int a, int b) { return h[a] != h[b] ? h[a] > h[b] : a < b; });
        const size_t per_slot = (size_t)std::max(1, c->geom.n_cov) * A.ncols_s * 4;
        const int max_slots = (int)std::min<size_t>(63, (48 * 1024) / (2 * per_slot)) - 1;   // observation + mismatch tables, one trash row each
        A.n_slots = std::max(0, std::min<int>((int)qs.size(), max_slots));
        for (int s = 0; s < A.n_slots; s++) { A.qslot[qs[s]] = (int8_t)s; A.slot_q[s] = (uint8_t)qs[s]; }
    }
    const size_t smem = (size_t)c->geom.n_cov * (A.n_slots + 1) * A.ncols_s * 4 * 2;
    int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
    // descriptors (48 B/read, indexed by read) and the overflow skip bitmasks live in scratch buffers that are free in this phase
    CUDA_TRY(c, c->keys_a.reserve(n * 6 + 8, c->stream));
    CUDA_TRY(c, c->vals_b.reserve(n + 8, c->stream));
    A.gen_list = c->vals_b.p;
    A.desc = reinterpret_cast<ReadDesc*>(c->keys_a.p);
    A.ovf_cap = (uint32_t)std::min<uint64_t>(n, (n >> 4) + 4096);
    CUDA_TRY(c, c->vals_a.reserve((size_t)A.ovf_cap * OVF_WORDS + 8, c->stream));
    A.ovf_bits = c->vals_a.p;
    A.ovf_count = c->scan_tmp.p;   // two u32 (overflow slots, GEN chunk reads), zeroed below
    A.gen_count = c->scan_tmp.p + 1;
    CUDA_TRY(c, cudaMemsetAsync(A.ovf_count, 0, 8, c->stream));
    c->begin("bqsr_g_prep", (double)n_work * (4 * 7 + 2 + 1 + 8 + 8 + 4 + 48) + (double)c->n_cigar * 4 * ((double)n_work / (double)n));
    bqsr_prep_kernel<<<(unsigned)((n_work + 127) / 128), 128, 0, c->stream>>>(A);
    c->end(); LAUNCH_CHECK(c);
    c->begin("bqsr_g_gen_list", (double)n_work * 20);
    gen_list_kernel<<<(unsigned)((n_work + 255) / 256), 256, 0, c->stream>>>(A);
    c->end(); LAUNCH_CHECK(c);
    const uint64_t rpw = 32 / A.lanes_per_read;
    CUDA_TRY(c, cudaFuncSetAttribute(bqsr_chunk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
    CUDA_TRY(c, cudaFuncSetAttribute(bqsr_chunk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
    if (!in_list) {
        const uint64_t steps = (n + rpw - 1) / rpw;
        uint64_t grid = std::min<uint64_t>((steps + 7) / 8, (uint64_t)sms * CHUNK_MINB);
        grid = std::max<uint64_t>(grid, (n + (4u << 20) - 1) / (4u << 20));   // <= 4 M reads per CTA keeps the 32-bit shared counters far from overflow
        c->begin("bqsr_g_chunk", bytes);
        bqsr_chunk_kernel<false><<<(unsigned)grid, 256, smem, c->stream>>>(A, nullptr, 0);
        c->end(); LAUNCH_CHECK(c);
    }
    uint32_t n_gen = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&n_gen, A.gen_count, 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    if (n_gen) {
        const uint64_t steps_g = ((uint64_t)n_gen + rpw - 1) / rpw;
        const uint64_t grid_g = std::min<uint64_t>((steps_g + 7) / 8, (uint64_t)sms * CHUNK_MINB);
        c->begin("bqsr_g_chunk_list", (double)n_gen * (48 + 19 + 8 + 225 + 75));
        bqsr_chunk_kernel<true><<<(unsigned)grid_g, 256, smem, c->stream>>>(A, A.gen_list, n_gen);
        c->end(); LAUNCH_CHECK(c);
    }
    return E_OK;
}

// the count kernel's QUAL classifier: an index (q >> sh) & 7 that separates EVERY QUAL value present in the arena, at most four of them >= 6
struct FastPlan { bool ok = false; int S = 0; uint32_t sh = 0, lut_lo = 0, lut_hi = 0; uint8_t slot_q[4] = {0, 0, 0, 0}; };
FastPlan plan_fast(const elp_ctx* c, const uint32_t present[4]) {
    FastPlan P;
    if (const char* e = getenv("ELPREP_B200_GATHER")) if (std::string(e) == "general") return P;
    if (present[3] || (present[2] >> 30)) return P;                       // a value > 93 (or a byte >= 128): the general kernels report it
    std::vector<int> vals;
    for (int q = 0; q < 94; q++) if ((present[q >> 5] >> (q & 31)) & 1u) vals.push_back(q);
    std::vector<int> slots;
    for (int q : vals) if (q >= 6) slots.push_back(q);
    if (slots.empty() || slots.size() > 4 || vals.size() > 8) return P;
    if (c->geom.n_cov < 1 || c->geom.n_cov * 2 > MAX_CLS || c->h_ranges.lseq_max > 1024 || c->h_ranges.lseq_max < 1) return P;
    for (uint32_t sh = 0; sh <= 4; sh++) {
        uint32_t seen = 0; bool good = true;
        for (int q : vals) { const uint32_t ix = ((uint32_t)q >> sh) & 7u; if (seen & (1u << ix)) { good = false; break; } seen |= 1u << ix; }
        if (!good) continue;
        uint8_t lut[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int q : vals) {
            uint8_t b = q > 2 ? 0x80 : 0;
            for (size_t s = 0; s < slots.size(); s++) if (slots[s] == q) b |= (uint8_t)(1u << s);
            lut[((uint32_t)q >> sh) & 7u] = b;
        }
        P.ok = true; P.S = (int)slots.size(); P.sh = sh;
        P.lut_lo = (uint32_t)lut[0] | ((uint32_t)lut[1] << 8) | ((uint32_t)lut[2] << 16) | ((uint32_t)lut[3] << 24);
        P.lut_hi = (uint32_t)lut[4] | ((uint32_t)lut[5] << 8) | ((uint32_t)lut[6] << 16) | ((uint32_t)lut[7] << 24);
        for (size_t s = 0; s < slots.size(); s++) P.slot_q[s] = (uint8_t)slots[s];
        return P;
    }
    return P;
}

template <int S> int launch_count(elp_ctx* c, CountArgs K, bool indel, unsigned grid) {
    // CTA-private mismatch tables when they are small (<= 24 KB); otherwise the global table takes the (sparse) mismatches directly
    const size_t mm = ((size_t)K.n_cls * S * 32 * K.lpr + (size_t)(K.n_cls / 2) * S * 16);
    K.mm_cells = mm * 4 <= 24 * 1024 ? (uint32_t)mm : 0u;
    const size_t smem0 = (size_t)CNT_WARPS * (CNT_STAGES * 7 * 512 + CNT_RECRING * K.rec_bytes) + (size_t)K.mm_cells * 4, smem1 = (size_t)CNT_WARPS * (CNT_STAGES * 9 * 512 + CNT_RECRING * K.rec_bytes) + (size_t)K.mm_cells * 4;
    if (!indel) {
        CUDA_TRY(c, cudaFuncSetAttribute(bqsr_count_kernel<S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0));
        bqsr_count_kernel<S, false><<<grid, CNT_WARPS * 32, smem0, c->stream>>>(K);
    } else {
        CUDA_TRY(c, cudaFuncSetAttribute(bqsr_count_kernel<S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
        bqsr_count_kernel<S, true><<<grid, CNT_WARPS * 32, smem1, c->stream>>>(K);
    }
    return E_OK;
}

}  // namespace

int phase_bqsr_gather(elp_ctx* c) {
    if (!c->sorted) return c->fail(E_STATE, "elp_bqsr_gather called before elp_sort_markdup");
    int rc = upload_side_inputs(c);
    if (rc) return rc;
    const size_t cells = c->geom.cells();
    CUDA_TRY(c, cudaMemsetAsync(c->d_tables, 0, cells * 2 * sizeof(int64_t), c->stream));
    const uint64_t n = c->n;
    c->gather_eligible = 0;
    if (n) {
        GatherArgs A{};
        A.n = n; A.refid = c->s_refid.p; A.pos = c->s_pos.p; A.nref = c->s_nref.p; A.pnext = c->s_pnext.p; A.tlen = c->s_tlen.p; A.rg = c->s_rg.p; A.lseq = c->s_lseq.p;
        A.flag = c->s_flag.p; A.mapq = c->s_mapq.p; A.optf = c->s_optf.p; A.qual_off = c->s_qual_off.p; A.seq_off = c->s_seq_off.p; A.cigar_off = c->s_cigar_off.p; A.ncigar = c->s_ncigar.p;
        A.cigar = c->cigar.p; A.seq = c->seq.p; A.qual = c->qual.p; A.rg_cov = c->d_rg_cov; A.n_rg = c->n_rg; A.contig_len = c->d_contig_len; A.n_contigs = c->n_contigs;
        A.refhot = c->d_refhot_ptrs; A.ref_len = c->d_ref_len; A.sites = c->d_site_ptrs; A.n_sites = c->d_n_sites;
        A.geom = c->geom; A.tables = reinterpret_cast<unsigned long long*>(c->d_tables); A.err = c->d_err;
        uint64_t ref_bytes = 0; for (auto l : c->ref_len) ref_bytes += l;
        // SURVEY.md 8d: N_eligible * (19 + 4 + 4 c + L/2 + L) + genome bytes once; per-read averages of the arenas stand in for c and L
        const double per_read = 23.0 + ((double)c->n_cigar * 4 + (double)(c->n_seq - ARENA_FRONT_PAD) + (double)(c->n_qual - ARENA_FRONT_PAD)) / (double)n;
        uint32_t present[4] = {0, 0, 0, 0};
        CUDA_TRY(c, cudaMemcpyAsync(present, c->d_qpresent, 16, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        const FastPlan F = plan_fast(c, present);
        if (!F.ok) {
            // eligible reads are not counted on this path: the roofline line charges all reads (an upper bound, stated in DESIGN.md)
            c->gather_eligible = n;
            rc = gather_general(c, A, nullptr, 0, (double)n * per_read + (double)ref_bytes);
            if (rc) return rc;
        } else {
            const int n_cls = 2 * c->geom.n_cov;
            const int lpr = std::min(32, std::max(1, (c->h_ranges.lseq_max + 31) / 32)), rpw = 32 / lpr;
            int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
            // small device words: [0,64) class histogram | [64,129) region bases | [136,265) list counters | [272,274) segment counts | [276,278) queue heads
            uint32_t* sm = c->d_bq_small;
            uint32_t *d_hist = sm, *d_region = sm + 64, *d_keycnt = sm + 136, *d_nseg = sm + 272, *d_next = sm + 276;
            CUDA_TRY(c, cudaMemsetAsync(sm, 0, 512 * 4, c->stream));
            const uint64_t seg_cap = n / ((uint64_t)SEG_PASSES * rpw) + 2 * MAX_CLS + 16;
            CUDA_TRY(c, c->bq_recs.reserve(2 * n + 8, c->stream));
            CUDA_TRY(c, c->bq_segs.reserve(2 * seg_cap, c->stream));
            CUDA_TRY(c, c->mate.reserve(n + 4, c->stream));
            c->begin("bqsr_g_class_hist", (double)n * 6);
            class_hist_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)sms * 8), 256, 0, c->stream>>>(n, A.rg, A.flag, A.rg_cov, A.n_rg, n_cls, d_hist);
            class_scan_kernel<<<1, 32, 0, c->stream>>>(n_cls, d_hist, d_region);
            c->end(); LAUNCH_CHECK(c); c->launches++;
            Prep2Args P{};
            P.n_cls = n_cls; P.region_base = d_region; P.key_count = d_keycnt; P.recs = c->bq_recs.p; P.cx_list = c->mate.p; P.lpr = lpr; P.max_cycle = c->max_cycle;
            c->begin("bqsr_g_prep2", (double)n * (4 * 7 + 2 + 1 + 8 + 8 + 4 + 8) + (double)c->n_cigar * 4);
            bqsr_prep2_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(A, P);
            c->end(); LAUNCH_CHECK(c);
            uint4* segs0 = c->bq_segs.p; uint4* segs1 = c->bq_segs.p + seg_cap;
            seg_build_kernel<<<1, 128, 0, c->stream>>>(n_cls, rpw, d_region, d_keycnt, segs0, segs1, d_nseg);
            c->launches++; LAUNCH_CHECK(c);
            CountArgs K{};
            K.qual = c->qual.p; K.seq = c->seq.p; K.refhot = c->d_refhot_ptrs; K.recs = c->bq_recs.p; K.tables = A.tables; K.geom = c->geom;
            K.lpr = lpr; K.rpw = rpw; K.rec_bytes = 32u * (uint32_t)rpw; K.n_cls = n_cls; K.sh = F.sh; K.lut_lo = F.lut_lo; K.lut_hi = F.lut_hi;
            for (int s = 0; s < 4; s++) K.slot_q[s] = F.slot_q[s];
            const unsigned grid = (unsigned)sms * CNT_MINB;
            for (int v = 0; v < 2; v++) {
                K.segs = v ? segs1 : segs0; K.n_seg = d_nseg + v; K.seg_next = d_next + v;
                c->begin(v ? "bqsr_g_count_indel" : "bqsr_g_count", 0);     // bytes are set below, once the list sizes are known
                switch (F.S) {
                    case 1: rc = launch_count<1>(c, K, v != 0, grid); break;
                    case 2: rc = launch_count<2>(c, K, v != 0, grid); break;
                    case 3: rc = launch_count<3>(c, K, v != 0, grid); break;
                    default: rc = launch_count<4>(c, K, v != 0, grid); break;
                }
                c->end();
                if (rc) return rc;
                LAUNCH_CHECK(c);
            }
            std::vector<uint32_t> kc(2 * n_cls + 1);
            CUDA_TRY(c, cudaMemcpyAsync(kc.data(), d_keycnt, kc.size() * 4, cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(c, cudaStreamSynchronize(c->stream));
            uint64_t n_simple = 0, n_indel = 0;
            for (int k = 0; k < 2 * n_cls; k++) (k & 1 ? n_indel : n_simple) += kc[k];
            const uint32_t n_cx = kc[2 * n_cls];
            c->gather_eligible = n_simple + n_indel + n_cx;
            c->set_pending_bytes("bqsr_g_count", (double)n_simple * (per_read + 32) + (double)ref_bytes);
            c->set_pending_bytes("bqsr_g_count_indel", (double)n_indel * (per_read + 32));
            if (n_cx) { rc = gather_general(c, A, c->mate.p, n_cx, 0); if (rc) return rc; }
        }
    }
    c->begin("bqsr_g_derive_q", 0);
    derive_q_kernel<<<c->geom.n_cov * 94, 256, 0, c->stream>>>(c->geom, reinterpret_cast<long long*>(c->d_tables));
    c->end(); LAUNCH_CHECK(c);
    rc = check_device_errors(c);
    if (rc) return rc;
    c->gathered = true; c->finalized = false;
    return E_OK;
}
