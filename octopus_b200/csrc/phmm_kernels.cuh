// Kernels of the B200 pair-HMM engine. See phmm_device.cuh for the DP cores and DESIGN.md for the data layout.
#pragma once

#include "phmm_device.cuh"

namespace phmm {

// ---------------------------------------------------------------------------------------------------------
// Device-resident batch (struct of arrays, all pointers into HBM)
// ---------------------------------------------------------------------------------------------------------
struct DevHaps {
    int n;
    const long long* off;
    const char* seq;
    const char* mask_f; const int8_t* prior_f;
    const char* mask_r; const int8_t* prior_r;
    const int8_t* gap_open; const int8_t* gap_extend;
    const long long* begin;     // may be null
    const ColEntry* tab_f;      // column tables, same indexing as seq
    const ColEntry* tab_r;
    const uint32_t* npre_f;     // per-haplotype prefix counts of 'N'-like columns (flank_replay_may_differ_pre), or null
    const uint32_t* npre_r;
};
struct DevReads {
    int n;
    const long long* off;
    const char* bases;
    const uint8_t* quals;
    const uint8_t* mapq;
    const uint8_t* reverse;
    const long long* begin;
    const uint16_t* rowhalf;    // code | qual << 8 per base, same indexing as bases
    const int2* info;           // per read: .x = length, .y = flags
    // Regions (phmm_populate_regions): a read is scored against the haplotypes of its own region only. The result of pair (h, r) lives
    // at slot pbase[r] + h * pstride[r] of best[] / status[] / out[] (k_read_regions; one region: pbase = r, pstride = R).
    const int* region;          // region of each read
    const long long* pbase;
    const int* pstride;
};
// Templates (phmm_populate_regions_ex): region g owns templates [t0, t0 + nT), its [nH][nT] template values start at tout_off.
struct RegionInfo { int h0, nH, r0, nR; long long out_off; int lhs, rhs, use_flanks, t0; long long tout_off; int nT, pad; };
__device__ __forceinline__ long long pair_slot(const DevReads& rd, const int h, const int r) { return rd.pbase[r] + (long long)h * rd.pstride[r]; }
constexpr int kReadNonACGT  = 1;   // read holds a byte outside ACGT → generic path
constexpr int kReadUnsafe16 = 2;   // sum of qualities too large for a 16-bit lane, or a quality > 127
constexpr int kReadTooLong  = 4;   // longer than the fast path's shared-memory row budget
constexpr int kReadUnsafeFlank32 = 8;   // quality sum too large for the 14-bit score field of the flank-aware kernel (fast path still fine)
constexpr int kReadHasN = 16;           // read holds 'N' (and nothing else outside ACGT): all its DPs run on a 32-bit kernel (5th cap)
constexpr int kReadBadQual = 32;        // a quality above 127 (outside the parity domain, DESIGN.md): generic path

constexpr int kFastMaxReadLen = 1023;   // packed path: length bins of the pairing scheduler
constexpr int kWideMaxReadLen = 28000;  // 32-bit multi-lane path: one read's row entries must fit a block's shared memory

// Which kernel family serves a read (decided per call by k_sched_hist / k_sched_scatter):
//   0 packed  two alignments per lane group in s16x2 lanes (dp_pair / dp_band<Lanes16>), reads paired by length
//   1 wide    one alignment per lane group in 32-bit lanes (dp_band<Lanes32>): use_int_scores, reads whose quality sum could
//             overflow a 16-bit lane, reads longer than the pairing scheduler's bins, reads with 'N' the flank kernel cannot take
//   2 generic one thread per (read, haplotype) pair, int32, any alphabet
struct SchedMode { int packed_ok, wide_ok, force_wide, n_to_wide, wide_max_len; };
__host__ __device__ inline int read_route(const int2 inf, const SchedMode m)
{
    const int f = inf.y, L = inf.x;
    if ((f & (kReadNonACGT | kReadBadQual)) || L < 1) return 2;
    const bool n_wide = (f & kReadHasN) && (m.n_to_wide || (f & kReadUnsafeFlank32));
    if (m.packed_ok && !m.force_wide && !(f & (kReadUnsafe16 | kReadTooLong)) && !n_wide) return 0;
    if (m.wide_ok && L <= m.wide_max_len) return 1;
    return 2;
}

// ---------------------------------------------------------------------------------------------------------
// Preparation kernels
// ---------------------------------------------------------------------------------------------------------

// One thread per haplotype base: the two strand tables. flags[0] |= 1 if a prior / gap penalty is outside [0,127].
__global__ void k_build_tables(const long long n_bases, const char* __restrict__ seq,
                               const char* __restrict__ mask_f, const int8_t* __restrict__ prior_f,
                               const char* __restrict__ mask_r, const int8_t* __restrict__ prior_r,
                               const int8_t* __restrict__ go, const int8_t* __restrict__ ge,
                               ColEntry* __restrict__ tab_f, ColEntry* __restrict__ tab_r, int* __restrict__ flags)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bases) return;
    const int pf = prior_f[i], pr = prior_r[i], o = go[i], e = ge[i];
    if ((pf | pr | o | e) < 0) atomicOr(flags, 1);
    {   // one atomic per warp that saw a base with gap_open < gap_extend: the DP kernels then keep the general deletion update
        const unsigned act = __activemask();
        if (__any_sync(act, o < e) && (int)(threadIdx.x & 31) == __ffs(act) - 1) atomicOr(flags, kFlagOpenBelowExtend);
    }
    tab_f[i] = make_col_entry(seq[i], mask_f[i], pf & 127, o & 127, e & 127);
    tab_r[i] = make_col_entry(seq[i], mask_r[i], pr & 127, o & 127, e & 127);
}

// One warp per (haplotype, strand): inclusive prefix counts of the 'N'-like columns of the strand's table (ncol_class), restarting at
// every haplotype (lengths <= 65535: each half-word count fits).
__global__ void k_ncol_prefix(const int H, const long long* __restrict__ off, const ColEntry* __restrict__ tab_f, const ColEntry* __restrict__ tab_r,
                              uint32_t* __restrict__ pre_f, uint32_t* __restrict__ pre_r)
{
    const int w = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    const int h = w >> 1;
    if (h >= H) return;
    const ColEntry* tab = (w & 1) ? tab_r : tab_f;
    uint32_t* pre = (w & 1) ? pre_r : pre_f;
    const long long end = off[h + 1];
    uint32_t run = 0u;
    const unsigned le = 0xffffffffu >> (31 - lane);
    for (long long i0 = off[h]; i0 < end; i0 += 32) {
        const long long i = i0 + lane;
        const uint32_t cls = i < end ? ncol_class(tab[i].x) : 0u;
        const unsigned b_lo = __ballot_sync(0xffffffffu, (cls & 1u) != 0u), b_hi = __ballot_sync(0xffffffffu, cls != 0u);
        if (i < end) pre[i] = run + (uint32_t)__popc(b_lo & le) + ((uint32_t)__popc(b_hi & le) << 16);
        run += (uint32_t)__popc(b_lo) + ((uint32_t)__popc(b_hi) << 16);
    }
}

// What the host needs to know about a device-resident offset array: ends, longest and shortest item (the shortest as
// kOffsetBig - min so that a zero-initialised struct is the identity of all four atomicMax / store updates).
constexpr long long kOffsetBig = 1LL << 62;
struct OffsetSummary { long long first, last, len_max, inv_len_min; };
__global__ void k_offsets_summary(const long long* __restrict__ off, const int n, OffsetSummary* __restrict__ out)
{
    long long hi = 0, inv_lo = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long len = off[i + 1] - off[i];
        hi = max(hi, len); inv_lo = max(inv_lo, kOffsetBig - len);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o)); inv_lo = max(inv_lo, __shfl_xor_sync(0xffffffffu, inv_lo, o)); }
    if ((threadIdx.x & 31) == 0) { atomicMax(&out->len_max, hi); atomicMax(&out->inv_len_min, inv_lo); }
    if (blockIdx.x == 0 && threadIdx.x == 0) { out->first = off[0]; out->last = off[n]; }
}

// One warp per read: row half-words, length and eligibility flags.
__global__ void k_read_info(const int n_reads, const long long* __restrict__ off, const char* __restrict__ bases,
                            const uint8_t* __restrict__ quals, uint16_t* __restrict__ rowhalf, int2* __restrict__ info)
{
    const int r = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= n_reads) return;
    const long long b = off[r];
    const int L = (int)(off[r + 1] - b);
    int flags = 0, qsum = 0;
    for (int y = lane; y < L; y += 32) {
        const int c = base_code(bases[b + y]);
        const int q = quals[b + y];
        if (c < 0) flags |= kReadNonACGT;
        if (c == 4) flags |= kReadHasN;
        if (q > 127) flags |= kReadBadQual;
        qsum += q;
        rowhalf[b + y] = (uint16_t)((c < 0 ? 0 : c) | (q << 8));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        flags |= __shfl_xor_sync(0xffffffffu, flags, o);
        qsum += __shfl_xor_sync(0xffffffffu, qsum, o);
    }
    if (qsum > kMaxScore16) flags |= kReadUnsafe16;
    if (qsum > kMaxScoreFlank32) flags |= kReadUnsafeFlank32;
    if (L > kFastMaxReadLen) flags |= kReadTooLong;
    if (lane == 0) info[r] = make_int2(L, flags);
}

// Region of every read (binary search over the regions' first-read indices) and where its results go.
__global__ void k_read_regions(const int n_reads, const int n_regions, const RegionInfo* __restrict__ regs,
                               int* __restrict__ region, long long* __restrict__ pbase, int* __restrict__ pstride)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    int lo = 0, hi = n_regions;                 // largest g with regs[g].r0 <= r
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (regs[mid].r0 <= r) lo = mid; else hi = mid; }
    const RegionInfo g = regs[lo];
    region[r] = lo;
    pbase[r] = g.out_off - (long long)g.h0 * g.nR + (r - g.r0);
    pstride[r] = g.nR;
}

// Region of every template (binary search over the regions' first-template indices).
__global__ void k_template_regions(const int n_templates, const int n_regions, const RegionInfo* __restrict__ regs, int* __restrict__ region)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_templates) return;
    int lo = 0, hi = n_regions;                 // largest g with regs[g].t0 <= t (every region owns at least one template)
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (regs[mid].t0 <= t) lo = mid; else hi = mid; }
    region[t] = lo;
}

// Device-resident template offsets: non-decreasing, and the templates of every region cover exactly its reads. flags |= kFlagBadTemplates
// otherwise (checked before the template epilogue reads through the offsets).
__global__ void k_check_templates(const int n_templates, const long long* __restrict__ toff, const int* __restrict__ region,
                                  const RegionInfo* __restrict__ regs, int* __restrict__ flags)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_templates) return;
    const RegionInfo g = regs[region[t]];
    const long long a = toff[t], b = toff[t + 1];
    bool bad = b < a;
    if (t == g.t0 && a != g.r0) bad = true;
    if (t == g.t0 + g.nT - 1 && b != (long long)g.r0 + g.nR) bad = true;
    if (bad) atomicOr(flags, kFlagBadTemplates);
}

// ---------------------------------------------------------------------------------------------------------
// Device-side scheduling of the fast path: bucket the eligible reads by length (counting sort), pair reads of equal
// length, pad every length bucket to a multiple of G pairs (a warp's G pairs share one read length). Replaces a host
// pass over all reads; the host only reads back a handful of totals.
// ---------------------------------------------------------------------------------------------------------
constexpr int kLenBins = kFastMaxReadLen + 1;
struct SchedTotals { int n_pairs, n_generic, lmax_fast, lmax_all, n_eligible, bad; long long cells; int n_with_n, n_wide; };

// misc counters: [0] generic reads, [1] longest read, [2] bad, [3] packed reads holding 'N', [4] wide reads
__global__ void k_sched_hist(const int R, const int2* __restrict__ info, const SchedMode mode, int* __restrict__ hist,
                             int* __restrict__ generic, int* __restrict__ wide, int* __restrict__ misc,
                             const int* __restrict__ region, const RegionInfo* __restrict__ regs, const int band, unsigned long long* __restrict__ cells)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    // banded cells of the read against every haplotype of its region (the GCUPS numerator), one atomic per warp
    unsigned long long mine = r < R ? (unsigned long long)(2LL * (info[r].x + band) * band) * (unsigned long long)regs[region[r]].nH : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(cells, mine);
    if (r >= R) return;
    const int2 inf = info[r];
    if (inf.x < 1) atomicExch(misc + 2, 1);
    atomicMax(misc + 1, inf.x);
    const int route = read_route(inf, mode);
    if (route == 0) { atomicAdd(&hist[inf.x], 1); if (inf.y & kReadHasN) atomicAdd(misc + 3, 1); }
    else if (route == 1) wide[atomicAdd(misc + 4, 1)] = r;
    else generic[atomicAdd(misc + 0, 1)] = r;
}

// one block of kLenBins threads: exclusive scans of the per-length read counts and padded pair counts
__global__ void __launch_bounds__(kLenBins)
k_sched_scan(const int* __restrict__ hist, const int G, int* __restrict__ read_start, int* __restrict__ pair_start,
             int* __restrict__ cursors, const int* __restrict__ misc, const unsigned long long* __restrict__ cells, SchedTotals* __restrict__ tot)
{
    __shared__ int s_reads[kLenBins], s_pairs[kLenBins];
    const int l = threadIdx.x;
    const int c = hist[l];
    const int pairs = ((c + 1) / 2 + G - 1) / G * G;
    s_reads[l] = c; s_pairs[l] = pairs;
    __syncthreads();
    // Hillis-Steele inclusive scans (1024 elements)
    for (int d = 1; d < kLenBins; d <<= 1) {
        const int a = l >= d ? s_reads[l - d] : 0, b = l >= d ? s_pairs[l - d] : 0;
        __syncthreads();
        s_reads[l] += a; s_pairs[l] += b;
        __syncthreads();
    }
    read_start[l] = s_reads[l] - c;
    pair_start[l] = s_pairs[l] - pairs;
    cursors[l] = 0;
    const int ng = misc[0], nw = misc[4];
    int lmax = c ? l : 0;
    for (int o = 16; o > 0; o >>= 1) lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    __shared__ int s_lmax[kLenBins / 32];
    if ((l & 31) == 0) s_lmax[l >> 5] = lmax;
    __syncthreads();
    if (l == 0) {
        int m = 0;
        for (int i = 0; i < kLenBins / 32; ++i) m = max(m, s_lmax[i]);
        tot->n_pairs = s_pairs[kLenBins - 1];
        tot->n_eligible = s_reads[kLenBins - 1];
        tot->n_generic = ng;
        tot->n_wide = nw;
        tot->lmax_fast = max(m, 1);
        tot->lmax_all = max(misc[1], 1);
        tot->bad = misc[2];
        tot->n_with_n = misc[3];
        tot->cells = (long long)*cells;
    }
    if (l == kLenBins - 1) { read_start[kLenBins] = s_reads[l]; pair_start[kLenBins] = s_pairs[l]; }
}

__global__ void k_sched_scatter(const int R, const int2* __restrict__ info, const SchedMode mode, const int* __restrict__ read_start,
                                int* __restrict__ cursors, int* __restrict__ sorted)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int2 inf = info[r];
    if (read_route(inf, mode) == 0) sorted[read_start[inf.x] + atomicAdd(&cursors[inf.x], 1)] = r;
}

// pair slot j → (read, read | -1) or (-1, -1) padding
__global__ void k_sched_pairs(const SchedTotals* __restrict__ tot, const int* __restrict__ read_start, const int* __restrict__ pair_start,
                              const int* __restrict__ sorted, int* __restrict__ pairs)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= tot->n_pairs) return;
    int lo = 0, hi = kLenBins;                   // largest bin l with pair_start[l] <= j
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (pair_start[mid] <= j) lo = mid; else hi = mid; }
    const int local = j - pair_start[lo], first = read_start[lo], cnt = read_start[lo + 1] - first;
    const int a = 2 * local, b = 2 * local + 1;
    pairs[2 * j] = a < cnt ? sorted[first + a] : -1;
    pairs[2 * j + 1] = b < cnt ? sorted[first + b] : -1;
}

// Cooperative fill of one warp's shared row words for the read pair (r0, r1); r1 < 0 → second half padded.
__device__ __forceinline__ void fill_rows(RowEntry* rows, const DevReads& rd, const int r0, const int r1, const int L, const int lane)
{
    const uint16_t* h0 = rd.rowhalf + rd.off[r0];
    const uint16_t* h1 = r1 >= 0 ? rd.rowhalf + rd.off[r1] : nullptr;
    for (int y = lane; y < L; y += 32) rows[y] = make_row_entry(h0[y], h1 ? (uint32_t)h1[y] : 0u);
    if (lane == 0) rows[L] = pad_row_entry();
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------
// Raw kernel boundary (phmm_align_scores): explicit task lists
// ---------------------------------------------------------------------------------------------------------

struct LaneTask {          // one alignment: column-table index of its window start, strand, output slot
    long long tab_index;
    int reverse;
    int out_idx;
};
struct WarpWork {          // one warp: read pair (equal length) and the lane-task ranges of its two halves
    int read0, read1;      // read1 < 0: second half empty
    int first0, n0;        // lane tasks of read0: tasks[first0 .. first0+n0), n0 in 1..32
    int first1, n1;        // n1 in 0..32
    int L, pad;
};

constexpr int kFastWarpsPerBlock = 4;

// lanes that cooperate on one alignment (pair): the band's 2B diagonals in chunks of 32 (phmm_device.cuh, dp_band)
__host__ __device__ constexpr int lanes_per_alignment(const int band) { return band <= 16 ? 1 : band / 16; }
__host__ __device__ constexpr int chunk_of(const int band) { return band <= 8 ? 16 : 32; }

// Two alignments (one per packed half) of the lane group this thread belongs to; all lanes of the warp share L.
template <int BAND, bool OGE>
__device__ __forceinline__ uint32_t packed_dp(const RowEntry* __restrict__ rows, const int L, const ColEntry* t0, const ColEntry* t1,
                                              const uint32_t nucp, const int j, const uint32_t one)
{
    if constexpr (BAND <= 16) return dp_pair<BAND, OGE>(rows, L, t0, t1, nucp, one);
    else {
        const Lanes16::Tab tab {t0, t1};
        return dp_band<Lanes16, 32, lanes_per_alignment(BAND), OGE>(rows, L, tab, nucp, j, one);
    }
}

// warp-uniform: do the tables of this call allow the shorter deletion update (dp_pair, OGE)?
__device__ __forceinline__ bool open_ge_extend(const int* __restrict__ flags) { return (*flags & kFlagOpenBelowExtend) == 0; }

// One warp = one read pair; its 2 x (32 / NL) tasks, NL lanes each. The host cuts a read's tasks into chunks of 32 / NL.
template <int BAND>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32)
k_packed_tasks(const WarpWork* __restrict__ works, const int n_works, const LaneTask* __restrict__ tasks,
               const DevHaps hp, const DevReads rd, const int row_stride, const uint32_t nucp, int* __restrict__ scores,
               const int* __restrict__ flags, const uint32_t one)
{
    extern __shared__ RowEntry smem_rows[];
    constexpr int NL = lanes_per_alignment(BAND);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = lane / NL, j = lane % NL;
    const int w = blockIdx.x * kFastWarpsPerBlock + warp;
    if (w >= n_works) return;
    const WarpWork ww = works[w];
    RowEntry* rows = smem_rows + warp * row_stride;
    fill_rows(rows, rd, ww.read0, ww.read1, ww.L, lane);
    const bool v0 = slot < ww.n0, v1 = slot < ww.n1;
    const LaneTask a = tasks[v0 ? ww.first0 + slot : ww.first0];
    const LaneTask b = v1 ? tasks[ww.first1 + slot] : a;
    const ColEntry* t0 = (a.reverse ? hp.tab_r : hp.tab_f) + a.tab_index;
    const ColEntry* t1 = (b.reverse ? hp.tab_r : hp.tab_f) + b.tab_index;
    const uint32_t r = open_ge_extend(flags) ? packed_dp<BAND, true>(rows, ww.L, t0, t1, nucp, j, one) : packed_dp<BAND, false>(rows, ww.L, t0, t1, nucp, j, one);
    if (j == 0) {
        if (v0) scores[a.out_idx] = (int)(r & 0xFFFFu);
        if (v1) scores[b.out_idx] = (int)(r >> 16);
    }
}

// 32-bit lanes: one warp = one read (WarpWork.read0, tasks first0 .. first0 + n0, n0 <= 32 / NL), NL lanes per task.
template <int C, int NL>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32)
k_wide_tasks(const WarpWork* __restrict__ works, const int n_works, const LaneTask* __restrict__ tasks,
             const DevHaps hp, const DevReads rd, const int row_stride, const int nuc_prior, int* __restrict__ scores,
             const int* __restrict__ flags)
{
    extern __shared__ RowEntry smem_rows[];
    const int warps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = lane / NL, j = lane % NL;
    const int w = blockIdx.x * warps + warp;
    if (w >= n_works) return;
    const WarpWork ww = works[w];
    RowEntry* rows = smem_rows + warp * row_stride;
    const uint16_t* hr = rd.rowhalf + rd.off[ww.read0];
    for (int y = lane; y < ww.L; y += 32) rows[y] = make_row_entry32(hr[y]);
    if (lane == 0) rows[ww.L] = pad_row_entry32();
    __syncwarp();
    const bool v = slot < ww.n0;
    const LaneTask a = tasks[v ? ww.first0 + slot : ww.first0];
    const Lanes32::Tab tab {(a.reverse ? hp.tab_r : hp.tab_f) + a.tab_index};
    const uint32_t r = open_ge_extend(flags) ? dp_band<Lanes32, C, NL, true>(rows, ww.L, tab, (uint32_t)nuc_prior, j)
                                             : dp_band<Lanes32, C, NL, false>(rows, ww.L, tab, (uint32_t)nuc_prior, j);
    if (v && j == 0) scores[a.out_idx] = (int)r;
}

struct GenericTask { int read, hap, win_off, reverse, out_idx; };

template <int MAXK>
__global__ void k_generic_tasks(const GenericTask* __restrict__ tasks, const int n, const DevHaps hp, const DevReads rd,
                                const int band, const int nuc_prior, int* __restrict__ scores)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const GenericTask t = tasks[i];
    const long long ho = hp.off[t.hap] + t.win_off, ro = rd.off[t.read];
    const int L = (int)(rd.off[t.read + 1] - ro);
    const GenericModel gm {hp.seq + ho, (t.reverse ? hp.mask_r : hp.mask_f) + ho, (t.reverse ? hp.prior_r : hp.prior_f) + ho,
                           hp.gap_open + ho, hp.gap_extend + ho, nuc_prior};
    scores[t.out_idx] = generic_align<false, MAXK>(band, gm, rd.bases + ro, (const int8_t*)(rd.quals + ro), L,
                                                   nullptr, 1, 0, 0, nullptr, nullptr, nullptr);
}

// ---------------------------------------------------------------------------------------------------------
// Batch boundary (phmm_populate): fused classify → DP → min, then the floating-point epilogue
// ---------------------------------------------------------------------------------------------------------

struct PopParams {
    DevHaps hp;
    DevReads rd;
    const long long* pos_off;   // CSR over [H][R] pairs, or null
    const int32_t* pos;
    // device k-mer mapper output for the current tile (utils/kmer_mapper.hpp:120-159), or null: list index li (position of the
    // read in the tile's work list) and haplotype h own kpos[(li * H + h) * kMaxMapped .. ), kcnt[li * H + h] entries
    const int32_t* kpos;
    const uint8_t* kcnt;
    // fast-path DP tasks produced by the classify pass for the current tile: list slot li owns
    // ftasks[li * fcap .. li * fcap + fcnt[li]) entries (haplotype | window offset << 16)
    uint32_t* ftasks;
    int* fcnt;
    int fcap;
    // near-flank candidates of fast-path reads, same layout: gtasks for k_populate_flank (crossing cells as payload: any flank
    // geometry, reads with 'N'), atasks for k_populate_flank_acc (the lean form: in-flank penalty as payload; ACGT reads whose
    // window keeps at least two read bases outside the flanks whatever the path)
    uint32_t* gtasks;
    int* gcnt;
    int* flank_cursor;
    uint32_t* atasks;
    int* acnt;
    int* acc_cursor;
    int* any_acc_tasks;
    int fb_route;               // the atasks lists of this tile go to k_flank_fwd / k_flank_bwd (pair list, bands <= 16): any flank geometry, reads of >= 2*band bases
    int* fb_cursor;             // work counter of k_flank_bwd (k_flank_fwd uses acc_cursor)
    int* fb_rounds;             // rounds of forward scratch handed out so far (this tile)
    int* fb_round_base;         // per list slot: first round of the read's forward scratch, -1 = none left
    int fb_round_cap;
    int units_per_pair;         // fast kernel: a read pair's task lists are cut into this many work units of kRoundsPerUnit rounds
    const RegionInfo* regs;     // regions of the call (one for phmm_populate); the flank state is per region
    int Hmax;                   // most haplotypes any region has: per-read loops run over Hmax slots and skip the ones beyond the region
    int band, nuc_prior;
    int one;                    // the constant 1, opaque to the compiler (fma_add)
    int single_candidate;       // every pair has at most one candidate position (no listed / mapped positions): results are stored, not min-reduced
    int reserved_sms;           // the persistent DP kernels leave the SMs with %smid < reserved_sms to others (a collective running beside them)
    int shortcut;               // 1: reference behaviour (try_naive_evaluate first)
    int use_flanks;             // some region has a flank state && config.use_flank_state (the per-region values are in regs)
    int* best;                  // [H*R] integer penalties, kBestInf-initialised
    int* status;                // [H*R] zero-initialised
    int* flags;                 // [0] |= 2 on ShortHaplotypeError, |= 4 on slow-queue overflow
    // near-flank candidates, resolved by k_slow_flank
    int4* slow;                 // {read, hap, position a, unused}
    int* slow_count;
    int slow_cap;
    // The host never waits for the scheduler: it sizes tiles by upper bounds and the kernels clip them against the
    // device-resident totals (tile_pairs / tile_generic below).
    const SchedTotals* tot;
    int pair_base;              // first pair of the current tile
    int* any_flank_tasks;       // set by the classify pass when it queues a task for k_populate_flank
    // fast path work list: read pairs of equal length (second may be -1)
    const int* pair_reads;
    int n_pairs;                // tile size (upper bound)
    int* pair_cursor;           // persistent-warp work counter
    int row_stride;             // shared-memory row entries (8 bytes) per warp
    // The list the current tile's per-read kernels (k-mer mapper, classify pass, 32-bit DP kernels, generic pass) walk:
    // kind 0 = the pair list (two entries per pair, -1 = padding), 1 = wide reads, 2 = generic reads.
    const int* list;
    int list_kind, n_list, list_base;   // n_list: upper bound on the tile's entries; list_base: index of the tile's first entry
};

// flat index → (list slot, haplotype); 64-bit division is an expensive software routine, the index nearly always fits 32 bits
__device__ __forceinline__ void split_index(const long long i, const int H, int* li, int* h)
{
    if (i <= 0xFFFFFFFFll) { const unsigned u = (unsigned)i, q = u / (unsigned)H; *li = (int)q; *h = (int)(u - q * (unsigned)H); }
    else { *li = (int)(i / H); *h = (int)(i % H); }
}

// Persistent DP kernels fill every SM's register file; a collective (NCCL gather of the previous result) launched beside them finds no
// SM to run on until they finish. With reserved_sms > 0 the blocks that land on the first SMs exit at once (the work queue is dynamic:
// the others take it all), which leaves those SMs to the collective at a cost of reserved / 148 of the DP throughput.
__device__ __forceinline__ bool on_reserved_sm(const PopParams& p)
{
    if (p.reserved_sms <= 0) return false;
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    return (int)smid < p.reserved_sms;
}

__device__ __forceinline__ int tile_pairs(const PopParams& p) { return max(0, min(p.n_pairs, p.tot->n_pairs - p.pair_base)); }
__device__ __forceinline__ int list_total(const SchedTotals* tot, const int kind) { return kind == 0 ? 2 * tot->n_pairs : kind == 1 ? tot->n_wide : tot->n_generic; }
__device__ __forceinline__ int tile_list(const PopParams& p) { return max(0, min(p.n_list, list_total(p.tot, p.list_kind) - p.list_base)); }

__device__ __forceinline__ HapView hap_view(const DevHaps& hp, const int h, const bool reverse)
{
    const long long o = hp.off[h];
    return HapView {hp.seq + o, (reverse ? hp.mask_r : hp.mask_f) + o, (reverse ? hp.prior_r : hp.prior_f) + o,
                    hp.gap_open + o, hp.gap_extend + o, (int)(hp.off[h + 1] - o)};
}
__device__ __forceinline__ ReadView read_view(const DevReads& rd, const int r)
{
    const long long o = rd.off[r];
    return ReadView {rd.bases + o, rd.quals + o, (int)(rd.off[r + 1] - o)};
}

// Append one task to list slot li with a warp-aggregated counter update: the lanes of a warp that append to the same list
// (normally all of them: consecutive threads are consecutive haplotypes of one read) share a single atomicAdd.
__device__ __forceinline__ int list_append_slot(int* counts, const int li)
{
    const unsigned active = __activemask();
    const unsigned peers = __match_any_sync(active, li);
    const int leader = __ffs(peers) - 1, lane = threadIdx.x & 31;
    int base = 0;
    if (lane == leader) base = atomicAdd(counts + li, __popc(peers));
    base = __shfl_sync(peers, base, leader);
    return base + __popc(peers & ((1u << lane) - 1u));
}

// as list_append_slot, for lanes that may append to different lists (route) of the same slot
__device__ __forceinline__ int list_append_slot2(int* counts, const int li, const int route)
{
    const unsigned active = __activemask();
    const unsigned peers = __match_any_sync(active, li * 4 + route);
    const int leader = __ffs(peers) - 1, lane = threadIdx.x & 31;
    int base = 0;
    if (lane == leader) base = atomicAdd(counts + li, __popc(peers));
    base = __shfl_sync(peers, base, leader);
    return base + __popc(peers & ((1u << lane) - 1u));
}

__device__ __forceinline__ void push_slow(const PopParams& p, const int r, const int h, const int a)
{
    const int idx = atomicAdd(p.slow_count, 1);
    if (idx < p.slow_cap) p.slow[idx] = make_int4(r, h, a, 0);
    else atomicOr(p.flags, 4);
}

constexpr int kRoundsPerUnit = 8;   // dp_pair rounds per work unit of the fast kernel (bounds the tail imbalance of long task lists)
constexpr int kMaxMapped = 10;    // HaplotypeLikelihoodArray::maxMappingPositions (haplotype_likelihood_array.hpp:104)
constexpr int kKmer = 6;          // mapperKmerSize (:103)
constexpr int kKmerBins = 4096;

// ---------------------------------------------------------------------------------------------------------
// k-mer mapper (utils/kmer_mapper.hpp): K = 6 perfect hash A0 C1 G2 T3 (anything else 0), little-endian base 4 (:24-53)
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned kmer_base(const char b) { return b == 'C' ? 1u : b == 'G' ? 2u : b == 'T' ? 3u : 0u; }
__device__ __forceinline__ unsigned kmer_hash(const char* s)
{
    unsigned h = 0;
#pragma unroll
    for (int i = 0; i < kKmer; ++i) h |= kmer_base(s[i]) << (2 * i);
    return h;
}

// compute_kmer_hashes<6> for every read (:57-69): hash of the 6-mer starting at each base (entries past L-6 unused)
__global__ void k_read_kmers(const long long n_bases, const int n_reads, const long long* __restrict__ off, const char* __restrict__ bases,
                             uint16_t* __restrict__ rhash)
{
    const int r = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= n_reads) return;
    const long long b = off[r];
    const int L = (int)(off[r + 1] - b);
    for (int y = lane; y + kKmer <= L; y += 32) rhash[b + y] = (uint16_t)kmer_hash(bases + b + y);
}

// populate_kmer_hash_table<6> (:85-98) per haplotype, stored HASH-MAJOR: binsT[hash * H + h] = position | 1 << 16 for a bin with one
// k-mer, first item | item count << 16 for a fuller one (0 = empty; positions, item indices and counts are < 2^16: the mapper
// takes haplotypes of up to 65 535 bases), items[hap base offset + ...] = k-mer positions, ascending within a bin.
// One block per haplotype.
__global__ void k_build_kmer_table(const int H, const long long* __restrict__ off, const char* __restrict__ seq,
                                   uint32_t* __restrict__ binsT, uint16_t* __restrict__ items)
{
    __shared__ int hist[kKmerBins + 1];
    __shared__ int cursor[kKmerBins];
    const int h = blockIdx.x;
    if (h >= H) return;
    const long long o = off[h];
    const int nt = (int)(off[h + 1] - o) - kKmer + 1;
    for (int i = threadIdx.x; i <= kKmerBins; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < nt; i += blockDim.x) atomicAdd(&hist[kmer_hash(seq + o + i) + 1], 1);
    __syncthreads();
    // inclusive scan of the shifted counts by one warp (chunks of 32 with a running carry): hist[b] = k-mers with hash < b
    if (threadIdx.x < 32) {
        int run = 0;
        for (int base = 0; base <= kKmerBins; base += 32) {
            const int i = base + threadIdx.x;
            int v = i <= kKmerBins ? hist[i] : 0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int n = __shfl_up_sync(0xffffffffu, v, d); if ((int)threadIdx.x >= d) v += n; }
            if (i <= kKmerBins) hist[i] = v + run;
            run += __shfl_sync(0xffffffffu, v, 31);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kKmerBins; i += blockDim.x) cursor[i] = hist[i];
    __syncthreads();
    // fill in ascending position order within a bin: the vote loop relies on nothing but the set, the order keeps runs reproducible
    for (int i = threadIdx.x; i < nt; i += blockDim.x) {
        const unsigned hh = kmer_hash(seq + o + i);
        const int slot = atomicAdd(&cursor[hh], 1);
        items[o + slot] = (uint16_t)i;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kKmerBins; i += blockDim.x) {
        const int first = hist[i], n = hist[i + 1] - hist[i];
        uint32_t v = 0u;
        if (n == 1) v = (uint32_t)items[o + first] | (1u << 16);
        else if (n > 1) v = (uint32_t)first | ((uint32_t)n << 16);
        binsT[(size_t)i * H + h] = v;
    }
}

// map_query_to_target (:120-159) for every (read of the work list, haplotype): the first <= 10 mapping begins (ascending)
// whose vote count equals the maximum. votes[d] = number of query k-mers qi whose k-mer also starts at target position qi + d.
// One THREAD per pair, consecutive lanes = consecutive haplotypes of one read: the read's k-mer hash is a broadcast load, the
// bin lookup is ONE coalesced line because the bin table is stored hash-major (binsT[hash][haplotype], k_build_kmer_table) and a bin
// with a single k-mer (nearly all of them: ~300 k-mers over 4096 bins) carries the position inline — no second dependent load;
// the per-thread vote array lives in local memory (L1) and is handled a 32-bit word at a time where possible (clear, final scan).
// CountT = uint8_t when no diagonal can collect more than 255 votes (one vote per query k-mer at most: reads of <= 260 bases),
// else uint16_t. Haplotypes with more than MAXT k-mers are handled in tiles of MAXT diagonals, ascending, so the "first ten at the
// maximum" order is kept (round 1 refused them).
// Measured alternatives (profiles/README.md): round 1's haplotype-major bins (two dependent, uncoalesced L2 loads per k-mer) 6.4 ms per C2
// step; a warp per pair with shared-memory vote tiles 13 ms (the per-pair latency chain is paid by every warp instead of being
// spread over 32 pairs).
template <int MAXT, typename CountT>
__global__ void k_kmer_map(const int* __restrict__ list, const int n_list_max, const SchedTotals* __restrict__ tot, const int base, const int kind,
                           const DevHaps hp, const DevReads rd,
                           const uint16_t* __restrict__ rhash, const uint32_t* __restrict__ binsT, const uint16_t* __restrict__ items,
                           int32_t* __restrict__ kpos, uint8_t* __restrict__ kcnt, const RegionInfo* __restrict__ regs, const int Hmax)
{
    constexpr int PER = 4 / (int)sizeof(CountT);
    const int H = hp.n;
    // the tile's work list: 2 entries per read pair, or the wide / generic reads; clipped against the scheduler's totals
    const int n_list = max(0, min(n_list_max, list_total(tot, kind) - base));
    const long long total = (long long)n_list * Hmax, step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        int li, hl;
        split_index(i, Hmax, &li, &hl);
        const int r = list[li];
        uint8_t n_out = 0;
        int h = 0;
        bool in_region = false;
        if (r >= 0) { const RegionInfo g = regs[rd.region[r]]; h = g.h0 + hl; in_region = hl < g.nH; }
        if (in_region) {
            const long long ro = rd.off[r], ho = hp.off[h];
            const int nq = (int)(rd.off[r + 1] - ro) - kKmer + 1, nt = (int)(hp.off[h + 1] - ho) - kKmer + 1;
            if (nq > 0 && nt > 0) {
                uint32_t words[MAXT / PER];
                CountT* counts = reinterpret_cast<CountT*>(words);
                const uint32_t* bs = binsT + h;
                const uint16_t* it = items + ho;
                int32_t* out = kpos + (size_t)i * kMaxMapped;
                unsigned best = 0;
                for (int d0 = 0; d0 < nt; d0 += MAXT) {
                    const int dn = min(MAXT, nt - d0), nwords = (dn + PER - 1) / PER;
                    for (int w = 0; w < nwords; ++w) words[w] = 0u;
                    unsigned max_hit = 0;
                    for (int qi = 0; qi < nq; ++qi) {
                        const uint32_t bin = bs[(size_t)rhash[ro + qi] * H];
                        const int n = (int)(bin >> 16);
                        if (n == 0) continue;
                        if (n == 1) {                                        // the k-mer's position, inline
                            const int d = (int)(bin & 0xFFFFu) - qi - d0;
                            if (d >= 0 && d < dn) { const unsigned c = ++counts[d]; max_hit = c > max_hit ? c : max_hit; }
                            continue;
                        }
                        const int e0 = (int)(bin & 0xFFFFu);
                        for (int e = e0; e < e0 + n; ++e) {
                            const int d = (int)it[e] - qi - d0;               // the reference keeps target_index >= query_index
                            if (d >= 0 && d < dn) { const unsigned c = ++counts[d]; max_hit = c > max_hit ? c : max_hit; }
                        }
                    }
                    if (max_hit > best) { best = max_hit; n_out = 0; }       // a higher count: what earlier tiles listed is void
                    if (max_hit == best && best > 0) {
                        for (int w = 0; w < nwords && n_out < kMaxMapped; ++w) {
                            uint32_t v = words[w];
                            if (v == 0u) continue;
#pragma unroll
                            for (int b = 0; b < PER; ++b) {
                                const unsigned c = v & ((1u << (8 * sizeof(CountT))) - 1u);
                                v >>= 4 * sizeof(CountT); v >>= 4 * sizeof(CountT);
                                const int t = w * PER + b;
                                if (c == best && t < dn && n_out < kMaxMapped) out[n_out++] = d0 + t;
                            }
                        }
                    }
                }
            }
        }
        kcnt[i] = n_out;
    }
}

// Fast-path DP over the task lists the classify pass (k_populate_generic<.., true>) produced. Persistent warps: each warp
// repeatedly claims G consecutive read pairs of equal length (G = 1, 2 or 4 lane groups; G > 1 keeps the lanes busy when a
// read has fewer than 32 tasks, i.e. few haplotypes), stages each pair's row entries in shared memory once, and runs
// dp_pair over the pairs' task lists (32/G + 32/G tasks per group and round, two alignments per lane), folding the
// scores into best[] with atomicMin. Nothing but the DP lives in this kernel: the register-resident band gets the whole
// register budget. The host pads the pair list so that the G pairs of a warp share one read length ((-1,-1) = idle group).
// Resident blocks per SM the register allocation of the packed kernels is held to: 4 (128 registers). Measured alternatives
// (profiles/r02m_*): band 16 at 5 blocks / 96 registers keeps its steady-state loop spill-free (310 instructions per column against 308)
// and is still 9 % SLOWER on C3 (4 772 vs 5 244 GCUPS); 6 blocks / 80 registers spill 22 local accesses per column (-38 %); band 8 at
// 6 blocks -14 %; bands >= 32 at 5 blocks spill heavily (-39 % on C4). More warps do not help an ALU-pipe-bound loop, and the tighter
// allocation costs register-bank conflicts. The macros stay as a measurement hook (tools/gpu_r02_m.sh builds the variants).
#ifndef PHMM_FAST_MIN_BLOCKS_16
#define PHMM_FAST_MIN_BLOCKS_16 4
#endif
#ifndef PHMM_FAST_MIN_BLOCKS_8
#define PHMM_FAST_MIN_BLOCKS_8 4
#endif
#ifndef PHMM_FAST_MIN_BLOCKS_32
#define PHMM_FAST_MIN_BLOCKS_32 4
#endif
__host__ __device__ constexpr int fast_min_blocks(const int band) { return band <= 8 ? PHMM_FAST_MIN_BLOCKS_8 : band == 16 ? PHMM_FAST_MIN_BLOCKS_16 : PHMM_FAST_MIN_BLOCKS_32; }

template <int BAND, int G>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32, fast_min_blocks(BAND))
k_populate_fast(const PopParams p)
{
    extern __shared__ RowEntry smem_rows[];
    constexpr int NL = lanes_per_alignment(BAND);       // lanes per task (pair of alignments): bands >= 32 split their diagonals
    constexpr int LG = 32 / G;                          // lanes per group
    constexpr int TPR = LG / NL;                        // tasks per group and round (per packed half)
    static_assert(TPR >= 1, "a lane group must hold at least one task");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = lane / LG, gl = lane % LG;
    const int slot = gl / NL, jl = gl % NL;
    if (on_reserved_sm(p)) return;
    RowEntry* rows = smem_rows + (warp * G + grp) * p.row_stride;
    const uint32_t nucp = (uint32_t)p.nuc_prior | ((uint32_t)p.nuc_prior << 16);
    const int n_pairs = tile_pairs(p);
    const bool oge = open_ge_extend(p.flags);
    for (;;) {
        int u = 0;
        if (lane == 0) u = atomicAdd(p.pair_cursor, 1);
        u = __shfl_sync(0xffffffffu, u, 0);
        const int jb = (u / p.units_per_pair) * G, part = u % p.units_per_pair;
        if (jb >= n_pairs) break;
        const int j = jb + grp;
        const int r0 = j < n_pairs ? p.pair_reads[2 * j] : -1;
        const int r1 = r0 >= 0 ? p.pair_reads[2 * j + 1] : -1;
        const int n0 = r0 >= 0 ? p.fcnt[2 * j] : 0, n1 = r1 >= 0 ? p.fcnt[2 * j + 1] : 0;
        int nmax = max(n0, n1), L = r0 >= 0 ? p.rd.info[r0].x : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o)); L = max(L, __shfl_xor_sync(0xffffffffu, L, o)); }
        const int c_begin = part * kRoundsPerUnit * TPR, c_end = min(nmax, c_begin + kRoundsPerUnit * TPR);
        if (c_begin >= nmax) continue;
        __syncwarp();
        if (r0 >= 0) {   // cooperative fill by the group's lanes
            const uint16_t* h0 = p.rd.rowhalf + p.rd.off[r0];
            const uint16_t* h1 = r1 >= 0 ? p.rd.rowhalf + p.rd.off[r1] : nullptr;
            for (int y = gl; y < L; y += LG) rows[y] = make_row_entry(h0[y], h1 ? (uint32_t)h1[y] : 0u);
            if (gl == 0) rows[L] = pad_row_entry();
        }
        __syncwarp();
        const int rb = r1 >= 0 ? r1 : r0;
        const ColEntry* tab0 = (r0 >= 0 && p.rd.reverse[r0]) ? p.hp.tab_r : p.hp.tab_f;
        const ColEntry* tab1 = (rb >= 0 && p.rd.reverse[rb]) ? p.hp.tab_r : p.hp.tab_f;
        const uint32_t* q0 = p.ftasks + (size_t)(2 * (size_t)max(j, 0)) * p.fcap;
        const uint32_t* q1 = q0 + p.fcap;
        for (int c = c_begin; c < c_end; c += TPR) {
            const bool v0 = c + slot < n0, v1 = c + slot < n1;
            // idle half-lanes replay a valid task (result discarded): of their own group if it has one, else of any lane
            const bool have = (n0 > 0) || (n1 > 0);
            uint32_t t0 = 0, t1 = 0;
            const ColEntry *b0 = tab0, *b1 = tab1;
            if (have) {
                t0 = n0 > 0 ? q0[v0 ? c + slot : 0] : q1[0];
                t1 = n1 > 0 ? q1[v1 ? c + slot : 0] : t0;
                if (n0 == 0) b0 = tab1;
                if (n1 == 0) b1 = tab0;
            }
            const unsigned anyone = __ballot_sync(0xffffffffu, have);
            const int src = __ffs(anyone) - 1;
            const uint32_t s0 = __shfl_sync(0xffffffffu, t0, src), s1 = __shfl_sync(0xffffffffu, t1, src);
            const unsigned long long sb0 = __shfl_sync(0xffffffffu, (unsigned long long)b0, src), sb1 = __shfl_sync(0xffffffffu, (unsigned long long)b1, src);
            if (!have) { t0 = s0; t1 = s1; b0 = (const ColEntry*)sb0; b1 = (const ColEntry*)sb1; }
            const int h0 = (int)(t0 & 0xFFFFu), a0 = (int)(t0 >> 16), h1 = (int)(t1 & 0xFFFFu), a1 = (int)(t1 >> 16);
            const ColEntry *c0 = b0 + p.hp.off[h0] + a0, *c1 = b1 + p.hp.off[h1] + a1;
            const uint32_t res = oge ? packed_dp<BAND, true>(rows, L, c0, c1, nucp, jl, (uint32_t)p.one) : packed_dp<BAND, false>(rows, L, c0, c1, nucp, jl, (uint32_t)p.one);
            if (jl == 0) {
                // at most one candidate per pair (single_candidate): its value IS the pair's minimum — a plain store, no read of best[]
                if (v0) { int* dst = p.best + pair_slot(p.rd, h0, r0); const int v = (int)(res & 0xFFFFu); if (p.single_candidate) *dst = v; else atomicMin(dst, v); }
                if (v1) { int* dst = p.best + pair_slot(p.rd, h1, r1); const int v = (int)(res >> 16); if (p.single_candidate) *dst = v; else atomicMin(dst, v); }
            }
        }
    }
}

// The packed DP of bands 32 and 64 with one WARP per chunk of 32 diagonals (dp_band_roles): a group of NL = B / 16 warps owns a read
// pair; lane l of every warp of the group works on the group's task l of the round (32 + 32 tasks per round), warp j on chunk j.
// Same work list, task words and result stores as k_populate_fast<B, 1>; used when a read has enough tasks to fill 32 lanes (H >= 17).
__host__ __device__ constexpr int kRoleWordsPerGroup(const int nl) { return 3 * nl * 32 + 32; }
template <int BAND>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32, PHMM_FAST_MIN_BLOCKS_32)
k_populate_roles(const PopParams p)
{
    extern __shared__ RowEntry smem_rows[];
    constexpr int NL = lanes_per_alignment(BAND);
    static_assert(NL == 2 || NL == 4, "role warps: bands 32 and 64");
    constexpr int NG = kFastWarpsPerBlock / NL;         // groups per block
    constexpr int GT = NL * 32;                         // threads per group
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = warp / NL, role = warp % NL, gt = role * 32 + lane;
    if (on_reserved_sm(p)) return;
    RowEntry* rows = smem_rows + grp * p.row_stride;
    uint32_t* xchg = reinterpret_cast<uint32_t*>(smem_rows + NG * p.row_stride) + grp * kRoleWordsPerGroup(NL);
    volatile int* claim = reinterpret_cast<volatile int*>(xchg + 3 * NL * 32);
    const int bar = 1 + grp;
    const uint32_t nucp = (uint32_t)p.nuc_prior | ((uint32_t)p.nuc_prior << 16);
    const int n_pairs = tile_pairs(p);
    const bool oge = open_ge_extend(p.flags);
    for (;;) {
        if (gt == 0) *claim = atomicAdd(p.pair_cursor, 1);
        group_barrier(bar, GT);
        const int u = *claim;
        const int j = u / p.units_per_pair, part = u % p.units_per_pair;
        if (j >= n_pairs) break;
        const int r0 = p.pair_reads[2 * j];
        const int r1 = r0 >= 0 ? p.pair_reads[2 * j + 1] : -1;
        const int n0 = r0 >= 0 ? p.fcnt[2 * j] : 0, n1 = r1 >= 0 ? p.fcnt[2 * j + 1] : 0;
        const int nmax = max(n0, n1), L = r0 >= 0 ? p.rd.info[r0].x : 0;
        const int c_begin = part * kRoundsPerUnit * 32, c_end = min(nmax, c_begin + kRoundsPerUnit * 32);
        if (c_begin < nmax) {
            const uint16_t* h0 = p.rd.rowhalf + p.rd.off[r0];
            const uint16_t* h1 = r1 >= 0 ? p.rd.rowhalf + p.rd.off[r1] : nullptr;
            for (int y = gt; y < L; y += GT) rows[y] = make_row_entry(h0[y], h1 ? (uint32_t)h1[y] : 0u);
            if (gt == 0) rows[L] = pad_row_entry();
            group_barrier(bar, GT);
            const int rb = r1 >= 0 ? r1 : r0;
            const ColEntry* tab0 = p.rd.reverse[r0] ? p.hp.tab_r : p.hp.tab_f;
            const ColEntry* tab1 = p.rd.reverse[rb] ? p.hp.tab_r : p.hp.tab_f;
            const uint32_t* q0 = p.ftasks + (size_t)(2 * (size_t)j) * p.fcap;
            const uint32_t* q1 = q0 + p.fcap;
            for (int c = c_begin; c < c_end; c += 32) {
                const bool v0 = c + lane < n0, v1 = c + lane < n1;
                // idle half-lanes replay a valid task (result discarded); nmax > c_begin, so at least one of the lists is not empty
                const uint32_t t0 = n0 > 0 ? q0[v0 ? c + lane : 0] : q1[0];
                const uint32_t t1 = n1 > 0 ? q1[v1 ? c + lane : 0] : t0;
                const ColEntry* b0 = n0 > 0 ? tab0 : tab1;
                const ColEntry* b1 = n1 > 0 ? tab1 : b0;
                const int h0i = (int)(t0 & 0xFFFFu), a0 = (int)(t0 >> 16), h1i = (int)(t1 & 0xFFFFu), a1 = (int)(t1 >> 16);
                const Lanes16::Tab tab {b0 + p.hp.off[h0i] + a0, b1 + p.hp.off[h1i] + a1};
                const uint32_t res = oge ? dp_band_roles<Lanes16, 32, NL, true>(rows, L, tab, nucp, role, lane, (uint32_t)p.one, xchg, bar)
                                         : dp_band_roles<Lanes16, 32, NL, false>(rows, L, tab, nucp, role, lane, (uint32_t)p.one, xchg, bar);
                if (role == 0) {
                    if (v0) { int* dst = p.best + pair_slot(p.rd, h0i, r0); const int v = (int)(res & 0xFFFFu); if (p.single_candidate) *dst = v; else atomicMin(dst, v); }
                    if (v1) { int* dst = p.best + pair_slot(p.rd, h1i, r1); const int v = (int)(res >> 16); if (p.single_candidate) *dst = v; else atomicMin(dst, v); }
                }
            }
        }
        group_barrier(bar, GT);        // the rows and the claim word are free again
    }
}

// Work claim of the per-read flank kernels: a warp is cut into G = 32 >> lg lane groups of 1 << lg lanes and claims G consecutive list
// slots; a group owns one read (its row entries in its own shared-memory region). Every lane learns its group's slot, read, task count
// (counts[slot]) and read length, and the warp's round count (a lane takes `per_lane` tasks per round). rounds < 0: the list is exhausted.
struct FbClaim { int li, r, n, L, rounds, base; };
__device__ __forceinline__ FbClaim fb_claim(const PopParams& p, int* cursor, const int* __restrict__ counts, const int n_list, const int lane, const int lg,
                                            const int per_lane)
{
    const int G = 32 >> lg;
    int li0 = 0;
    if (lane == 0) li0 = atomicAdd(cursor, G);
    li0 = __shfl_sync(0xffffffffu, li0, 0);
    FbClaim c;
    c.li = li0 + (lane >> lg);
    if (li0 >= n_list) { c.li = -1; c.r = -1; c.n = 0; c.L = 0; c.rounds = -1; c.base = -1; return c; }
    c.r = c.li < n_list ? p.list[c.li] : -1;
    c.n = c.r >= 0 ? counts[c.li] : 0;
    c.L = c.n > 0 ? p.rd.info[c.r].x : 0;
    const int per_round = per_lane << lg;
    int rounds = (c.n + per_round - 1) / per_round;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rounds = max(rounds, __shfl_xor_sync(0xffffffffu, rounds, o));
    c.rounds = rounds; c.base = -1;
    return c;
}

// Near-flank candidates the packed flank kernels do not take (reads with 'N', reads shorter than 2 * band, candidates they report
// as tied; band 32: every candidate that is not lean): the payload-carrying 32-bit DP (dp_flank32), one alignment per lane, persistent
// warps over the tile's work list. A lane group owns a read (row entries broadcast from its shared-memory region): whole warps
// (lg = 5) when the lists are dense, groups of 4 lanes when they hold the packed kernels' ties — one or two per read, which a warp per
// read served with one or two of its 32 lanes (9 % of a flank-state step for 1 % of its candidates, profiles/r02r_launches_C2_flank.csv).
template <int BAND>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32)
k_populate_flank(const PopParams p, const int row_stride, const int lg)
{
    extern __shared__ RowEntry smem_rows[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int LG = 1 << lg, gl = lane & (LG - 1);
    RowEntry* rows = smem_rows + (size_t)(warp * (32 >> lg) + (lane >> lg)) * row_stride;
    constexpr int K = 2 * BAND;
    if (*p.any_flank_tasks == 0) return;          // nothing was queued for this kernel
    const int n_list = tile_list(p);
    for (;;) {
        const FbClaim cl = fb_claim(p, p.flank_cursor, p.gcnt, n_list, lane, lg, 1);
        if (cl.rounds < 0) break;
        if (cl.rounds == 0) continue;
        const int r = cl.r, n = cl.n, L = cl.L;
        __syncwarp();
        unsigned qmin = 255u;
        if (n > 0) {
            const uint16_t* hr = p.rd.rowhalf + p.rd.off[r];
            for (int y = gl; y < L; y += LG) { const uint16_t half = hr[y]; rows[y] = make_row_entry32(half); qmin = min(qmin, (unsigned)half >> 8); }
            if (gl == 0) rows[L] = pad_row_entry32();
        }
        __syncwarp();
        for (int o = LG >> 1; o > 0; o >>= 1) qmin = min(qmin, __shfl_xor_sync(0xffffffffu, qmin, o));
        if (n == 0) continue;       // (no warp-level operation below)
        const bool low_quality = qmin < 2u;                 // see flank_replay_may_differ
        const RegionInfo reg = p.regs[p.rd.region[r]];
        const ColEntry* tab = p.rd.reverse[r] ? p.hp.tab_r : p.hp.tab_f;
        const uint32_t* q = p.gtasks + (size_t)cl.li * p.fcap;
        const int W = L + K - 1;
        for (int c = 0; c < cl.rounds; ++c) {
            const int i = (c << lg) + gl;
            if (i >= n) continue;
            const uint32_t t = q[i];
            const int h = (int)(t & 0xFFFFu), a = (int)(t >> 16);
            const int hap_len = (int)(p.hp.off[h + 1] - p.hp.off[h]);
            int lhs, rhs;
            window_flanks(a, W, hap_len, reg.lhs, reg.rhs, &lhs, &rhs);
            int xl = lhs, xr = W - rhs;
            const bool all_flank = xr <= xl;        // flanks overlap: every operation is inside a flank
            if (all_flank) { xl = 0; xr = W + 1; }
            if (xr >= W) xr = W + 1;
            int score, flank, mask;
            dp_flank32<BAND>(rows, L, tab + p.hp.off[h] + a, p.nuc_prior, xl, xr, &score, &flank, &mask);
            if (all_flank) { flank = score; mask = L; }
            const int v = discount_flank(score, flank, L, mask, 0);
            // an in-flank 'N' column the DP may have charged less than the reference's replay does: exact traceback path instead
            const bool replay_differs = reg.use_flanks != 0 && flank_replay_may_differ(tab + p.hp.off[h] + a, W, lhs, rhs, low_quality);
            if (replay_differs) push_slow(p, r, h, a);
            else atomicMin(p.best + pair_slot(p.rd, h, r), v);
        }
    }
}

// The lean flank-aware kernel (dp_flank_acc): same shape as k_populate_flank, over the atasks lists.
template <int BAND>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32, BAND <= 16 ? 4 : 1)
k_populate_flank_acc(const PopParams p)
{
    extern __shared__ RowEntry smem_rows[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    RowEntry* rows = smem_rows + warp * p.row_stride;
    constexpr int K = 2 * BAND;
    if (*p.any_acc_tasks == 0 || on_reserved_sm(p)) return;
    const int n_list = tile_list(p);
    for (;;) {
        int li = 0;
        if (lane == 0) li = atomicAdd(p.acc_cursor, 1);
        li = __shfl_sync(0xffffffffu, li, 0);
        if (li >= n_list) break;
        const int r = p.list[li];
        const int n = r >= 0 ? p.acnt[li] : 0;
        if (n == 0) continue;
        const int L = p.rd.info[r].x;
        const RegionInfo reg = p.regs[p.rd.region[r]];
        __syncwarp();
        unsigned qmin = 255u;
        {
            const uint16_t* hr = p.rd.rowhalf + p.rd.off[r];
            for (int y = lane; y < L; y += 32) { const uint16_t half = hr[y]; rows[y] = make_row_entry_facc(half); qmin = min(qmin, (unsigned)half >> 8); }
            if (lane == 0) rows[L] = pad_row_entry_facc();
            __syncwarp();
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) qmin = min(qmin, __shfl_xor_sync(0xffffffffu, qmin, o));
        const bool low_quality = qmin < 2u;                 // see flank_replay_may_differ
        const ColEntry* tab = p.rd.reverse[r] ? p.hp.tab_r : p.hp.tab_f;
        const uint32_t* q = p.atasks + (size_t)li * p.fcap;
        const int W = L + K - 1;
        for (int c = 0; c < n; c += 32) {
            const bool valid = c + lane < n;
            const uint32_t t = q[valid ? c + lane : 0];
            const int h = (int)(t & 0xFFFFu), a = (int)(t >> 16);
            const int hap_len = (int)(p.hp.off[h + 1] - p.hp.off[h]);
            int lhs, rhs;
            window_flanks(a, W, hap_len, reg.lhs, reg.rhs, &lhs, &rhs);
            const int xl = lhs, xr = (W - rhs >= W) ? W + 1 : W - rhs;
            int score, flank;
            dp_flank_acc<BAND>(rows, L, tab + p.hp.off[h] + a, p.nuc_prior, xl, xr, &score, &flank, (uint32_t)p.one);
            // an in-flank 'N' column the DP may have charged less than the reference's replay does: exact traceback path instead
            const bool replay_differs = flank_replay_may_differ(tab + p.hp.off[h] + a, W, lhs, rhs, low_quality);
            if (valid) {
                if (replay_differs) push_slow(p, r, h, a);
                else atomicMin(p.best + pair_slot(p.rd, h, r), score - flank);
            }
        }
    }
}

constexpr int kFlankFbMaxBand = 16;     // widest band served by k_flank_fwd / k_flank_bwd: their register band holds 2 * band diagonals (band 32 spills: it keeps the lean labelled kernel)
// words of one round's forward arrays: 64 candidates = 32 lanes x (4 boundary slots x {M, D} x 2B diagonals), lane-interleaved
__host__ __device__ constexpr size_t fb_round_words(const int band) { return (size_t)kFbSlots * 2 * 2 * (size_t)band * 32; }

// The packed forward / backward flank kernels (dp_flank_fwd / dp_flank_bwd). Both packed halves carry the SAME read, so a lane works
// on TWO of a read's near-flank candidates (two haplotype windows) at once. A warp is cut into G = 32 >> lg lane groups of LG = 1 << lg
// lanes; a group owns one read (list slot) at a time — its row entries in its own shared-memory region — and handles 2 * LG of the
// read's candidates per round: the host picks lg from the haplotype count so that regions with few haplotypes still fill the lanes
// (the fast kernel's G, for the same reason). Two launches over the same atasks lists with the same (list slot, round, lane, half)
// → candidate mapping:
//   k_flank_fwd  forward pass up to the last flank boundary of the lane's two windows; the band's arrivals at the boundary columns go
//                to `pair_scratch` (fb_round_words(BAND) words per warp-round, handed out by an atomic counter; reads that find no
//                room are marked and k_flank_bwd sends their candidates to the labelled DP);
//   k_flank_bwd  backward pass from the window end down to the first boundary, crossing cells from F + B (fb_finish), flank discount,
//                minimum into best[]. A candidate whose co-optimal paths cross a boundary at different cells (FbResult::tie, ~1 %) is
//                appended to the read's gtasks list: k_populate_flank, launched after these two, resolves it with the labelled DP.
// (One fused kernel measured 0.9 x the labelled kernel: its code overflows the instruction cache, profiles/r02n.)
template <int BAND>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32, 4)
k_flank_fwd(const PopParams p, uint32_t* __restrict__ pair_scratch, const int row_stride, const int lg)
{
    extern __shared__ RowEntry smem_rows[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int LG = 1 << lg, gl = lane & (LG - 1);
    RowEntry* rows = smem_rows + (size_t)(warp * (32 >> lg) + (lane >> lg)) * row_stride;
    constexpr int K = 2 * BAND;
    if (*p.any_acc_tasks == 0 || on_reserved_sm(p)) return;
    const int n_list = tile_list(p);
    const uint32_t nucp = (uint32_t)p.nuc_prior | ((uint32_t)p.nuc_prior << 16);
    const bool oge = open_ge_extend(p.flags);
    for (;;) {
        FbClaim cl = fb_claim(p, p.acc_cursor, p.acnt, n_list, lane, lg, 2);
        if (cl.rounds < 0) break;
        if (cl.rounds == 0) continue;
        if (lane == 0) {
            cl.base = atomicAdd(p.fb_rounds, cl.rounds);
            if (cl.base + cl.rounds > p.fb_round_cap) cl.base = -1;
        }
        cl.base = __shfl_sync(0xffffffffu, cl.base, 0);
        if (gl == 0 && cl.li < n_list) p.fb_round_base[cl.li] = cl.base;
        if (cl.base < 0) continue;                            // no scratch left: k_flank_bwd hands these reads' candidates to the labelled DP
        const int L = cl.L, n = cl.n, r = cl.r;
        __syncwarp();
        if (n > 0) {
            const uint16_t* hr = p.rd.rowhalf + p.rd.off[r];
            for (int y = gl; y < L; y += LG) { const uint32_t half = hr[y]; rows[y] = make_row_entry(half, half); }
            if (gl == 0) rows[L] = pad_row_entry();
        }
        __syncwarp();
        if (n == 0) continue;       // (no warp-level operation below: a group without candidates just waits for the next claim)
        const RegionInfo reg = p.regs[p.rd.region[r]];
        const ColEntry* tab = p.rd.reverse[r] ? p.hp.tab_r : p.hp.tab_f;
        const uint32_t* q = p.atasks + (size_t)cl.li * p.fcap;
        const int W = L + K - 1;
        for (int c = 0; c < cl.rounds; ++c) {
            const int i0 = (c << (lg + 1)) + 2 * gl, i1 = i0 + 1;
            if (i0 >= n) continue;
            const uint32_t w0 = q[i0], w1 = i1 < n ? q[i1] : w0;             // an odd last candidate is replayed in the idle half (result discarded)
            const int h0 = (int)(w0 & 0xFFFFu), a0 = (int)(w0 >> 16), h1 = (int)(w1 & 0xFFFFu), a1 = (int)(w1 >> 16);
            int lhs0, rhs0, lhs1, rhs1;
            window_flanks(a0, W, (int)(p.hp.off[h0 + 1] - p.hp.off[h0]), reg.lhs, reg.rhs, &lhs0, &rhs0);
            window_flanks(a1, W, (int)(p.hp.off[h1 + 1] - p.hp.off[h1]), reg.lhs, reg.rhs, &lhs1, &rhs1);
            const FbBounds g = fb_bounds(lhs0, W - rhs0, lhs1, W - rhs1, W);
            const ColEntry *c0 = tab + p.hp.off[h0] + a0, *c1 = tab + p.hp.off[h1] + a1;
            const auto fscr = [&]() { return pair_scratch + (size_t)(cl.base + c) * fb_round_words(BAND) + (threadIdx.x & 31); };
            if (oge) dp_flank_fwd<BAND, true>(rows, L, c0, c1, nucp, g, fscr, 32, (uint32_t)p.one);
            else dp_flank_fwd<BAND, false>(rows, L, c0, c1, nucp, g, fscr, 32, (uint32_t)p.one);
        }
    }
}

template <int BAND>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32, 4)
k_flank_bwd(const PopParams p, const uint32_t* pair_scratch, uint32_t* __restrict__ thread_scratch, const int row_stride, const int lg)
{
    extern __shared__ RowEntry smem_rows[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int LG = 1 << lg, gl = lane & (LG - 1);
    RowEntry* rows = smem_rows + (size_t)(warp * (32 >> lg) + (lane >> lg)) * row_stride;
    constexpr int K = 2 * BAND;
    if (*p.any_acc_tasks == 0 || on_reserved_sm(p)) return;
    const int n_list = tile_list(p);
    // the backward arrays of this thread: lane-interleaved within the warp's own region (constant stride: immediate store offsets)
    constexpr size_t bstride = 32;
    const auto bscr_fn = [&]() { return thread_scratch + (size_t)(blockIdx.x * kFastWarpsPerBlock + (threadIdx.x >> 5)) * fb_scratch_words(BAND) * 32 + (threadIdx.x & 31); };
    const uint32_t nucp = (uint32_t)p.nuc_prior | ((uint32_t)p.nuc_prior << 16);
    for (;;) {
        FbClaim cl = fb_claim(p, p.fb_cursor, p.acnt, n_list, lane, lg, 2);
        if (cl.rounds < 0) break;
        if (cl.rounds == 0) continue;
        const int L = cl.L, n = cl.n, r = cl.r;
        const uint32_t* q = p.atasks + (size_t)max(cl.li, 0) * p.fcap;
        int base = cl.li < n_list ? p.fb_round_base[cl.li] : 0;
        base = __shfl_sync(0xffffffffu, base, 0);             // one value per claim (lane 0's slot always exists)
        if (base < 0) {                                       // the forward kernel found no scratch for this claim: labelled DP for all its candidates
            for (int i = gl; i < n; i += LG) {
                const int slot = atomicAdd(p.gcnt + cl.li, 1);
                if (slot < p.fcap) p.gtasks[(size_t)cl.li * p.fcap + slot] = q[i];
                else atomicOr(p.flags, 8);
            }
            if (n > 0) *p.any_flank_tasks = 1;
            continue;
        }
        __syncwarp();
        unsigned qmin = 255u;
        if (n > 0) {
            const uint16_t* hr = p.rd.rowhalf + p.rd.off[r];
            for (int y = gl; y < L; y += LG) { const uint32_t half = hr[y]; rows[y] = make_row_entry(half, half); qmin = min(qmin, half >> 8); }
            for (int y = L + gl; y < L + K; y += LG) rows[y] = pad_row_entry();     // the backward pass reads pad rows down to L + 2B - 1
        }
        __syncwarp();
        for (int o = LG >> 1; o > 0; o >>= 1) qmin = min(qmin, __shfl_xor_sync(0xffffffffu, qmin, o));
        if (n == 0) continue;       // (no warp-level operation below)
        const bool low_quality = qmin < 2u;                 // see flank_replay_may_differ
        for (int c = 0; c < cl.rounds; ++c) {
            // Register discipline: the band takes 64 of the 128 registers and ptxas issues a cell's row-entry load ahead of its use only if it
            // finds ~8 spare ones (LDS-to-use distance 2 instructions and short_scoreboard 1.6 stalls per issue without them, profiles/r02q —
            // the forward kernel, with nothing to do after its DP, loads three cells ahead). So nothing but the list slot, the read, its two
            // sizes and the two task words lives across the DP: each side of it derives what it needs from OPAQUE copies of those.
            int li_o = cl.li, r_o = r, n_o = n, L_o = L;
            asm volatile("" : "+r"(li_o), "+r"(r_o), "+r"(n_o), "+r"(L_o));
            const int i0 = (c << (lg + 1)) + 2 * gl, i1 = i0 + 1;
            if (i0 >= n_o) continue;
            uint32_t x0, x1;
            {
                const uint32_t* q = p.atasks + (size_t)li_o * p.fcap;
                const uint32_t w0 = q[i0], w1 = i1 < n_o ? q[i1] : w0;           // the forward kernel's mapping, exactly
                const RegionInfo reg = p.regs[p.rd.region[r_o]];
                const ColEntry* tab = p.rd.reverse[r_o] ? p.hp.tab_r : p.hp.tab_f;
                const int W = L_o + K - 1;
                const int h0 = (int)(w0 & 0xFFFFu), a0 = (int)(w0 >> 16), h1 = (int)(w1 & 0xFFFFu), a1 = (int)(w1 >> 16);
                int lhs0, rhs0, lhs1, rhs1;
                window_flanks(a0, W, (int)(p.hp.off[h0 + 1] - p.hp.off[h0]), reg.lhs, reg.rhs, &lhs0, &rhs0);
                window_flanks(a1, W, (int)(p.hp.off[h1 + 1] - p.hp.off[h1]), reg.lhs, reg.rhs, &lhs1, &rhs1);
                const FbBounds g = fb_bounds(lhs0, W - rhs0, lhs1, W - rhs1, W);
                dp_flank_bwd<BAND>(rows, L_o, tab + p.hp.off[h0] + a0, tab + p.hp.off[h1] + a1, nucp, g, bscr_fn, bstride, (uint32_t)p.one);
                x0 = w0; x1 = w1;
            }
            asm volatile("" : "+r"(li_o), "+r"(r_o), "+r"(n_o), "+r"(L_o), "+r"(x0), "+r"(x1));
            const bool v1 = i1 < n_o;
            const int W = L_o + K - 1;
            const RegionInfo reg = p.regs[p.rd.region[r_o]];
            const uint32_t* npre = p.rd.reverse[r_o] ? p.hp.npre_r : p.hp.npre_f;
            const int h0 = (int)(x0 & 0xFFFFu), a0 = (int)(x0 >> 16), h1 = (int)(x1 & 0xFFFFu), a1 = (int)(x1 >> 16);
            int lhs0, rhs0, lhs1, rhs1;
            window_flanks(a0, W, (int)(p.hp.off[h0 + 1] - p.hp.off[h0]), reg.lhs, reg.rhs, &lhs0, &rhs0);
            window_flanks(a1, W, (int)(p.hp.off[h1 + 1] - p.hp.off[h1]), reg.lhs, reg.rhs, &lhs1, &rhs1);
            const FbBounds g = fb_bounds(lhs0, W - rhs0, lhs1, W - rhs1, W);
            FbResult f0, f1;
            fb_finish(K, L_o, g, pair_scratch + (size_t)(base + c) * fb_round_words(BAND) + lane, 32, bscr_fn(), bstride, &f0, &f1);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                if (half && !v1) continue;
                const FbResult f = half ? f1 : f0;
                const int h = half ? h1 : h0, a = half ? a1 : a0;
                // an in-flank 'N' column the DP may have charged less than the reference's replay does: exact traceback path instead
                if (flank_replay_may_differ_pre(npre + p.hp.off[h], a, W, half ? lhs1 : lhs0, half ? rhs1 : rhs0, low_quality)) push_slow(p, r_o, h, a);
                else if (f.tie) {
                    const int slot = atomicAdd(p.gcnt + li_o, 1);
                    if (slot < p.fcap) p.gtasks[(size_t)li_o * p.fcap + slot] = half ? x1 : x0;
                    else atomicOr(p.flags, 8);
                    *p.any_flank_tasks = 1;
                } else atomicMin(p.best + pair_slot(p.rd, h, r_o), discount_flank(f.score, f.flank, L_o, f.mask, 0));
            }
        }
    }
}

// Generic path of populate: reads the fast path cannot take (non-ACGT bases, 16-bit-unsafe qualities, very long reads)
// or every read when the band is > 32 / int32 scores were requested. One thread per (haplotype, read) pair.
// With FASTQ it is the classify pass of the fast path instead: the same candidate walk over the fast work list (the pair
// list, entries may be -1), but score-only DP candidates are appended to the read's task list for k_populate_fast.
template <int MAXK, bool FASTQ>
__device__ __forceinline__ void populate_one_pair(const PopParams& p, const int li, const int hl)
{
    const int r = p.list[li];
    if (r < 0) return;
    const RegionInfo reg = p.regs[p.rd.region[r]];
    if (hl >= reg.nH) return;                      // a slot beyond this read's region
    const int h = reg.h0 + hl;
    const long long slot_hr = pair_slot(p.rd, h, r);
    const bool rev = p.rd.reverse[r] != 0;
    const HapView hv = hap_view(p.hp, h, rev);
    const ReadView rv = read_view(p.rd, r);
    const long long orig = (p.rd.begin ? p.rd.begin[r] : 0) - (p.hp.begin ? p.hp.begin[h] : 0);
    int npos = 0;
    const int32_t* pp = nullptr;
    if (p.pos_off) { const long long o = p.pos_off[slot_hr]; npos = (int)(p.pos_off[slot_hr + 1] - o); pp = p.pos + o; }
    else if (p.kcnt) { npos = p.kcnt[(size_t)li * p.Hmax + hl]; pp = p.kpos + ((size_t)li * p.Hmax + hl) * kMaxMapped; }
    EnumState st {false, false};
    int best = kBestInf;
    // DP candidates are collected first and queued after the walk: a shortcut value of 0 (exact match at some candidate
    // position) cannot be improved on — every candidate's penalty is >= 0 and the pair's result is their minimum — so the
    // pair's DPs are skipped without changing the result.
    constexpr int kMaxPending = 12;
    int pend_a[kMaxPending];
    unsigned pend_flank = 0u;
    int n_pend = 0;
    auto flush_pending = [&](const int count) {
        for (int i2 = 0; i2 < count; ++i2) {
            const int v = pend_a[i2];
            // reads with 'N' on the pair list: every DP on the 32-bit flank kernel (its lookup has the fifth cap); on the wide
            // list the score-only kernel has it too
            const bool to_32bit = FASTQ && p.list_kind == 0 && (p.rd.info[r].y & kReadHasN);
            if (!((pend_flank >> i2) & 1u) && !to_32bit) {
                if (FASTQ) {
                    const int slot = list_append_slot(p.fcnt, li);
                    if (slot < p.fcap) p.ftasks[(size_t)li * p.fcap + slot] = (uint32_t)h | ((uint32_t)v << 16);
                    else atomicOr(p.flags, 8);
                } else {
                    const GenericModel gm {hv.seq + v, hv.snv_mask + v, hv.snv_prior + v, hv.gap_open + v, hv.gap_extend + v, p.nuc_prior};
                    best = min(best, generic_align<false, MAXK>(p.band, gm, rv.bases, (const int8_t*)rv.quals, rv.len, nullptr, 1, 0, 0, nullptr, nullptr, nullptr));
                }
            } else {
                if (FASTQ && p.band <= 32 && !(p.rd.info[r].y & kReadUnsafeFlank32)) {
                    // which flank-aware kernel: window-coordinate flanks of this candidate (pair_hmm.hpp:573-588)
                    int route = 0;                                   // 0: crossing-cell kernel, 1: lean kernel, 2: plain score-only DP
                    if ((pend_flank >> i2) & 1u) {
                        const int W = rv.len + 2 * p.band - 1;
                        int lhs, rhs;
                        window_flanks(v, W, hv.len, reg.lhs, reg.rhs, &lhs, &rhs);
                        const int xl = lhs, xr = W - rhs;
                        if (xr <= xl) route = to_32bit ? 0 : 2;      // the flanks cover the whole window: the result is the plain score (:757-759)
                        else if (lhs == 0 && rhs == 0 && !to_32bit) route = 2;   // no flank column inside the window: nothing to discount
                        else if (!(p.rd.info[r].y & kReadHasN) && p.atasks &&
                                 (p.fb_route ? rv.len >= 2 * p.band : flank_mask_cannot_zero(rv.len, p.band, xl, xr >= W ? W + 1 : xr))) route = 1;
                    }
                    uint32_t* tasks = route == 0 ? p.gtasks : route == 1 ? p.atasks : p.ftasks;
                    int* counts = route == 0 ? p.gcnt : route == 1 ? p.acnt : p.fcnt;
                    const int slot = list_append_slot2(counts, li, route);
                    if (slot < p.fcap) tasks[(size_t)li * p.fcap + slot] = (uint32_t)h | ((uint32_t)v << 16);
                    else atomicOr(p.flags, 8);
                    if (route == 0) *p.any_flank_tasks = 1;
                    if (route == 1) *p.any_acc_tasks = 1;
                } else push_slow(p, r, h, v);
            }
        }
    };
    for (int c = 0; c < npos + 2; ++c) {
        int pos;
        const int k = candidate_slot(c, npos, pp, orig, rv.len, hv.len, p.band, st, &pos);
        if (k < 0) { p.status[slot_hr] = 2 | (min(pos, 0x7FFF) << 16); atomicOr(p.flags, 2); continue; }
        if (k == 0) continue;
        int v;
        const CandKind kind = classify_candidate(hv, rv, p.band, pos, p.shortcut != 0, reg.use_flanks != 0, reg.lhs, reg.rhs, &v);
        if (kind == CAND_VALUE) best = min(best, v);
        else if (kind == CAND_DP || kind == CAND_DP_FLANK) {
            if (n_pend == kMaxPending) {      // a long caller-supplied list: queue what has been collected and go on (no pair is truncated)
                flush_pending(n_pend);
                n_pend = 0; pend_flank = 0u;
            }
            pend_a[n_pend] = v;
            if (kind == CAND_DP_FLANK) pend_flank |= 1u << n_pend;
            ++n_pend;
        }
    }
    if (best == 0) n_pend = 0;
    flush_pending(n_pend);
    if (best != kBestInf) atomicMin(p.best + slot_hr, best);
}


template <int MAXK, bool FASTQ>
__global__ void k_populate_generic(const PopParams p)
{
    const int n_list = tile_list(p);
    const long long total = (long long)n_list * p.Hmax, step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        int li, hl;
        split_index(i, p.Hmax, &li, &hl);
        populate_one_pair<MAXK, FASTQ>(p, li, hl);
    }
}

// Score-only DP tasks of the wide list (32-bit lanes, dp_band<Lanes32>): persistent warps, one READ per warp (row entries in
// shared memory), 32 / NL tasks per round with NL lanes each. Serves use_int_scores, reads whose quality sum does not fit a
// 16-bit lane, reads beyond the pairing scheduler's length bins (long reads), and reads with 'N' at bands > 32.
template <int C, int NL>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32)
k_populate_wide(const PopParams p)
{
    extern __shared__ RowEntry smem_rows[];
    constexpr int TPR = 32 / NL;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = lane / NL, j = lane % NL;
    RowEntry* rows = smem_rows + warp * p.row_stride;
    if (on_reserved_sm(p)) return;
    const int n_list = tile_list(p);
    const bool oge = open_ge_extend(p.flags);
    for (;;) {
        int li = 0;
        if (lane == 0) li = atomicAdd(p.pair_cursor, 1);
        li = __shfl_sync(0xffffffffu, li, 0);
        if (li >= n_list) break;
        const int r = p.list[li];
        const int n = r >= 0 ? p.fcnt[li] : 0;
        if (n == 0) continue;
        const int L = p.rd.info[r].x;
        __syncwarp();
        {
            const uint16_t* hr = p.rd.rowhalf + p.rd.off[r];
            for (int y = lane; y < L; y += 32) rows[y] = make_row_entry32(hr[y]);
            if (lane == 0) rows[L] = pad_row_entry32();
            __syncwarp();
        }
        const ColEntry* tab = p.rd.reverse[r] ? p.hp.tab_r : p.hp.tab_f;
        const uint32_t* q = p.ftasks + (size_t)li * p.fcap;
        for (int c = 0; c < n; c += TPR) {
            const bool valid = c + slot < n;
            const uint32_t t = q[valid ? c + slot : 0];
            const int h = (int)(t & 0xFFFFu), a = (int)(t >> 16);
            const Lanes32::Tab tb {tab + p.hp.off[h] + a};
            const uint32_t res = oge ? dp_band<Lanes32, C, NL, true>(rows, L, tb, (uint32_t)p.nuc_prior, j, (uint32_t)p.one)
                                     : dp_band<Lanes32, C, NL, false>(rows, L, tb, (uint32_t)p.nuc_prior, j, (uint32_t)p.one);
            if (valid && j == 0) atomicMin(p.best + pair_slot(p.rd, h, r), (int)res);
        }
    }
}

// Near-flank candidates: traceback DP + flank discount (pair_hmm.hpp:743-764). Grid-stride over the slow queue; each
// thread owns an interleaved back-pointer scratch (cell c of thread t at bp[c * nthreads + t]).
template <int MAXK>
__global__ void k_slow_flank(const PopParams p, unsigned char* __restrict__ bp)
{
    const int nthreads = gridDim.x * blockDim.x, tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = min(*p.slow_count, p.slow_cap);
    for (int i = tid; i < n; i += nthreads) {
        const int4 t = p.slow[i];
        const int r = t.x, h = t.y, a = t.z;
        const HapView hv = hap_view(p.hp, h, p.rd.reverse[r] != 0);
        const ReadView rv = read_view(p.rd, r);
        const int W = rv.len + 2 * p.band - 1;
        const GenericModel gm {hv.seq + a, hv.snv_mask + a, hv.snv_prior + a, hv.gap_open + a, hv.gap_extend + a, p.nuc_prior};
        int lhs, rhs, fp, fs, ms;
        const RegionInfo reg = p.regs[p.rd.region[r]];
        window_flanks(a, W, hv.len, reg.lhs, reg.rhs, &lhs, &rhs);
        const int score = generic_align<true, MAXK>(p.band, gm, rv.bases, (const int8_t*)rv.quals, rv.len, bp + tid, (size_t)nthreads,
                                                    lhs, rhs, &fp, &fs, &ms);
        const int v = discount_flank(score, fs, rv.len, ms, fp);
        if (v != kBestInf) atomicMin(p.best + pair_slot(p.rd, h, r), v);
    }
}

// Per-call seam with traceback (reference hmm.align(..., first_pos, align1, align2), simd_pair_hmm.hpp:491-509): one
// thread, for parity with the reference's API — throughput comes from the batched entry points.
// buf layout: truth[W] mask[W] prior[W] go[W] ge[W] target[L] quals[L]; out: {score, first_pos}; strings after bp.
__global__ void k_align_one(const int band, const int L, const char* __restrict__ buf, const int nuc_prior,
                            unsigned char* __restrict__ bp, int* __restrict__ out, char* __restrict__ align1, char* __restrict__ align2)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int W = L + 2 * band - 1;
    const GenericModel gm {buf, buf + W, (const int8_t*)(buf + 2 * W), (const int8_t*)(buf + 3 * W), (const int8_t*)(buf + 4 * W), nuc_prior};
    int fp, fs, ms;
    out[0] = generic_align<true, kGenericMaxDiag>(band, gm, buf + 5 * W, (const int8_t*)(buf + 5 * W + L), L, bp, 1, 0, 0, &fp, &fs, &ms, align1, align2);
    out[1] = fp;
}

// ---------------------------------------------------------------------------------------------------------
// HaplotypeLikelihoodModel::align for explicit (read, haplotype) pairs (haplotype_likelihood_model.cpp:335-431):
// best alignment over the candidate mapping positions, with CIGAR (pair_hmm.hpp:152-188, 321-340, 784-823).
// ---------------------------------------------------------------------------------------------------------
struct AlignParams {
    DevHaps hp;
    DevReads rd;
    const int2* pairs;          // {read, hap}
    int n_pairs;
    const long long* pos_off;   // CSR over the pair list, or null
    const int32_t* pos;
    int band, nuc_prior, use_flanks, lhs_flank, rhs_flank;
    int use_mapq, mapq_cap, mapq_trigger;
    long long* mapping_position;
    double* likelihood;
    char* cigar;
    int cigar_stride;
    int* status;
    unsigned char* bp;          // interleaved back-pointer scratch: cell c of thread t at bp[c * nthreads + t]
    char* strings;              // per thread 4 * str_cap bytes
    int str_cap;
    int raw_offsets;            // 1: hmm::align semantics — pos[i] is pair i's target offset (phmm_align_pairs)
    // register traceback kernel (k_align_reads_fast): 0 = unused, else its band; longest read it takes; shared row stride; word scratch
    int fast_band, fast_max_len, fast_row_stride;
    uint32_t* bp32;
};

__device__ __forceinline__ int cigar_emit(char* out, int w, const int cap, int len, const char op)
{
    char tmp[12];
    int n = 0;
    do { tmp[n++] = (char)('0' + len % 10); len /= 10; } while (len > 0);
    while (n > 0 && w < cap - 1) out[w++] = tmp[--n];
    if (w < cap - 1) out[w++] = op;
    return w;
}

// make_cigar (pair_hmm.hpp:152-188) as text; returns false if it did not fit
__device__ inline bool make_cigar_text(const char* a1, const char* a2, char* out, const int cap)
{
    int n = 0;
    while (a1[n]) ++n;
    int i = 0, w = 0;
    while (i < n) {
        int j = i;
        while (j < n && a1[j] == a2[j]) ++j;
        if (j != i) { w = cigar_emit(out, w, cap, j - i, '='); if (j == n) break; }
        i = j;
        if (a1[i] == '-') { j = i + 1; while (j < n && a1[j] == '-') ++j; w = cigar_emit(out, w, cap, j - i, 'I'); }
        else if (a2[i] == '-') { j = i + 1; while (j < n && a2[j] == '-') ++j; w = cigar_emit(out, w, cap, j - i, 'D'); }
        else { j = i + 1; while (j < n && a1[j] != a2[j] && a1[j] != '-' && a2[j] != '-') ++j; w = cigar_emit(out, w, cap, j - i, 'X'); }
        i = j;
    }
    out[w < cap ? w : cap - 1] = 0;
    return w < cap - 1;
}

// One pair of the align list. RunDP(hv, rv, a, lhs, rhs, &fp, &fs, &ms, cur1, cur2) -> score runs the traceback DP of the window at
// offset a and leaves the two alignment strings in cur1 / cur2 (fp == -1: the path left the band).
// p.raw_offsets != 0 selects hmm::align itself (pair_hmm.hpp:858-874: ONE explicit target offset per pair — pos[i] — no in-range rule,
// no fallback; what DeNovoModel / haplotype_filter call): a window that does not fit yields {offset 0, lowest(), empty CIGAR}.
template <typename RunDP>
__device__ __forceinline__ void align_pair(const AlignParams& p, const int i, char* s0, RunDP&& run_dp)
{
    const int r = p.pairs[i].x, h = p.pairs[i].y;
    const HapView hv = hap_view(p.hp, h, p.rd.reverse[r] != 0);
    const ReadView rv = read_view(p.rd, r);
    const long long orig = (p.rd.begin ? p.rd.begin[r] : 0) - (p.hp.begin ? p.hp.begin[h] : 0);
    int npos = 0;
    const int32_t* pp = nullptr;
    if (p.pos_off) { const long long o = p.pos_off[i]; npos = (int)(p.pos_off[i + 1] - o); pp = p.pos + o; }
    char *cur1 = s0, *cur2 = s0 + p.str_cap, *best1 = s0 + 2 * p.str_cap, *best2 = s0 + 3 * p.str_cap;
    EnumState st {false, false};
    int best = kBestInf, status = 0;
    long long best_off = 0;
    bool best_exact = false, have = false;
    const int n_slots = p.raw_offsets ? 1 : npos + 2;
    for (int c = 0; c < n_slots && status == 0; ++c) {
        int pos;
        if (p.raw_offsets) pos = p.pos[i];
        else {
            const int k = candidate_slot(c, npos, pp, orig, rv.len, hv.len, p.band, st, &pos);
            if (k < 0) { status = 2 | (min(pos, 0x7FFF) << 16); break; }
            if (k == 0) continue;
        }
        int v; long long off; bool exact = false;
        bool eq = pos >= 0 && pos + rv.len <= hv.len;                         // try_naive_align (:321-340)
        for (int a = 0; eq && a < rv.len; ++a) if (rv.bases[a] != hv.seq[pos + a]) eq = false;
        if (eq) { v = 0; off = pos; exact = true; }
        else {
            const int W = rv.len + 2 * p.band - 1;
            const int a = pos - p.band > 0 ? pos - p.band : 0;
            if (pos < 0 || a + W > hv.len) { v = kBestInf; off = 0; cur1[0] = 0; cur2[0] = 0; }          // :802-807
            else {
                const bool near_flank = p.use_flanks && (pos < p.lhs_flank + p.band || pos + rv.len + p.band > hv.len - p.rhs_flank);
                int lhs = 0, rhs = 0, fp, fs, ms;
                if (near_flank) window_flanks(a, W, hv.len, p.lhs_flank, p.rhs_flank, &lhs, &rhs);
                int score = run_dp(hv, rv, a, lhs, rhs, &fp, &fs, &ms, cur1, cur2);
                if (fp == -1) { status = 4; break; }                                             // HMMOverflow (:815-817)
                if (near_flank) { if (rv.len - ms < 2) fs = 0; score = fs <= score ? score - fs : score + fs; }   // :659-672
                v = score; off = (long long)pos - p.band + fp;                                    // :820
            }
        }
        // :355 listed positions win on '>', :365 the original position on '>=', :388-391 the fallback unconditionally
        const bool take = p.raw_offsets ? true : (c < npos ? (v < best) : (c == npos ? (v <= best) : true));
        if (take || !have) {
            if (take) {
                best = v; best_off = off; best_exact = exact; have = true;
                char* t = cur1; cur1 = best1; best1 = t; t = cur2; cur2 = best2; best2 = t;
            }
        }
    }
    p.status[i] = status;
    char* cg = p.cigar + (size_t)i * p.cigar_stride;
    cg[0] = 0;
    if (status == 0) {
        p.mapping_position[i] = best_off;
        p.likelihood[i] = finish_likelihood(best, p.use_mapq != 0, p.rd.mapq ? p.rd.mapq[r] : 0, p.mapq_cap, p.mapq_trigger);
        bool ok = true;
        if (best_exact) { const int w = cigar_emit(cg, 0, p.cigar_stride, rv.len, '='); cg[w] = 0; }
        else if (best != kBestInf) ok = make_cigar_text(best1, best2, cg, p.cigar_stride);
        if (!ok) p.status[i] = 3;
    } else {
        p.mapping_position[i] = 0;
        p.likelihood[i] = -1.7976931348623157e308;
    }
}

// Reads the register traceback can take: alphabet ACGTN, qualities <= 127, quality sum inside the 16-bit score field, row entries
// of every thread of a block in shared memory.
__device__ __forceinline__ bool align_fast_ok(const AlignParams& p, const int r)
{
    const int2 inf = p.rd.info[r];
    return p.fast_band != 0 && (inf.y & (kReadNonACGT | kReadBadQual | kReadUnsafe16)) == 0 && inf.x >= 1 && inf.x <= p.fast_max_len;
}

// Generic traceback (any band / alphabet): one thread per pair, band in local memory, byte back-pointers. Serves what the register
// kernel below cannot take.
template <int MAXK>
__global__ void k_align_reads(const AlignParams p)
{
    const int nthreads = gridDim.x * blockDim.x, tid = blockIdx.x * blockDim.x + threadIdx.x;
    char* s0 = p.strings + (size_t)tid * 4 * p.str_cap;
    for (int i = tid; i < p.n_pairs; i += nthreads) {
        if (align_fast_ok(p, p.pairs[i].x)) continue;            // k_align_reads_fast's
        align_pair(p, i, s0, [&](const HapView& hv, const ReadView& rv, const int a, const int lhs, const int rhs, int* fp, int* fs, int* ms, char* c1, char* c2) {
            const GenericModel gm {hv.seq + a, hv.snv_mask + a, hv.snv_prior + a, hv.gap_open + a, hv.gap_extend + a, p.nuc_prior};
            return generic_align<true, MAXK>(p.band, gm, rv.bases, (const int8_t*)rv.quals, rv.len, p.bp + tid, (size_t)nthreads, lhs, rhs, fp, fs, ms, c1, c2);
        });
    }
}

// Register traceback (dp_traceback_forward + traceback_walk): one thread per pair, the band in registers, one back-pointer word
// per cell (coalesced across the threads), the thread's read staged in shared memory.
constexpr int kAlignFastThreads = 64;
template <int BAND>
__global__ void __launch_bounds__(kAlignFastThreads)
k_align_reads_fast(const AlignParams p)
{
    extern __shared__ uint16_t smem_rows16[];
    uint16_t* rows = smem_rows16 + (size_t)threadIdx.x * p.fast_row_stride;     // stride = 2 * odd: the threads of a warp hit distinct banks
    const int nthreads = gridDim.x * blockDim.x, tid = blockIdx.x * blockDim.x + threadIdx.x;
    char* s0 = p.strings + (size_t)tid * 4 * p.str_cap;
    for (int i = tid; i < p.n_pairs; i += nthreads) {
        const int r = p.pairs[i].x;
        if (!align_fast_ok(p, r)) continue;
        {
            const long long ro = p.rd.off[r];
            const int L = p.rd.info[r].x;
            for (int y = 0; y < L; ++y) rows[y] = p.rd.rowhalf[ro + y];
            rows[L] = 0;                                                         // the pad row: code 0, quality 0
        }
        const ColEntry* tabs = p.rd.reverse[r] ? p.hp.tab_r : p.hp.tab_f;
        const int h = p.pairs[i].y;
        align_pair(p, i, s0, [&](const HapView& hv, const ReadView& rv, const int a, const int lhs, const int rhs, int* fp, int* fs, int* ms, char* c1, char* c2) {
            int score, x_end, state;
            dp_traceback_forward<BAND>(TbRows2 {rows}, rv.len, tabs + p.hp.off[h] + a, p.nuc_prior, p.bp32 + tid, (size_t)nthreads, &score, &x_end, &state);
            const TbModel gm {hv.seq + a, hv.snv_mask + a, hv.snv_prior + a, hv.gap_open + a, hv.gap_extend + a, p.nuc_prior};
            traceback_walk<BAND>(p.bp32 + tid, (size_t)nthreads, gm, rv.bases, rv.quals, rv.len, x_end, state, lhs, rhs, fp, fs, ms, c1, c2);
            return score;
        });
    }
}


// N1 (SURVEY.md §8f): ConstantMixtureGenotypeLikelihoodModel::evaluate on the resident [H][R] matrix
// (core/models/genotype/constant_mixture_genotype_likelihood_model.cpp:30-140): one block per genotype,
// ln p(reads | g) = sum_r ( log_sum_exp_{h in g} lnl[h][r] - ln ploidy ); homozygous genotypes reduce to a plain sum.
__global__ void __launch_bounds__(256)
k_genotype_likelihoods(const double* __restrict__ lnl, const int R, const int* __restrict__ genotypes, const int ploidy, double* __restrict__ out)
{
    __shared__ double partial[256];
    const int g = blockIdx.x;
    const int* gt = genotypes + (size_t)g * ploidy;
    bool homo = true;
    for (int k = 1; k < ploidy; ++k) homo = homo && gt[k] == gt[0];
    const double ln_ploidy = log((double)ploidy);
    double acc = 0.0;
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        if (homo) { acc += lnl[(size_t)gt[0] * R + r]; continue; }
        double mx = lnl[(size_t)gt[0] * R + r];
        for (int k = 1; k < ploidy; ++k) mx = fmax(mx, lnl[(size_t)gt[k] * R + r]);
        double sum = 0.0;
        for (int k = 0; k < ploidy; ++k) sum += exp(lnl[(size_t)gt[k] * R + r] - mx);
        acc += mx + log(sum) - ln_ploidy;
    }
    partial[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) { if ((int)threadIdx.x < s) partial[threadIdx.x] += partial[threadIdx.x + s]; __syncthreads(); }
    if (threadIdx.x == 0) out[g] = ploidy == 0 ? 0.0 : partial[0];
}

__global__ void k_fill_int(int* __restrict__ p, const long long n, const int v)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// Floating-point epilogue (haplotype_likelihood_model.cpp:285-303): out[h][r] in double.
__global__ void k_epilogue(const int* __restrict__ best, int* __restrict__ status, const DevReads rd, const RegionInfo* __restrict__ regs,
                           const int Hmax, const int use_mapq, const int mapq_cap, const int mapq_trigger, double* __restrict__ out,
                           const long long out_row_extra /* single region only: output row stride minus the read count */)
{
    // thread t = (haplotype slot, read), reads fastest: consecutive threads write consecutive outputs within a region
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)Hmax * rd.n) return;
    int hl, r;
    split_index(t, rd.n, &hl, &r);
    const RegionInfo g = regs[rd.region[r]];
    if (hl >= g.nH) return;
    const long long i = pair_slot(rd, g.h0 + hl, r);
    const int b = best[i];
    if (b == kBestInf && status[i] == 0) status[i] = 1;
    // `out` may be another GPU's memory (a peer mapping, phmm_ipc_open): plain coalesced stores, nothing is read back
    out[i + hl * out_row_extra] = finish_likelihood(b, use_mapq != 0, rd.mapq[r], mapq_cap, mapq_trigger);
}

// Template epilogue: k_epilogue for the reads of one template and HaplotypeLikelihoodModel::evaluate(AlignedTemplate)
// (haplotype_likelihood_model.cpp:306-320) in one pass — the per-read doubles never reach memory. Thread = (haplotype slot, template),
// templates fastest: consecutive threads store consecutive outputs of a region's [nH][nT] matrix at tout_off.
__global__ void k_template_epilogue(const int* __restrict__ best, int* __restrict__ status, const DevReads rd, const RegionInfo* __restrict__ regs,
                                    const int Hmax, const int n_templates, const long long* __restrict__ toff, const int* __restrict__ tregion,
                                    const int use_mapq, const int mapq_cap, const int mapq_trigger, const int* __restrict__ flags,
                                    double* __restrict__ tout)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)Hmax * n_templates) return;
    if (*flags & kFlagBadTemplates) return;        // offsets that k_check_templates rejected are not followed
    int hl, t;
    split_index(i, n_templates, &hl, &t);
    const RegionInfo g = regs[tregion[t]];
    if (hl >= g.nH) return;
    const long long row = g.out_off + (long long)hl * g.nR - g.r0;     // pair_slot(rd, g.h0 + hl, r) == row + r
    double acc = 0.0;
    for (long long r = toff[t], end = toff[t + 1]; r < end; ++r) {
        const long long s = row + r;
        const int b = best[s];
        if (b == kBestInf && status[s] == 0) status[s] = 1;
        // the sum in read order from 0.0, like std::accumulate; __dadd_rn keeps the additions out of any fused multiply-add
        acc = __dadd_rn(acc, finish_likelihood(b, use_mapq != 0, rd.mapq[r], mapq_cap, mapq_trigger));
    }
    tout[g.tout_off + (long long)hl * g.nT + (t - g.t0)] = acc;
}

} // namespace phmm
