// Device-side building blocks of the B200 pair-HMM engine (sm_100a).
//
// Recurrence: the integer min-plus banded DP of the reference kernel
//   /root/reference/src/core/models/pairhmm/simd_pair_hmm.hpp:240-324 (align_helper)
// restated in (x, y) prefix coordinates (x truth-window bases, y read bases consumed; band 0 <= x-y <= 2B-1):
//   S          = min(m, i, d)                                    (:284, :308)
//   m(x+1,y+1) = S + sub(x, y)                                   (:121-132 update_match_state)
//   d(x+1,y)   = min(d + gap_extend[x], min(mg, i) + gap_open[x])            (:293, :317; I→D allowed)
//   i(x,y+1)   = min(i + gap_extend[x-1], mg + gap_open[x-1]) + nuc_prior    (:295, :318-319; no D→I)
//   y == 0: m = 0 (free start, rolling_initializer.hpp:39-51); mg = 0 for odd x, +inf for even x (the gap
//   transitions of even-x cells are computed before the initialiser touches them, :282-283 vs :317-319)
//   result = min over x of S(x, L)                               (:285-291, :309-315, :323)
//
// The implementations that live here:
//   * dp_pair<BAND>  — the fast path. One THREAD owns TWO alignments packed as s16x2 in every register and sweeps
//     the band column by column (x outer, diagonal k = x-y unrolled in registers). No shuffles, no shared-memory
//     DP state. The per-cell work is 10 integer instructions for 2 cells using Blackwell's DPX packed-16 ops
//     (VIMNMX3.S16x2, VIADDMNMX.S16x2, VIMNMX.S16x2) and PRMT byte-table lookups for the emission.
//   * dp_band / dp_band_roles — the same cell with the band's diagonals split over lanes or warps (bands 32 ... 256, 32-bit lanes).
//   * dp_flank_fwd / dp_flank_bwd / fb_finish — the flank-aware path, packed: forward pass to the flank boundary, backward pass
//     (cost-to-go) from the window end, crossing cell = argmin F + B; dp_flank32 / dp_flank_acc — the labelled one-alignment-per-
//     thread forms that reproduce the reference's traceback tie-breaks (fallback for ties, reads with 'N', short reads, band 32).
//   * dp_traceback_forward + traceback_walk — best alignment + CIGAR (register band, one back-pointer word per cell).
//   * generic_align  — int32, any band, any alphabet, optional traceback + flank replay. Exactness fallback.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace phmm {

// ---------------------------------------------------------------------------------------------------------
// Encodings shared by the preparation kernels and the DP kernels
// ---------------------------------------------------------------------------------------------------------

// Haplotype column table entry (8 bytes per haplotype base per strand):
//   .x = four emission caps, byte b = cost cap when the read base has code b (A0 C1 G2 T3):
//          0                                   if truth[x] == base
//          min(snv_prior[x] if snv_mask[x]==base else 127,  2 if truth[x]=='N' else 127)   otherwise
//        sub(x, y) = min(qual[y], cap[x][read[y]])  — identical to update_match_state for quals, priors in [0,127].
//        All caps are < 0x80, which lets PRMT's sign-replicate mode manufacture the zero bytes of the packed lanes.
//   .y = gap_open[x] | gap_extend[x] << 8 | capN[x] << 16   (capN: the cap for a read base 'N': 0 if truth[x] == 'N',
//        else snv_prior[x] if snv_mask[x] == 'N', else 127; top byte zero)
typedef uint2 ColEntry;

constexpr uint32_t kCapInf   = 127u;      // "no cap": min(q, 127) == q for every int8 quality
constexpr uint32_t kInf16    = 0x7000u;   // +inf of the packed 16-bit lanes; kInf16 + 2*127 + nuc stays < 0x8000
constexpr uint32_t kInf16x2  = kInf16 | (kInf16 << 16);
constexpr int      kInf32    = 1 << 28;   // +inf of the int32 kernel
constexpr int      kFlagOpenBelowExtend = 16;    // engine flag word: some haplotype base has gap_open < gap_extend (see dp_pair, OGE)
constexpr int      kFlagBadTemplates = 32;       // engine flag word: device-resident template offsets failed k_check_templates
constexpr int      kMaxScore16 = 0x7000 - 1024;  // a read whose sum of qualities is below this cannot overflow a 16-bit lane

// Read row half-word: code | qual << 8 (code: A0 C1 G2 T3, N4). Reads with an 'N' are served by the 32-bit kernel (its
// PRMT lookup has a fifth cap); reads containing any other byte take the generic path.
__host__ __device__ inline int base_code(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : c == 'N' ? 4 : -1; }

// The DP cores are __host__ __device__ so that tests/ can run the very same code on the CPU (with the few
// sm_100a instructions emulated below) against the CPU checker without a GPU. The product library never calls the
// host instantiations: every exported entry point launches kernels.
#define PHMM_HD __host__ __device__ __forceinline__

#ifdef __CUDA_ARCH__
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ uint32_t vmin2(uint32_t a, uint32_t b) { return __vmins2(a, b); }                              // VIMNMX.S16x2
__device__ __forceinline__ uint32_t vminu2(uint32_t a, uint32_t b) { return __vminu2(a, b); }                             // VIMNMX.U16x2
__device__ __forceinline__ uint32_t vmaxu2(uint32_t a, uint32_t b) { return __vmaxu2(a, b); }                             // VIMNMX.U16x2 (max)
__device__ __forceinline__ uint32_t vmin3(uint32_t a, uint32_t b, uint32_t c) { return __vimin3_s16x2(a, b, c); }       // VIMNMX3.S16x2
__device__ __forceinline__ uint32_t vaddmin(uint32_t a, uint32_t b, uint32_t c) { return __viaddmin_s16x2(a, b, c); }   // VIADDMNMX.S16x2: min(a+b, c)
template <typename T> __device__ __forceinline__ T ldg(const T* p) { return __ldg(p); }
#else
inline uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)   // PTX prmt.b32 default mode, incl. sign replication (nibble bit 3)
{
    const uint64_t src = (uint64_t)a | ((uint64_t)b << 32);
    uint32_t d = 0;
    for (int i = 0; i < 4; ++i) {
        const uint32_t n = (sel >> (4 * i)) & 0xF;
        uint32_t byte = (uint32_t)(src >> (8 * (n & 7))) & 0xFF;
        if (n & 8) byte = (byte & 0x80) ? 0xFF : 0x00;
        d |= byte << (8 * i);
    }
    return d;
}
inline uint32_t emu_pack(int lo, int hi) { return ((uint32_t)lo & 0xFFFFu) | (((uint32_t)hi & 0xFFFFu) << 16); }
inline int emu_lo(uint32_t v) { return (int16_t)(v & 0xFFFF); }
inline int emu_hi(uint32_t v) { return (int16_t)(v >> 16); }
inline int emu_min(int a, int b) { return a < b ? a : b; }
inline uint32_t vmin2(uint32_t a, uint32_t b) { return emu_pack(emu_min(emu_lo(a), emu_lo(b)), emu_min(emu_hi(a), emu_hi(b))); }
inline uint32_t vmin3(uint32_t a, uint32_t b, uint32_t c) { return vmin2(vmin2(a, b), c); }
inline uint32_t vminu2(uint32_t a, uint32_t b)
{
    const uint32_t al = a & 0xFFFFu, bl = b & 0xFFFFu, ah = a >> 16, bh = b >> 16;
    return (al < bl ? al : bl) | ((ah < bh ? ah : bh) << 16);
}
inline uint32_t vmaxu2(uint32_t a, uint32_t b)
{
    const uint32_t al = a & 0xFFFFu, bl = b & 0xFFFFu, ah = a >> 16, bh = b >> 16;
    return (al > bl ? al : bl) | ((ah > bh ? ah : bh) << 16);
}
inline uint32_t vaddmin(uint32_t a, uint32_t b, uint32_t c)
{
    return emu_pack(emu_min((int16_t)(emu_lo(a) + emu_lo(b)), emu_lo(c)), emu_min((int16_t)(emu_hi(a) + emu_hi(b)), emu_hi(c)));
}
template <typename T> inline T ldg(const T* p) { return *p; }
#endif

// Row entry of a read PAIR (one per read position y, shared by every lane that aligns this pair), 8 bytes so that one
// LDS.64 broadcast feeds a cell:
//   .x  PRMT selector: nibble0 = code0, nibble1 = 8 (sign-replicate → 0x00), nibble2 = 4|code1, nibble3 = 8
//   .y  qual0 | qual1 << 16
// so that  cap = prmt(caps0, caps1, row.x) = cap0[code0] | cap1[code1] << 16   and   qual = row.y
typedef uint2 RowEntry;
PHMM_HD RowEntry make_row_entry(uint32_t half0, uint32_t half1)
{
    // half = code | qual << 8
    RowEntry r;
    r.x = prmt(half0, half1, 0x2240u) | 0x8480u;   // bytes [code0, code1, 0, 0] + the two sign-replicate flags
    r.y = prmt(half0, half1, 0x2521u);             // bytes [qual0, 0, qual1, 0]
    return r;
}
PHMM_HD RowEntry pad_row_entry() { RowEntry r; r.x = 0x8480u; r.y = 0u; return r; }   // code 0 / qual 0: sub = min(0, cap) = 0

// Column table entry of one haplotype base (prior, go, ge must be in [0,127]; checked by the preparation kernel).
PHMM_HD ColEntry make_col_entry(const char truth, const char snv_mask, const int snv_prior, const int gap_open, const int gap_extend)
{
    const uint32_t ncost = truth == 'N' ? 2u : kCapInf;
    uint32_t caps = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const char base = b == 0 ? 'A' : b == 1 ? 'C' : b == 2 ? 'G' : 'T';
        uint32_t cap = 0;
        if (truth != base) {
            cap = snv_mask == base ? (uint32_t)snv_prior : kCapInf;
            if (ncost < cap) cap = ncost;
        }
        caps |= cap << (8 * b);
    }
    const uint32_t cap_n = truth == 'N' ? 0u : (snv_mask == 'N' ? (uint32_t)snv_prior : kCapInf);
    ColEntry e;
    e.x = caps;
    e.y = (uint32_t)gap_open | ((uint32_t)gap_extend << 8) | (cap_n << 16);
    return e;
}   // code 0 / qual 0 for both halves: sub = min(0, cap) = 0

// a + b computed as a * one + b with `one` (== 1) opaque to the compiler: an IMAD on the FMA pipe instead of an IADD that ptxas
// would fuse into a VIADDMNMX on the (binding) ALU pipe
#ifdef __CUDA_ARCH__
__device__ __forceinline__ uint32_t fma_add(uint32_t a, uint32_t b, uint32_t one) { uint32_t d; asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(one), "r"(b)); return d; }
#else
inline uint32_t fma_add(uint32_t a, uint32_t b, uint32_t one) { return a * one + b; }
#endif

// ---------------------------------------------------------------------------------------------------------
// Fast path: two alignments per thread, s16x2 lanes, band state in registers
// ---------------------------------------------------------------------------------------------------------
//
// rows : shared-memory row entries of this lane's read pair, rows[0..L-1] real, rows[L] = pad_row_entry()
// t0/t1: column tables of the two haplotype windows (already offset to the window start); W = L + 2*BAND - 1
//        entries are read at indices 0..W-1 only
// Returns best0 | best1 << 16 (each the integer phred score of reference hmm.align()).
//
// Column x holds the cells k = x - y, k in [max(0, x-L), min(2B-1, x)], processed in DESCENDING k so that the
// insertion chain i(x, y+1) ← (x, y) runs through one register (i_run); M[k] / D[k] carry the match / deletion
// arrivals to the next column in place. Row L uses the pad row entry (qual 0 → sub 0), so after the cell
// (x, L) is processed M[x-L] holds S(x, L) and is never touched again: the end-row minimum is min_k M[k].
//
// Four column bodies, all fully unrolled over k with M / D in registers:
//   steady    2B <= x <= L      every cell exists
//   prologue  x < 2B, x <= L    cell (x, 0) is the free start; cells k < x follow — entered through a jump table
//   epilogue  x > L, x >= 2B    cells k >= x - L; leaves the unrolled sequence after the row-L cell
//   general   x < 2B, x > L     (reads shorter than the band) both limits, per-cell predicates
#define PHMM_REP8(F, b)  F(b + 7) F(b + 6) F(b + 5) F(b + 4) F(b + 3) F(b + 2) F(b + 1) F(b + 0)
#define PHMM_REP64(F)    PHMM_REP8(F, 56) PHMM_REP8(F, 48) PHMM_REP8(F, 40) PHMM_REP8(F, 32) PHMM_REP8(F, 24) PHMM_REP8(F, 16) PHMM_REP8(F, 8) PHMM_REP8(F, 0)

// OGE ("open >= extend"): the caller knows gap_open[x] >= gap_extend[x] for every column of both windows (true of every penalty
// array the reference's short-read error models produce — the PacBio tables break it inside long homopolymers, custom models may;
// k_build_tables raises kFlagOpenBelowExtend for such arrays and the kernels then instantiate OGE = false). Then
//   min(d + ge, min(m, i) + go) == min(d + ge, min(m, i, d) + go)        (d + go >= d + ge)
// and the deletion update re-uses S = min(m, i, d), which the match update needs anyway: 5 ALU-pipe instructions per cell pair
// instead of 6 (the ALU pipe is what binds this kernel, DESIGN.md section 4).
template <int BAND, bool OGE = false>
PHMM_HD uint32_t dp_pair(const RowEntry* __restrict__ rows, const int L,
                         const ColEntry* __restrict__ t0, const ColEntry* __restrict__ t1,
                         const uint32_t nucp /* nuc_prior in both halves */,
                         const uint32_t one = 1u /* the kernels pass an opaque 1: the cell's additions become IMADs on the FMA pipe (fma_add) */)
{
    constexpr int K = 2 * BAND;
    static_assert(K <= 64, "register band limited to 64 diagonals");
    uint32_t M[K], D[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { M[k] = 0u; D[k] = kInf16x2; }
    const int W = L + K - 1;
    ColEntry e0 = ldg(t0), e1 = ldg(t1);
    uint32_t go_prev = 0u, ge_prev = 0u;
    const RowEntry w0 = rows[0];

#define PHMM_CELL(k)                                                                        \
    {                                                                                       \
        const RowEntry w   = rp[-(k)];                                                      \
        const uint32_t sub = vmin2(w.y, prmt(caps0, caps1, w.x));                           \
        const uint32_t m = M[(k) < K ? (k) : 0], d = D[(k) < K ? (k) : 0];                  \
        const uint32_t s = vmin3(m, i_run, d);                                              \
        M[(k) < K ? (k) : 0] = fma_add(s, sub, one);                                        \
        if ((k) + 1 < K) D[((k) + 1) < K ? (k) + 1 : 0] = vaddmin(d, ge, fma_add(OGE ? s : vmin2(m, i_run), go, one)); \
        i_run = vaddmin(i_run, gep, fma_add(m, gop, one));                                  \
    }
#define PHMM_CASE_PROLOGUE(k) case (k) + 1: if ((k) < K) PHMM_CELL(k)
#define PHMM_CASE_ROW0(k)     case (k): if ((k) < K) M[(k) < K ? (k) : 0] = sub0; break;

    for (int x = 0; x <= W; ++x) {
        const int xn = (x + 1 < W) ? x + 1 : W - 1;
        const ColEntry n0 = ldg(t0 + xn), n1 = ldg(t1 + xn);
        const uint32_t caps0 = e0.x, caps1 = e1.x;
        const uint32_t go = prmt(e0.y, e1.y, 0x3430u);   // gap_open[x]   of both halves (byte 3 of .y is the zero source)
        const uint32_t ge = prmt(e0.y, e1.y, 0x3531u);   // gap_extend[x]
        const uint32_t gop = go_prev + nucp;             // gap_open[x-1] + nuc_prior
        const uint32_t gep = ge_prev + nucp;             // gap_extend[x-1] + nuc_prior
        const RowEntry* rp = rows + x;
        uint32_t i_run = kInf16x2;
        if (x >= K) {
            if (x <= L) {
                // steady state: every cell of the column exists
#pragma unroll
                for (int k = K - 1; k >= 0; --k) PHMM_CELL(k)
            } else {
                // epilogue: rows beyond L do not exist; stop after the row-L cell so that M[x-L] keeps S(x, L)
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    PHMM_CELL(k)
                    if (k == klo) break;
                }
            }
        } else {
            // cell (x, 0): S = 0, so m(x+1, 1) = sub(x, 0), and i(x, 1) = gap_open[x-1] + nuc for odd x, +inf for even x
            const uint32_t sub0 = vmin2(w0.y, prmt(caps0, caps1, w0.x));
            i_run = (x & 1) ? gop : kInf16x2;
            if (x <= L) {
                // prologue: cells k = x-1 .. 0 all exist — jump into the unrolled sequence at k = x-1
                switch (x) { PHMM_REP64(PHMM_CASE_PROLOGUE) default: break; }
                switch (x) { PHMM_REP64(PHMM_CASE_ROW0) default: break; }
            } else {
                // reads shorter than the band: both limits apply
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    if (k < x && k >= klo) PHMM_CELL(k)
                }
                switch (x) { PHMM_REP64(PHMM_CASE_ROW0) default: break; }
            }
        }
        go_prev = go; ge_prev = ge;
        // The next column's entries were loaded at the top of this column and must not be waited for before its end.
        // Left to itself ptxas copies them into e0 / e1 right after issuing the loads (a full L2 round trip per column,
        // 13 % of the kernel's stall samples in profiles/r01d). z is always 0 — no lane ever has its sign bit set — but
        // it is only known once the column's last cell is done, which pins the copy behind the column body.
        const uint32_t z = i_run & 0x80008000u;
        e0.x = n0.x + z; e0.y = n0.y + z; e1.x = n1.x + z; e1.y = n1.y + z;
    }
#undef PHMM_CELL
#undef PHMM_CASE_PROLOGUE
#undef PHMM_CASE_ROW0
    uint32_t best = M[0];
#pragma unroll
    for (int k = 1; k < K; ++k) best = vmin2(best, M[k]);
    return best;
}

// ---------------------------------------------------------------------------------------------------------
// Multi-lane band: the 2B diagonals of one alignment (pair) split over NL neighbouring lanes of a warp
// ---------------------------------------------------------------------------------------------------------
//
// Bands of 32 and more do not fit one thread's registers (band 32 = 128 band registers: the single-thread kernel spilled
// and ran at 46 % of the ALU pipe, profiles/r02a). Here every lane owns a CHUNK of C consecutive diagonals (C = 32, or 16
// for the 16-diagonal band) and sweeps it column by column exactly like dp_pair sweeps the whole band; NL = 2B / C lanes
// cooperate on one alignment. The two dependencies that cross a chunk boundary:
//   I  (x, y) -> (x, y+1): diagonal k -> k-1, SAME column  => the lane above must have finished the column first
//   D  (x, y) -> (x+1, y): diagonal k -> k+1, NEXT column  => the lane below must have started the previous column
// are both met when lane j+1 runs exactly ONE column ahead of lane j: in a step every lane first computes its TOP cell (whose
// D arrival the lane above needs for the last cell of the same step: one SHFL up), then the rest of its column, and hands
// the insertion chain leaving its bottom diagonal to the lane below for the next step (one SHFL down). Two shuffles per
// C cells; the price is the skew (NL - 1 extra steps) and divergence while neighbouring lanes are in different column
// bodies (prologue / steady / epilogue) — measured in profiles/.
// The lane functions are __host__ __device__ and split at the two exchange points so that tests/cpu_emul can run NL lanes
// in lock-step on the CPU; dp_band below is the device driver with the real shuffles.
//
// Traits select the value type: Lanes16 = two alignments per lane group packed s16x2 (as dp_pair), Lanes32 = one alignment
// in 32-bit lanes (int scores, long or high-quality-sum reads, reads holding 'N': the PRMT lookup has the fifth cap).
PHMM_HD uint32_t umin32(uint32_t a, uint32_t b) { return a < b ? a : b; }
#ifdef __CUDA_ARCH__
__device__ __forceinline__ uint32_t umin3_32(uint32_t a, uint32_t b, uint32_t c) { return __vimin3_u32(a, b, c); }            // VIMNMX3.U32
__device__ __forceinline__ uint32_t uaddmin32(uint32_t a, uint32_t b, uint32_t c) { return __viaddmin_u32(a, b, c); }        // VIADDMNMX.U32: min(a+b, c)
#else
inline uint32_t umin3_32(uint32_t a, uint32_t b, uint32_t c) { return umin32(umin32(a, b), c); }
inline uint32_t uaddmin32(uint32_t a, uint32_t b, uint32_t c) { return umin32(a + b, c); }
#endif

struct Lanes16 {
    typedef uint32_t V;
    struct Tab { const ColEntry* t0; const ColEntry* t1; };
    struct Ent { ColEntry a, b; };
    struct Col { uint32_t caps0, caps1, go, ge; };
    static PHMM_HD V inf() { return kInf16x2; }
    static PHMM_HD V both(const int v) { return (uint32_t)v | ((uint32_t)v << 16); }
    static PHMM_HD Ent load(const Tab& t, const int x) { Ent e; e.a = ldg(t.t0 + x); e.b = ldg(t.t1 + x); return e; }
    static PHMM_HD Col decode(const Ent& e)
    {
        Col c; c.caps0 = e.a.x; c.caps1 = e.b.x; c.go = prmt(e.a.y, e.b.y, 0x3430u); c.ge = prmt(e.a.y, e.b.y, 0x3531u); return c;
    }
    // keep the prefetched entries out of the live registers until the column is done (see dp_pair); tie is never negative
    static PHMM_HD void pin(Ent& dst, const Ent& src, const V tie)
    {
        const uint32_t z = tie & 0x80008000u;
        dst.a.x = src.a.x + z; dst.a.y = src.a.y + z; dst.b.x = src.b.x + z; dst.b.y = src.b.y + z;
    }
    static PHMM_HD V sub(const RowEntry& w, const Col& c) { return vmin2(w.y, prmt(c.caps0, c.caps1, w.x)); }
    static PHMM_HD V min2(V a, V b) { return vmin2(a, b); }
    static PHMM_HD V min3(V a, V b, V c) { return vmin3(a, b, c); }
    static PHMM_HD V addmin(V a, V b, V c) { return vaddmin(a, b, c); }
};
struct Lanes32 {
    typedef uint32_t V;
    struct Tab { const ColEntry* t0; };
    struct Ent { ColEntry a; };
    struct Col { uint32_t caps0, caps1, go, ge; };      // caps1 = the cap for a read 'N' (second PRMT operand, bytes 1..3 zero)
    static PHMM_HD V inf() { return (uint32_t)kInf32; }
    static PHMM_HD V both(const int v) { return (uint32_t)v; }
    static PHMM_HD Ent load(const Tab& t, const int x) { Ent e; e.a = ldg(t.t0 + x); return e; }
    static PHMM_HD Col decode(const Ent& e)
    {
        Col c; c.caps0 = e.a.x; c.caps1 = (e.a.y >> 16) & 0xFFu; c.go = e.a.y & 0xFFu; c.ge = (e.a.y >> 8) & 0xFFu; return c;
    }
    static PHMM_HD void pin(Ent& dst, const Ent& src, const V tie) { const uint32_t z = tie & 0x80000000u; dst.a.x = src.a.x + z; dst.a.y = src.a.y + z; }
    static PHMM_HD V sub(const RowEntry& w, const Col& c) { return umin32(w.y, prmt(c.caps0, c.caps1, w.x)); }   // rows: make_row_entry32
    static PHMM_HD V min2(V a, V b) { return umin32(a, b); }
    static PHMM_HD V min3(V a, V b, V c) { return umin3_32(a, b, c); }
    static PHMM_HD V addmin(V a, V b, V c) { return uaddmin32(a, b, c); }
};

#define PHMM_REP32(F)    PHMM_REP8(F, 24) PHMM_REP8(F, 16) PHMM_REP8(F, 8) PHMM_REP8(F, 0)

template <class T, int C>
struct BandLane {
    typename T::V M[C], D[C];
    typename T::V i_run;      // before the top phase: the I arrival entering this lane's top diagonal; after the rest phase: the one leaving its bottom diagonal
    typename T::V d_out;      // after the top phase: the D arrival this lane's top cell sends to the bottom diagonal of the lane above
    typename T::Ent e, next;  // table entries of the column being processed / prefetched for the next one
    typename T::Col col;
    typename T::V gop, gep, go_prev, ge_prev;
    uint32_t one;             // 1; opaque to the compiler in the kernels, so that the cells' additions are IMADs on the FMA pipe (fma_add)
    bool active;
};

// first_col: the first window column this lane processes (j * C); the penalties of the column before it feed its insertions
template <class T, int C>
PHMM_HD void band_lane_init(BandLane<T, C>& s, const typename T::Tab& tab, const int first_col, const uint32_t one = 1u)
{
    s.one = one;
#pragma unroll
    for (int k = 0; k < C; ++k) { s.M[k] = 0u; s.D[k] = T::inf(); }
    s.i_run = T::inf(); s.d_out = T::inf();
    s.e = T::load(tab, first_col);
    s.go_prev = 0u; s.ge_prev = 0u;
    if (first_col > 0) { const typename T::Col c = T::decode(T::load(tab, first_col - 1)); s.go_prev = c.go; s.ge_prev = c.ge; }
    s.active = false;
}

// Phase 1 of a step: column operands and the top cell (diagonal C-1 of the chunk), which exists from local column C on.
// xl = column relative to the lane's first column, x = xl + first_col the window column, W the window length.
template <class T, int C, bool OGE = false>
PHMM_HD void band_lane_top(BandLane<T, C>& s, const RowEntry* __restrict__ rows, const int L, const int xl, const int x, const int W,
                           const typename T::Tab& tab, const typename T::V nucp, const bool is_top_lane)
{
    s.d_out = T::inf();
    s.active = xl >= 0 && xl <= L + C - 1;
    if (!s.active) return;
    s.next = T::load(tab, x + 1 < W ? x + 1 : W - 1);
    s.col = T::decode(s.e);
    s.gop = s.go_prev + nucp;
    s.gep = s.ge_prev + nucp;
    if (is_top_lane) s.i_run = T::inf();
    if (xl >= C) {
        const RowEntry w = rows[xl - (C - 1)];
        const typename T::V sub = T::sub(w, s.col), m = s.M[C - 1], d = s.D[C - 1];
        const typename T::V sm = T::min3(m, s.i_run, d);
        s.M[C - 1] = fma_add(sm, sub, s.one);
        s.d_out = T::addmin(d, s.col.ge, fma_add(OGE ? sm : T::min2(m, s.i_run), s.col.go, s.one));      // OGE: see dp_pair
        s.i_run = T::addmin(s.i_run, s.gep, fma_add(m, s.gop, s.one));
    }
}

// Phase 2: the remaining cells of the column. d_in = the d_out of the lane below (same step); ignored by the bottom lane.
template <class T, int C, bool OGE = false>
PHMM_HD void band_lane_rest(BandLane<T, C>& s, const RowEntry* __restrict__ rows, const int L, const int xl, const int x,
                            const typename T::V d_in, const bool is_bottom_lane)
{
    if (!s.active) { s.i_run = T::inf(); return; }
    s.D[0] = is_bottom_lane ? T::inf() : d_in;
    const RowEntry* rp = rows + xl;
    const typename T::Col col = s.col;
    const typename T::V gop = s.gop, gep = s.gep;
    const uint32_t one = s.one;
    typename T::V i_run = s.i_run;
#define PHMM_BCELL(k)                                                                          \
    {                                                                                           \
        const RowEntry w = rp[-(k)];                                                            \
        const typename T::V sub = T::sub(w, col);                                               \
        const typename T::V m = s.M[(k) < C ? (k) : 0], d = s.D[(k) < C ? (k) : 0];            \
        const typename T::V sm = T::min3(m, i_run, d);                                          \
        s.M[(k) < C ? (k) : 0] = fma_add(sm, sub, one);                                         \
        if ((k) + 1 < C) s.D[((k) + 1) < C ? (k) + 1 : 0] = T::addmin(d, col.ge, fma_add(OGE ? sm : T::min2(m, i_run), col.go, one)); \
        i_run = T::addmin(i_run, gep, fma_add(m, gop, one));                                    \
    }
#define PHMM_BCASE_PROLOGUE(k) case (k) + 1: if ((k) + 1 < C) PHMM_BCELL(k)
#define PHMM_BCASE_ROW0(k)     case (k): if ((k) < C) s.M[(k) < C ? (k) : 0] = sub0; break;
    if (xl >= C) {
        if (xl <= L) {
#pragma unroll
            for (int k = C - 2; k >= 0; --k) PHMM_BCELL(k)
        } else {
            const int klo = xl - L;              // the row-L cell; klo == C-1 means the top cell was it
#pragma unroll
            for (int k = C - 2; k >= 0; --k) {
                if (k < klo) break;
                PHMM_BCELL(k)
            }
        }
    } else {
        // the free-start cell (x, 0) sits on this chunk's diagonal xl
        const typename T::V sub0 = T::sub(rows[0], col);
        i_run = (x & 1) ? gop : T::inf();
        if (xl <= L) {
            switch (xl) { PHMM_REP32(PHMM_BCASE_PROLOGUE) default: break; }
        } else {
            const int klo = xl - L;
#pragma unroll
            for (int k = C - 2; k >= 0; --k) {
                if (k < xl && k >= klo) PHMM_BCELL(k)
            }
        }
        switch (xl) { PHMM_REP32(PHMM_BCASE_ROW0) default: break; }
    }
#undef PHMM_BCELL
#undef PHMM_BCASE_PROLOGUE
#undef PHMM_BCASE_ROW0
    s.go_prev = col.go; s.ge_prev = col.ge;
    T::pin(s.e, s.next, i_run);
    s.i_run = i_run;
}

template <class T, int C>
PHMM_HD typename T::V band_lane_result(const BandLane<T, C>& s)
{
    typename T::V best = s.M[0];
#pragma unroll
    for (int k = 1; k < C; ++k) best = T::min2(best, s.M[k]);
    return best;
}

#ifdef __CUDACC__
// Device driver. Lanes j = 0..NL-1 of a group are NL consecutive lanes of the warp (group-aligned); every lane of the warp
// must call this with the same L (the loop and its shuffles are warp-wide). Returns the group's result in all of its lanes.
template <class T, int C, int NL, bool OGE = false>
__device__ __forceinline__ typename T::V dp_band(const RowEntry* __restrict__ rows, const int L, const typename T::Tab& tab,
                                                 const typename T::V nucp, const int j, const uint32_t one = 1u)
{
    BandLane<T, C> s;
    const int W = L + NL * C - 1;
    band_lane_init<T, C>(s, tab, j * C, one);
    for (int t = 0; t <= W; ++t) {
        const int x = t - (NL - 1 - j), xl = x - j * C;
        band_lane_top<T, C, OGE>(s, rows, L, xl, x, W, tab, nucp, j == NL - 1);
        typename T::V d_in = T::inf();
        if (NL > 1) d_in = __shfl_up_sync(0xffffffffu, s.d_out, 1);
        band_lane_rest<T, C, OGE>(s, rows, L, xl, x, d_in, j == 0);
        if (NL > 1) { const typename T::V v = __shfl_down_sync(0xffffffffu, s.i_run, 1); s.i_run = (j == NL - 1) ? T::inf() : v; }
    }
    typename T::V best = band_lane_result<T, C>(s);
#pragma unroll
    for (int o = 1; o < NL; o <<= 1) best = T::min2(best, __shfl_xor_sync(0xffffffffu, best, o));
    return best;
}

// The same band with one WARP per chunk ("role") instead of one lane: warp j of a group of NL warps owns chunk j of 32 tasks (one per
// lane), the two hand-overs go through shared memory and a named barrier each. Why: with the chunks in neighbouring lanes, the lane
// that owns the upper diagonals is ~C columns behind the lower one in PHASE (still in its prologue / already in its epilogue while the
// other runs the steady body) and lanes in different column bodies are divergent — the warp runs both bodies one after the other, 70 %
// lane efficiency at L = 150, C = 32, NL = 2. A warp per role has every lane of a warp in the same body, and a role that has nothing to
// do in a step only waits at the barriers, where it costs no issue slot.
//   xchg: shared memory of the group, 3 * NL * 32 words: [0] D hand-over, [1] I hand-over, [2] the roles' partial results.
//   All 32 lanes of all NL warps must call this with the same L (the loop and its barriers are group-wide).
__device__ __forceinline__ void group_barrier(const int id, const int nthreads)
{
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}

template <class T, int C, int NL, bool OGE = false>
__device__ __forceinline__ typename T::V dp_band_roles(const RowEntry* __restrict__ rows, const int L, const typename T::Tab& tab,
                                                       const typename T::V nucp, const int j, const int lane, const uint32_t one,
                                                       typename T::V* xchg, const int barrier_id)
{
    BandLane<T, C> s;
    const int W = L + NL * C - 1;
    band_lane_init<T, C>(s, tab, j * C, one);
    typename T::V* d_slots = xchg + lane;
    typename T::V* i_slots = xchg + NL * 32 + lane;
    typename T::V* r_slots = xchg + 2 * NL * 32 + lane;
    for (int t = 0; t <= W; ++t) {
        const int x = t - (NL - 1 - j), xl = x - j * C;
        band_lane_top<T, C, OGE>(s, rows, L, xl, x, W, tab, nucp, j == NL - 1);
        if (j < NL - 1) d_slots[j * 32] = s.d_out;
        group_barrier(barrier_id, NL * 32);
        const typename T::V d_in = j > 0 ? d_slots[(j - 1) * 32] : T::inf();
        band_lane_rest<T, C, OGE>(s, rows, L, xl, x, d_in, j == 0);
        if (j > 0) i_slots[j * 32] = s.i_run;
        group_barrier(barrier_id, NL * 32);
        s.i_run = j < NL - 1 ? i_slots[(j + 1) * 32] : T::inf();
    }
    // the next call's first write to r_slots is two barriers (at least one whole step) away from the reads below
    typename T::V best = band_lane_result<T, C>(s);
    if (j > 0) r_slots[j * 32] = best;
    group_barrier(barrier_id, NL * 32);
    if (j == 0) {
#pragma unroll
        for (int o = 1; o < NL; ++o) best = T::min2(best, r_slots[o * 32]);
    }
    return best;          // complete in role 0 only
}
#endif

// ---------------------------------------------------------------------------------------------------------
// Flank-aware path: one alignment per thread, 32-bit lanes = score | label | payload, band state in registers
// ---------------------------------------------------------------------------------------------------------
//
// hmm::evaluate needs, for a read within `band` of a haplotype flank, the penalty the OPTIMAL path accrues inside the
// flanks (pair_hmm.hpp:743-764 via simd_pair_hmm.hpp:352-430). In window coordinates the flanks are the truth indices
// < xl and >= xr; the path is monotone in x, so its in-flank penalty is  V(first arrival at column xl) +
// (total - V(first arrival at column xr))  and the in-flank read bases are  y_l + (L - y_r). Instead of storing
// back-pointers, every DP value carries a payload naming the cell through which ITS OWN best path crossed into
// column xl / xr (diagonal k and arrival type M/D); the arrival values of those two columns are kept aside.
// A payload is only meaningful if the DP picks predecessors exactly as the reference's traceback does: the reference
// breaks score ties by state label (M 0 < I 1 < D 3 in the two low bits, simd_pair_hmm.hpp:147-163), so values are
// laid out  [31:18] score  [17:16] label  [15:8] payload R  [7:0] payload L  and compared as whole words — the three
// candidates of every min carry distinct labels, so the payload never takes part in a decision.
constexpr uint32_t kF32ScoreShift = 18;
constexpr uint32_t kF32LabelMask  = 3u << 16;
constexpr uint32_t kF32LabI       = 1u << 16;
constexpr uint32_t kF32LabD       = 3u << 16;
constexpr uint32_t kF32Inf        = 0x3800u << kF32ScoreShift;       // +inf score (14336), leaves room for +2*127+nuc below 2^14
constexpr int      kMaxScoreFlank32 = 0x3800 - 1024;                  // read quality-sum bound for this path
constexpr uint32_t kF32Valid = 0x80u, kF32TypeD = 0x40u;

// Row entries of this kernel (one read, not a pair): .x = PRMT selector picking the cap byte of the read base into byte 0
// and zeros elsewhere (code | 0x5550 — bytes 1..3 of the second operand are zero; code 4 = 'N' picks byte 0 of the second PRMT operand, the column's capN), .y = base quality.
PHMM_HD RowEntry make_row_entry32(uint32_t half) { RowEntry r; r.x = (half & 7u) | 0x5550u; r.y = half >> 8; return r; }
PHMM_HD RowEntry pad_row_entry32() { RowEntry r; r.x = 0x5550u; r.y = 0u; return r; }

// One place where the reference's flank replay does NOT re-add what its DP charged: a mismatch against a truth 'N' inside a flank
// is replayed as exactly 2 (simd_pair_hmm.hpp:388-392) although the DP charged min(q', 2) (update_match_state, :121-142). The
// payload DP below reports what the DP charged, so a candidate whose flanks hold an 'N' column that could have been matched for
// less than 2 — the read has a quality below 2, or the column's SNV prior is below 2 — must take the exact traceback path
// (generic_align<true>) instead. An 'N' column is recognisable from its table entry: all four caps <= 2 (any other column has at
// least two caps of 127). lhs / rhs: flank sizes in window coordinates (window_flanks); overlapping flanks cover every column.
PHMM_HD bool flank_replay_may_differ(const ColEntry* __restrict__ tab, const int W, const int lhs, const int rhs, const bool read_has_quality_below_2)
{
    for (int x = 0; x < W; ++x) {
        if (x >= lhs && x < W - rhs) { x = W - rhs - 1; continue; }      // skip the non-flank middle
        const uint32_t caps = ldg(tab + x).x;
        if ((caps & 0xFCFCFCFCu) == 0u && (read_has_quality_below_2 || caps != 0x02020202u)) return true;
    }
    return false;
}

// The same test from per-haplotype prefix counts (k_ncol_prefix): pre[i] = counts over the haplotype's bases up to and including
// base i — low half: 'N'-like columns (all four caps <= 3) whose caps are not all exactly 2, high half: all 'N'-like columns.
// preh points at the haplotype's first base, a is the window start inside the haplotype. Four loads instead of a loop over the
// flank columns (which a lane of the flank kernels runs with a dependent load per column).
PHMM_HD bool flank_replay_may_differ_pre(const uint32_t* __restrict__ preh, const int a, const int W, const int lhs, const int rhs,
                                         const bool read_has_quality_below_2)
{
    const int l_end = lhs < W ? (lhs > 0 ? lhs : 0) : W;
    int r_beg = W - (rhs > 0 ? rhs : 0);
    if (r_beg < l_end) r_beg = l_end;
    const int i0 = a, i1 = a + l_end, i2 = a + r_beg, i3 = a + W;           // flank columns: [i0, i1) and [i2, i3)
    const uint32_t c = ((i1 > 0 ? ldg(preh + i1 - 1) : 0u) - (i0 > 0 ? ldg(preh + i0 - 1) : 0u)) +
                       ((i3 > 0 ? ldg(preh + i3 - 1) : 0u) - (i2 > 0 ? ldg(preh + i2 - 1) : 0u));
    return (c & 0xFFFFu) != 0u || (read_has_quality_below_2 && (c >> 16) != 0u);
}
PHMM_HD uint32_t ncol_class(const uint32_t caps)   // bit 0: counts for the low half, bit 16: for the high half
{
    if ((caps & 0xFCFCFCFCu) != 0u) return 0u;
    return caps != 0x02020202u ? 0x00010001u : 0x00010000u;
}

// rows: shared-memory row entries (make_row_entry32), rows[L] = pad_row_entry32().
// tab : column table of the window. xl / xr: first non-flank column and first right-flank column (0 <= xl < xr <= W);
// xl == 0 / xr > W mean "no left / right flank". Outputs the integer score, the in-flank penalty and the in-flank read bases.
// Column bodies as in dp_pair: steady / prologue (jump table) / epilogue (early exit after the row-L cell) / general.
template <int BAND>
PHMM_HD void dp_flank32(const RowEntry* __restrict__ rows, const int L, const ColEntry* __restrict__ tab, const int nuc_prior,
                        const int xl, const int xr, int* score_out, int* flank_out, int* mask_out)
{
    constexpr int K = 2 * BAND;
    static_assert(K <= 64, "register band limited to 64 diagonals");
    uint32_t M[K], D[K];
    uint32_t bnd[4][K];          // arrivals at columns xl (M, D) and xr (M, D)
    uint32_t end_s[K];           // S(L + k, L) with label and payload
#pragma unroll
    for (int k = 0; k < K; ++k) { M[k] = 0u; D[k] = kF32Inf | kF32LabD; end_s[k] = 0xFFFFFFFFu; }
    const int W = L + K - 1;
    const uint32_t nucS = (uint32_t)nuc_prior << kF32ScoreShift;
    ColEntry e = ldg(tab);
    uint32_t go_prev = 0u, ge_prev = 0u;
    const RowEntry w0 = rows[0];

#define PHMM_FCELL(k, CAPTURE)                                                                          \
    {                                                                                                   \
        const RowEntry w = rp[-(k)];                                                                    \
        const uint32_t sub = umin32(w.y, prmt(caps, cap_n, w.x));                                       \
        const uint32_t m = M[(k) < K ? (k) : 0], d = D[(k) < K ? (k) : 0];                              \
        const uint32_t mi = umin32(m, i_run);                                                           \
        const uint32_t S = umin32(mi, d);                                                               \
        CAPTURE                                                                                         \
        M[(k) < K ? (k) : 0] = (S & ~kF32LabelMask) + (sub << kF32ScoreShift);                          \
        if ((k) + 1 < K) D[((k) + 1) < K ? (k) + 1 : 0] = umin32(d + geS, mi + goS) | kF32LabD;         \
        i_run = umin32(i_run + gepS, m + gopS) | kF32LabI;                                              \
    }
#define PHMM_FCASE_PROLOGUE(k) case (k) + 1: if ((k) < K) PHMM_FCELL(k, )
#define PHMM_FCASE_ROW0(k)     case (k): if ((k) < K) M[(k) < K ? (k) : 0] = sub0; break;

    for (int x = 0; x <= W; ++x) {
        const int xn = (x + 1 < W) ? x + 1 : W - 1;
        const ColEntry nx = ldg(tab + xn);
        const uint32_t caps = e.x, cap_n = (e.y >> 16) & 0xFFu;
        const uint32_t goS = (e.y & 0xFFu) << kF32ScoreShift, geS = ((e.y >> 8) & 0xFFu) << kF32ScoreShift;
        const uint32_t gopS = go_prev + nucS, gepS = ge_prev + nucS;
        const RowEntry* rp = rows + x;
        uint32_t i_run = kF32Inf | kF32LabI;
        if (x >= K) {
            if (x < L) {
#pragma unroll
                for (int k = K - 1; k >= 0; --k) PHMM_FCELL(k, )
            } else {
                // epilogue: the row-L cell (k == x - L) keeps the labelled S — the end-cell choice compares it with its label
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    PHMM_FCELL(k, if (k == klo) end_s[k] = S;)
                    if (k == klo) break;
                }
            }
        } else {
            const uint32_t sub0 = umin32(w0.y, prmt(caps, cap_n, w0.x)) << kF32ScoreShift;   // m(x+1, 1) = sub(x, 0)
            i_run = (x & 1) ? (gopS | kF32LabI) : (kF32Inf | kF32LabI);                    // i(x, 1) out of the free-start cell
            if (x < L) {
                switch (x) { PHMM_REP64(PHMM_FCASE_PROLOGUE) default: break; }
            } else {
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    if (k < x && k >= klo) PHMM_FCELL(k, if (k == klo) end_s[k] = S;)
                }
            }
            switch (x) { PHMM_REP64(PHMM_FCASE_ROW0) default: break; }
        }
        // the arrivals now held in M[k] / D[k] belong to column x+1: at the two flank boundaries record them and stamp
        // the crossing (diagonal, arrival type) into their payload
        if (x + 1 == xl || x + 1 == xr) {
            const int which = (x + 1 == xl) ? 0 : 2;
            const int shift = (x + 1 == xl) ? 0 : 8;
            const int klo1 = x + 1 - L;             // cells of column x+1 exist for max(0, klo1) <= k <= min(K-1, x)  (row 0 excluded)
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (k >= klo1 && k <= x) {
                    bnd[which][k] = M[k]; bnd[which + 1][k] = D[k];
                    M[k] |= (kF32Valid | (uint32_t)k) << shift;
                    D[k] |= (kF32Valid | kF32TypeD | (uint32_t)k) << shift;
                }
            }
        }
        go_prev = goS; ge_prev = geS;
        // as in dp_pair: keep the prefetched entry out of `e` until the column is done (bit 17 of an I value is always 0)
        const uint32_t z = i_run & (2u << 16);
        e.x = nx.x + z; e.y = nx.y + z;
    }
#undef PHMM_FCELL
#undef PHMM_FCASE_PROLOGUE
#undef PHMM_FCASE_ROW0
    // end row: minimum over (score, label), earliest end on ties (simd_pair_hmm.hpp:285-291, 309-315 compare the labelled values)
    uint32_t best = end_s[0];
    int kbest = 0;
    for (int k = 1; k < K; ++k) if ((end_s[k] >> 16) < (best >> 16)) { best = end_s[k]; kbest = k; }
    const int total = (int)(best >> kF32ScoreShift), x_end = L + kbest;
    const uint32_t pl = best & 0xFFu, pr = (best >> 8) & 0xFFu;
    int v_l, y_l, v_r, y_r;
    if (xl <= 0) { v_l = 0; y_l = 0; }
    else if (pl & kF32Valid) { const int k = pl & 0x3F; v_l = (int)(bnd[(pl & kF32TypeD) ? 1 : 0][k] >> kF32ScoreShift); y_l = xl - k; }
    else if (x_end < xl) { v_l = total; y_l = L; }      // the whole path lies in the left flank
    else { v_l = 0; y_l = 0; }                          // the path starts at or beyond xl
    if (xr > W) { v_r = total; y_r = L; }
    else if (pr & kF32Valid) { const int k = pr & 0x3F; v_r = (int)(bnd[(pr & kF32TypeD) ? 3 : 2][k] >> kF32ScoreShift); y_r = xr - k; }
    else if (x_end >= xr) { v_r = 0; y_r = 0; }         // the path starts inside the right flank
    else { v_r = total; y_r = L; }                      // the path never reaches the right flank
    *score_out = total;
    *flank_out = v_l + (total - v_r);
    *mask_out = y_l + (L - y_r);
}

// ---------------------------------------------------------------------------------------------------------
// Flank-aware path, lean form: the payload is the in-flank penalty itself
// ---------------------------------------------------------------------------------------------------------
//
// dp_flank32 above names the cells where the best path crosses the flank boundaries and looks the arrival values up afterwards;
// it needs the boundary columns kept aside (4 x 2B registers) and measured 9.7 ALU-pipe instructions per cell (profiles/r02a:
// ALU pipe 84 % busy — the kernel is at its formulation's floor). When at least two read bases are certain to lie outside the
// flanks (flank_mask_cannot_zero below: the common case — the non-flank part of the window is wider than the band), the
// reference's result is simply score - (penalty accrued inside the flanks) (pair_hmm.hpp:755-764), and that penalty can ride
// along as an ADDITIVE payload: every transition's constant carries its penalty twice, in the score field and — in flank
// columns only — in the payload field. Values are  [31:16] score  [15:14] label  [13:0] in-flank penalty of this cell's own best
// path; whole-word unsigned comparisons reproduce the reference's choices exactly as in dp_flank32 (labels M 0 < I 1 < D 3).
// Per cell: PRMT + VIMNMX.U16x2 (the emission for both fields at once: the second PRMT operand is the column's cap table, the first
// the same table in flank columns and zero elsewhere), VIMNMX3 (S), LOP3 (clear the label), VIMNMX3 (D': three candidates, adds on the
// FMA pipe), LOP3 (D label), VIADDMNMX (I'), LOP3 (I label; it cannot be folded into the open constant: extension and opening would
// then tie on the label) = 8 ALU-pipe instructions against 9.7, and no boundary arrays (no local memory, 2B fewer live registers).
// Reads must be ACGT-only (four caps per PRMT operand) with a quality sum below kMaxScoreFlank32.
constexpr uint32_t kFAccLabelMask = 3u << 14, kFAccLabI = 1u << 14, kFAccLabD = 3u << 14;
constexpr uint32_t kFAccInf = 0x7000u << 16;

// .x = PRMT selector: byte 0 <- first operand [code] (flank copy), byte 2 <- second operand [code], bytes 1 / 3 <- 0x00 (sign
// replication of a byte < 0x80); .y = quality in both halves
PHMM_HD RowEntry make_row_entry_facc(uint32_t half) { const uint32_t c = half & 3u; RowEntry r; r.x = 0x8480u | c | ((4u + c) << 8); r.y = (half >> 8) | ((half >> 8) << 16); return r; }
PHMM_HD RowEntry pad_row_entry_facc() { RowEntry r; r.x = 0x8480u | (4u << 8); r.y = 0u; return r; }

// True when every path consumes at least two read bases outside the flanks: read base y is consumed at a truth index in
// [y, y + 2B - 1], so the bases with xl <= y and y + 2B - 1 < xr are outside whatever the path. (pair_hmm.hpp:757-759 zeroes the
// flank score otherwise; such candidates keep to dp_flank32.)
PHMM_HD bool flank_mask_cannot_zero(const int L, const int band, const int xl, const int xr)
{
    const int lo = xl > 0 ? xl : 0, hi = (L - 1 < xr - 2 * band) ? L - 1 : xr - 2 * band;
    return hi - lo + 1 >= 2;
}

template <int BAND>
PHMM_HD void dp_flank_acc(const RowEntry* __restrict__ rows, const int L, const ColEntry* __restrict__ tab, const int nuc_prior,
                          const int xl, const int xr, int* score_out, int* flank_out, const uint32_t one = 1u)
{
    constexpr int K = 2 * BAND;
    static_assert(K <= 64, "register band limited to 64 diagonals");
    uint32_t M[K], D[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { M[k] = 0u; D[k] = kFAccInf | kFAccLabD; }
    const int W = L + K - 1;
    ColEntry e = ldg(tab);
    uint32_t go_prev = 0u, ge_prev = 0u;
    const RowEntry w0 = rows[0];
    uint32_t best = 0xFFFFFFFFu;

#define PHMM_ACELL(k, CAPTURE)                                                                          \
    {                                                                                                   \
        const RowEntry w = rp[-(k)];                                                                    \
        const uint32_t subw = vminu2(w.y, prmt(caps_lo, caps_hi, w.x));                                 \
        const uint32_t m = M[(k) < K ? (k) : 0], d = D[(k) < K ? (k) : 0];                              \
        const uint32_t S = umin3_32(m, i_run, d);                                                       \
        CAPTURE                                                                                         \
        M[(k) < K ? (k) : 0] = fma_add(S & ~kFAccLabelMask, subw, one);                                 \
        if ((k) + 1 < K) D[((k) + 1) < K ? (k) + 1 : 0] = umin3_32(fma_add(d, geS, one), fma_add(m, goS, one), fma_add(i_run, goS, one)) | kFAccLabD; \
        i_run = uaddmin32(i_run, gepS, fma_add(m, gopS, one)) | kFAccLabI;                              \
    }
#define PHMM_ACASE_PROLOGUE(k) case (k) + 1: if ((k) < K) PHMM_ACELL(k, )
#define PHMM_ACASE_ROW0(k)     case (k): if ((k) < K) M[(k) < K ? (k) : 0] = sub0; break;
// the row-L cell: minimum over (score, label), earliest end on ties (simd_pair_hmm.hpp:285-291, 309-315)
#define PHMM_ACAPTURE(k) if (k == klo && (S >> 14) < (best >> 14)) best = S;

    for (int x = 0; x <= W; ++x) {
        const int xn = (x + 1 < W) ? x + 1 : W - 1;
        const ColEntry nx = ldg(tab + xn);
        const uint32_t fl = (x < xl || x >= xr) ? 1u : 0u;         // the penalties of this column's three transitions count as in-flank
        const uint32_t both = 0x10000u + fl;
        const uint32_t caps_hi = e.x, caps_lo = fl ? e.x : 0u;
        const uint32_t go = e.y & 0xFFu, ge = (e.y >> 8) & 0xFFu;
        const uint32_t goS = go * both, geS = ge * both;
        const uint32_t gopS = (go_prev + (uint32_t)nuc_prior) * both, gepS = (ge_prev + (uint32_t)nuc_prior) * both;
        const RowEntry* rp = rows + x;
        uint32_t i_run = kFAccInf | kFAccLabI;
        if (x >= K) {
            if (x < L) {
#pragma unroll
                for (int k = K - 1; k >= 0; --k) PHMM_ACELL(k, )
            } else {
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    PHMM_ACELL(k, PHMM_ACAPTURE(k))
                    if (k == klo) break;
                }
            }
        } else {
            const uint32_t sub0 = vminu2(w0.y, prmt(caps_lo, caps_hi, w0.x));      // the path starts here: m(x+1, 1) = sub(x, 0), in-flank or not
            i_run = (x & 1) ? (gopS | kFAccLabI) : (kFAccInf | kFAccLabI);
            if (x < L) {
                switch (x) { PHMM_REP64(PHMM_ACASE_PROLOGUE) default: break; }
            } else {
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    if (k < x && k >= klo) PHMM_ACELL(k, PHMM_ACAPTURE(k))
                }
            }
            switch (x) { PHMM_REP64(PHMM_ACASE_ROW0) default: break; }
        }
        go_prev = go; ge_prev = ge;
        const uint32_t z = i_run & 0x8000u;        // bit 15 of an I value is never set (label 1): pins the prefetch behind the column
        e.x = nx.x + z; e.y = nx.y + z;
    }
#undef PHMM_ACELL
#undef PHMM_ACASE_PROLOGUE
#undef PHMM_ACASE_ROW0
#undef PHMM_ACAPTURE
    *score_out = (int)(best >> 16);
    *flank_out = (int)(best & 0x3FFFu);
}

// ---------------------------------------------------------------------------------------------------------
// Flank-aware path, packed: forward pass up to a flank boundary + backward pass down to it (dp_flank_fb)
// ---------------------------------------------------------------------------------------------------------
//
// dp_flank32 / dp_flank_acc above reproduce the reference's traceback decisions with labelled 32-bit values — one alignment per
// thread, ~14 instructions per cell, 0.36 of the score-only kernel (DESIGN.md). What hmm::evaluate needs from the traceback
// (pair_hmm.hpp:743-764, replay simd_pair_hmm.hpp:352-430) is only WHERE the chosen path crosses the two flank boundaries: the path is
// monotone in x, so its in-flank penalty is  V(first arrival at column xl) + total - V(first arrival at column xr)  and its
// in-flank read bases are  y_l + L - y_r. The forward value F of a cell does not depend on the path chosen after it, and the
// cost-to-go B of a cell (the same recurrence run from the end row backwards) does not depend on the path before it; every optimal
// path crosses column xb at a cell where F + B equals the total score. So: the plain packed forward DP (dp_pair's cell, two
// alignments per thread, no labels) over the columns BEFORE the boundary, a packed backward DP over the columns FROM the window end
// down to the boundary, and the crossing cell is the argmin of F + B in that column — each column of the window is swept about
// once, at the packed kernels' cost per cell.
// The reference breaks score ties by state label (simd_pair_hmm.hpp:147-163); F + B cannot see which of several co-optimal paths its
// traceback would follow. When the minimisers of a boundary column disagree on (arrival value, read row) — the only things the
// discount depends on — the candidate is reported as `tie` and the kernel hands it to the exact labelled DP (dp_flank32) instead;
// when they agree, every co-optimal path gives the same discount and so does the reference's (~1-2 % of random candidates tie).
//
// Backward recurrence (cost-to-go by arrival state; transitions as in the header comment of this file; go/ge = column x,
// gop/gep = column x-1 plus nuc_prior):
//   A     = sub(x, y) + Bm(x+1, y+1)
//   Bd    = min(A, ge + Bd(x+1, y))                        a deletion can only be extended or left by a match
//   t     = min(A, go + Bd(x+1, y))                        M and I may open a deletion (I -> D allowed)
//   Bm    = min(t, gop + Bi(x, y+1))                       only M opens an insertion ...
//   Bi    = min(t, gep + Bi(x, y+1))                       ... I extends it (no D -> I)
//   B(x, L) = 0 in every state (free end);  start cell (x, 0): total = min(A, x odd ? gop + Bi(x, 1) : inf)  (the initialiser quirk)
// Per cell pair: PRMT, VIMNMX (sub), VIADDMNMX (Bd), 2 VIMNMX3 (Bm, Bi) on the ALU pipe and 4 additions as IMADs on the FMA pipe
// (5 + 4, as the forward cell's 5 + 3) — the band sweeps columns downwards and diagonals upwards, so that Bm stays in place, Bd moves
// one diagonal down and the insertion chain runs through one register.
//
// Boundaries: b[0], b[1] = xl, xr of the low half's alignment, b[2], b[3] of the high half's; a boundary is a window column in
// [1, W-1], anything else (0, negative, >= W) means "no such flank". At each boundary column the forward arrivals (M, D) and the
// backward values (Bm, Bd) of the whole band go to scratch (word ((slot * 2 + array) * 2B + k) * stride of the pass's own
// scratch), and fb_decide reads them back. Requires L >= 2B (the kernels route shorter reads to dp_flank32), ACGT reads,
// 16-bit-safe quality sums. The two passes are separate functions — and separate kernels (k_flank_fwd, k_flank_bwd): fused
// into one kernel their unrolled column bodies (6 x ~5 KB of code + jump tables, ~80 KB) overflow the SM's 32 KB instruction
// cache as soon as the resident warps are in different phases, and the kernel spends 11 stall cycles per issued instruction
// waiting for instructions (profiles/r02n_flankfb16_fused_ncu_raw.csv: issue slots 26 % used).
#define PHMM_REP8A(F, b)  F(b + 0) F(b + 1) F(b + 2) F(b + 3) F(b + 4) F(b + 5) F(b + 6) F(b + 7)
#define PHMM_REP64A(F)    PHMM_REP8A(F, 0) PHMM_REP8A(F, 8) PHMM_REP8A(F, 16) PHMM_REP8A(F, 24) PHMM_REP8A(F, 32) PHMM_REP8A(F, 40) PHMM_REP8A(F, 48) PHMM_REP8A(F, 56)

constexpr int kFbSlots = 4;            // boundary slots of a lane's two alignments: xl / xr of the low half, xl / xr of the high half
PHMM_HD size_t fb_scratch_words(const int band) { return (size_t)kFbSlots * 2 * 2 * (size_t)band; }     // per pass: slots x {M, D} x 2B diagonals
PHMM_HD bool fb_boundary_valid(const int b, const int W) { return b >= 1 && b <= W - 1; }

struct FbResult { int score, flank, mask, tie; };
// The four boundary columns of a lane's two alignments, two per word (16 bits each, 0 = no such boundary: a valid column is >= 1) —
// the passes keep them in two registers next to the band. The forward pass covers the columns [0, fb_fwd_end), the backward pass
// [fb_bwd_end, W].
struct FbBounds { uint32_t lo, hi; };          // lo = xl | xr << 16 of the low half's alignment, hi = of the high half's
PHMM_HD FbBounds fb_bounds(const int b0, const int b1, const int b2, const int b3, const int W)
{
    FbBounds g;
    g.lo = (fb_boundary_valid(b0, W) ? (uint32_t)b0 : 0u) | ((fb_boundary_valid(b1, W) ? (uint32_t)b1 : 0u) << 16);
    g.hi = (fb_boundary_valid(b2, W) ? (uint32_t)b2 : 0u) | ((fb_boundary_valid(b3, W) ? (uint32_t)b3 : 0u) << 16);
    return g;
}
PHMM_HD int fb_slot_column(const FbBounds& g, const int s) { const uint32_t w = s < 2 ? g.lo : g.hi; return (int)((s & 1) ? w >> 16 : w & 0xFFFFu); }
PHMM_HD int fb_fwd_end(const FbBounds& g)      // 0: nothing to do
{
    int e = fb_slot_column(g, 0);
#pragma unroll
    for (int s = 1; s < 4; ++s) { const int c = fb_slot_column(g, s); e = c > e ? c : e; }
    return e;
}
PHMM_HD int fb_bwd_end(const FbBounds& g)      // 0x7fffffff: nothing to do
{
    int e = 0x7fffffff;
#pragma unroll
    for (int s = 0; s < 4; ++s) { const int c = fb_slot_column(g, s); if (c > 0 && c < e) e = c; }
    return e;
}
// the next boundary column above / below v (0x7fffffff / 0: none)
PHMM_HD int fb_next_above(const FbBounds& g, const int v)
{
    int n = 0x7fffffff;
#pragma unroll
    for (int s = 0; s < 4; ++s) { const int c = fb_slot_column(g, s); if (c > v && c < n) n = c; }
    return n;
}
PHMM_HD int fb_next_below(const FbBounds& g, const int v)
{
    int n = 0;
#pragma unroll
    for (int s = 0; s < 4; ++s) { const int c = fb_slot_column(g, s); if (c < v && c > n) n = c; }
    return n;
}
// Slots that name the same column share one copy of the band (the packed words hold both halves anyway): the representative of
// slot s is the first slot with its column — the usual case is ONE stored column for a lane's two alignments.
PHMM_HD int fb_slot_rep(const FbBounds& g, const int s)
{
    const int c = fb_slot_column(g, s);
    if (s >= 1 && fb_slot_column(g, 0) == c) return 0;
    if (s >= 2 && fb_slot_column(g, 1) == c) return 1;
    if (s >= 3 && fb_slot_column(g, 2) == c) return 2;
    return s;
}

template <int K>
PHMM_HD void fb_store(uint32_t* __restrict__ dst, const size_t stride, const uint32_t (&a0)[K], const uint32_t (&a1)[K])
{
#pragma unroll
    for (int k = 0; k < K; ++k) { dst[(size_t)k * stride] = a0[k]; dst[(size_t)(K + k) * stride] = a1[k]; }
}
// the band's two arrays of a boundary column → scratch, once per slot whose boundary this column is (rolled over the slots)
#define PHMM_FB_STORE(A0, A1)                                                                           \
    {                                                                                                   \
        _Pragma("unroll 1") for (int s_ = 0; s_ < kFbSlots; ++s_)                                       \
            if (fb_slot_column(g, s_) == next && fb_slot_rep(g, s_) == s_) fb_store<K>(scr_fn() + (size_t)(s_ * 2) * K * stride, stride, A0, A1); \
    }
#define PHMM_FB_NEXT_ABOVE(v) { next = fb_next_above(g, (v)); }
#define PHMM_FB_NEXT_BELOW(v) { next = fb_next_below(g, (v)); }

// Forward pass: dp_pair's column sweep over [0, fe); at every boundary column the arrivals (M, D) of the band go to
// scr[((slot * 2 + {0, 1}) * 2B + k) * stride].
// scr_fn() returns the scratch pointer; it is called at the boundary columns only, so that a pointer the caller can re-derive from
// its indices does not occupy two registers through the sweep.
template <int BAND, bool OGE, class ScrFn>
PHMM_HD void dp_flank_fwd(const RowEntry* __restrict__ rows, const int L, const ColEntry* __restrict__ t0, const ColEntry* __restrict__ t1,
                          const uint32_t nucp, const FbBounds g, ScrFn scr_fn, const size_t stride, const uint32_t one = 1u)
{
    constexpr int K = 2 * BAND;
    static_assert(K <= 64, "register band limited to 64 diagonals");
    const int W = L + K - 1;
    const int fe = fb_fwd_end(g);
    if (fe <= 0) return;
    uint32_t M[K], D[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { M[k] = 0u; D[k] = kInf16x2; }
    ColEntry e0 = ldg(t0), e1 = ldg(t1);
    uint32_t go_prev = 0u, ge_prev = 0u;
    int next;
    PHMM_FB_NEXT_ABOVE(0)
#define PHMM_CELL(k)                                                                        \
    {                                                                                       \
        const RowEntry w   = rp[-(k)];                                                      \
        const uint32_t sub = vmin2(w.y, prmt(caps0, caps1, w.x));                           \
        const uint32_t m = M[(k) < K ? (k) : 0], d = D[(k) < K ? (k) : 0];                  \
        const uint32_t s = vmin3(m, i_run, d);                                              \
        M[(k) < K ? (k) : 0] = fma_add(s, sub, one);                                        \
        if ((k) + 1 < K) D[((k) + 1) < K ? (k) + 1 : 0] = vaddmin(d, ge, fma_add(OGE ? s : vmin2(m, i_run), go, one)); \
        i_run = vaddmin(i_run, gep, fma_add(m, gop, one));                                  \
    }
#define PHMM_CASE_PROLOGUE(k) case (k) + 1: if ((k) < K) PHMM_CELL(k)
#define PHMM_CASE_ROW0(k)     case (k): if ((k) < K) M[(k) < K ? (k) : 0] = sub0; break;
    for (int x = 0; x < fe; ++x) {
        const int xn = (x + 1 < W) ? x + 1 : W - 1;
        const ColEntry n0 = ldg(t0 + xn), n1 = ldg(t1 + xn);
        const uint32_t caps0 = e0.x, caps1 = e1.x;
        const uint32_t go = prmt(e0.y, e1.y, 0x3430u), ge = prmt(e0.y, e1.y, 0x3531u);
        const uint32_t gop = go_prev + nucp, gep = ge_prev + nucp;
        const RowEntry* rp = rows + x;
        uint32_t i_run = kInf16x2;
        if (x >= K) {
            if (x <= L) {
#pragma unroll
                for (int k = K - 1; k >= 0; --k) PHMM_CELL(k)
            } else {
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    PHMM_CELL(k)
                    if (k == klo) break;
                }
            }
        } else {
            const RowEntry w0 = rows[0];     // (loaded here, not kept in registers through the steady columns)
            const uint32_t sub0 = vmin2(w0.y, prmt(caps0, caps1, w0.x));
            i_run = (x & 1) ? gop : kInf16x2;
            switch (x) { PHMM_REP64(PHMM_CASE_PROLOGUE) default: break; }
            switch (x) { PHMM_REP64(PHMM_CASE_ROW0) default: break; }
        }
        go_prev = go; ge_prev = ge;
        if (x + 1 == next) {                 // M / D now hold the arrivals of column x + 1: a flank boundary of one of the halves
            PHMM_FB_STORE(M, D)
            PHMM_FB_NEXT_ABOVE(x + 1)
        }
        const uint32_t z = i_run & 0x80008000u;          // see dp_pair: keeps the prefetch out of e0 / e1 until the column is done
        e0.x = n0.x + z; e0.y = n0.y + z; e1.x = n1.x + z; e1.y = n1.y + z;
    }
#undef PHMM_CELL
#undef PHMM_CASE_PROLOGUE
#undef PHMM_CASE_ROW0
}

// Backward pass: cost-to-go over [be, W], columns downwards, diagonals upwards; at every boundary column (Bm, Bd) of the band go
// to scr[((slot * 2 + {0, 1}) * 2B + k) * stride]. Independent of the deletion-update form (OGE).
// The end row needs no special column body: rows[L .. L + 2B - 1] are pad entries (emission 0) and the band starts at 0, so every
// "cell" on or below row L computes cost-to-go 0 in all three states from zeros (a = 0 + 0, Bd = min(0 + ge, 0), Bm = Bi =
// min3(0, ..)) — exactly B(x, L) = 0, and the cells above it see the free end. The columns x >= L therefore run the plain steady
// body (their sub-row cells are wasted work, about as much as the jump-table body they replace cost in extra instructions — but 1 000
// instructions less code for the instruction cache). Band entries k > x keep the start cells' totals, entries k < x - L stay 0.
template <int BAND, class ScrFn>
PHMM_HD void dp_flank_bwd(const RowEntry* __restrict__ rows /* rows[0 .. L-1] real, rows[L .. L + 2*BAND - 1] pad */, const int L,
                          const ColEntry* __restrict__ t0, const ColEntry* __restrict__ t1,
                          const uint32_t nucp, const FbBounds g, ScrFn scr_fn, const size_t stride, const uint32_t one = 1u)
{
    constexpr int K = 2 * BAND;
    static_assert(K <= 64, "register band limited to 64 diagonals");
    const int W = L + K - 1;
    const int be = fb_bwd_end(g);
    if (be == 0x7fffffff) return;
    uint32_t BM[K], BD[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { BM[k] = 0u; BD[k] = 0u; }
    // Column operands, held as in the forward pass (6 registers + 4 loads in flight): caps / go / ge of column x, the penalty words of
    // column x - 1 (they make this column's insertion penalties and the next column's go / ge); each column issues the loads of the
    // next column's caps (column x - 1) and of the penalty words after it (column x - 2).
    uint32_t py0 = ldg(&t0[W - 1].y), py1 = ldg(&t1[W - 1].y);
    uint32_t caps0 = 0u, caps1 = 0u, go = 0u, ge = 0u;             // column x (column W: sub-row cells only, any penalties do)
    int next;
    PHMM_FB_NEXT_BELOW(W)
#define PHMM_BKCELL(k)                                                                      \
    {                                                                                       \
        const RowEntry w   = rp[-(k)];                                                      \
        const uint32_t sub = vmin2(w.y, prmt(caps0, caps1, w.x));                           \
        const uint32_t a   = fma_add(BM[(k) < K ? (k) : 0], sub, one);                      \
        const uint32_t dd  = ((k) + 1 < K) ? BD[((k) + 1) < K ? (k) + 1 : 0] : kInf16x2;    \
        BD[(k) < K ? (k) : 0] = vaddmin(dd, ge, a);                                         \
        const uint32_t od  = fma_add(dd, go, one);        /* open a deletion */             \
        BM[(k) < K ? (k) : 0] = vmin3(a, od, fma_add(i_run, gop, one));                     \
        i_run = vmin3(a, od, fma_add(i_run, gep, one));                                     \
    }
#define PHMM_BCASE_START(k) case (k): if ((k) < K) { const uint32_t a = fma_add(BM[(k) < K ? (k) : 0], sub0, one); BM[(k) < K ? (k) : 0] = (x & 1) ? vaddmin(i_run, gop, a) : a; } break;
    for (int x = W; x >= be; --x) {
        const int x1 = x >= 1 ? x - 1 : 0, x2 = x >= 2 ? x - 2 : 0;
        const uint32_t nx0 = ldg(&t0[x1].x), nx1 = ldg(&t1[x1].x), ny0 = ldg(&t0[x2].y), ny1 = ldg(&t1[x2].y);
        const uint32_t gop = prmt(py0, py1, 0x3430u) + nucp, gep = prmt(py0, py1, 0x3531u) + nucp;      // column x - 1
        const RowEntry* rp = rows + x;
        uint32_t i_run = kInf16x2;           // nothing below diagonal 0
        if (x >= K) {
#pragma unroll
            for (int k = 0; k < K; ++k) PHMM_BKCELL(k)
        } else {
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (k == x) break;
                PHMM_BKCELL(k)
            }
            const RowEntry w0 = rows[0];
            const uint32_t sub0 = vmin2(w0.y, prmt(caps0, caps1, w0.x));       // the start cell (x, 0): its total stays in BM[x]
            switch (x) { PHMM_REP64A(PHMM_BCASE_START) default: break; }
        }
        if (x == next) {
            PHMM_FB_STORE(BM, BD)
            PHMM_FB_NEXT_BELOW(x)
        }
        const uint32_t z = i_run & 0x80008000u;          // see dp_pair: keeps the prefetched words out of the live registers until the column is done
        caps0 = nx0 + z; caps1 = nx1 + z; go = gop - nucp; ge = gep - nucp;
        py0 = ny0 + z; py1 = ny1 + z;
    }
#undef PHMM_BKCELL
#undef PHMM_BCASE_START
}
#undef PHMM_FB_NEXT_ABOVE
#undef PHMM_FB_NEXT_BELOW
#undef PHMM_FB_STORE

// One boundary column, both halves of the packed words at once. The candidates of a half are, for every diagonal k, the arrival by M
// and by D at cell (xb, y = xb - k): total F + B, in-flank value F, read row y. The band arrays make the three kinds of diagonal
// uniform (no case distinction here):
//   k < xb - L   the path ended before the column: the forward pass left S(L + k, L) in M[k] (and d(L + k, L) >= it in D[k]), the
//                backward band is 0 there; y clamps to L
//   k >= xb      the path starts at or beyond the column: forward M[k] is still 0 and D[k] +inf, the backward pass left the start
//                cell's total in Bm[k]; y clamps to 0
//   otherwise    a cell of the column.
// Two sweeps over the 2B diagonals: the packed minimum T of all totals, then — over the candidates whose total equals T — the packed
// minimum and maximum of their F values and rows: the minimisers agree on (F, y) iff min == max for both. fscr / bscr: the slot's
// forward / backward arrays ({M, D} / {Bm, Bd}, K words each; written earlier by this very thread or by the forward kernel: no
// __restrict__, the loads must stay coherent). xb0 / xb1: the column as the low / high half sees it (<= 0: that half is not asked
// for; its lanes then hold another column's data and its result is ignored).
struct FbPick { int T, v, y, tie; };
PHMM_HD uint32_t fb_rows_of(const int xb0, const int xb1, const int k, const int L)
{
    int y0 = xb0 - k, y1 = xb1 - k;
    y0 = y0 < 0 ? 0 : (y0 > L ? L : y0);
    y1 = y1 < 0 ? 0 : (y1 > L ? L : y1);
    return (uint32_t)y0 | ((uint32_t)y1 << 16);
}
PHMM_HD void fb_decide(const uint32_t* fscr, const size_t fstride, const uint32_t* bscr, const size_t bstride, const int K,
                       const int xb0, const int xb1, const int L, FbPick* out0, FbPick* out1)
{
    uint32_t T = 0xFFFFFFFFu;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
        const uint32_t tm = fscr[(size_t)k * fstride] + bscr[(size_t)k * bstride];                  // < 0xE200 per half: no carry
        const uint32_t td = fscr[(size_t)(K + k) * fstride] + bscr[(size_t)(K + k) * bstride];
        T = vminu2(T, vminu2(tm, td));
    }
    const uint32_t ones = 0x00010001u;
    uint32_t v_lo = 0xFFFFFFFFu, v_hi = 0u, y_lo = 0xFFFFFFFFu, y_hi = 0u;
#pragma unroll 2
    for (int k = 0; k < K; ++k) {
        const uint32_t fm = fscr[(size_t)k * fstride], fd = fscr[(size_t)(K + k) * fstride];
        const uint32_t tm = fm + bscr[(size_t)k * bstride], td = fd + bscr[(size_t)(K + k) * bstride];
        const uint32_t nm = vminu2(tm - T, ones), nd = vminu2(td - T, ones);     // per half: 0 = this candidate attains T, 1 = it does not
        const uint32_t km = 0xFFFFFFFFu - nm * 0xFFFFu, kd = 0xFFFFFFFFu - nd * 0xFFFFu;            // per half: 0xFFFF / 0
        v_lo = vminu2(v_lo, vminu2(fm + nm * 0x8000u, fd + nd * 0x8000u));      // F < 0x7200: a non-minimiser moves beyond every real value
        v_hi = vmaxu2(v_hi, vmaxu2(fm & km, fd & kd));
        const uint32_t yk = fb_rows_of(xb0, xb1, k, L), nk = vminu2(nm, nd);    // the row is shared by the diagonal's two candidates
        y_lo = vminu2(y_lo, yk + nk * 0x8000u);
        y_hi = vmaxu2(y_hi, yk & (0xFFFFFFFFu - nk * 0xFFFFu));
    }
    out0->T = (int)(T & 0xFFFFu); out0->v = (int)(v_lo & 0xFFFFu); out0->y = (int)(y_lo & 0xFFFFu);
    out0->tie = ((v_lo ^ v_hi) & 0xFFFFu) != 0u || ((y_lo ^ y_hi) & 0xFFFFu) != 0u;
    out1->T = (int)(T >> 16); out1->v = (int)(v_lo >> 16); out1->y = (int)(y_lo >> 16);
    out1->tie = ((v_lo ^ v_hi) >> 16) != 0u || ((y_lo ^ y_hi) >> 16) != 0u;
}

// The crossing cells of both halves from the two passes' boundary columns → score, in-flank penalty, in-flank read bases, tie.
// Up to four sweeps (side x half; one per side when the halves share the column), rolled so that fb_decide exists once in the code.
PHMM_HD void fb_finish(const int K, const int L, const FbBounds& g, const uint32_t* fscr, const size_t fstride,
                       const uint32_t* bscr, const size_t bstride, FbResult* res0, FbResult* res1)
{
    FbPick l0 {0, 0, 0, 0}, l1 {0, 0, 0, 0}, r0 {0, 0, L, 0}, r1 {0, 0, L, 0};      // [side][half]: "no such flank" defaults
#pragma unroll 1
    for (int job = 0; job < 4; ++job) {
        const int side = job >> 1, second = job & 1;
        const int xa = fb_slot_column(g, side), xb = fb_slot_column(g, 2 + side);      // this side's column of the low / high half
        const int ra = fb_slot_rep(g, side), rb = fb_slot_rep(g, 2 + side);
        const bool shared = xa > 0 && xb > 0 && ra == rb;
        int rep, q0, q1;
        if (!second) { if (xa <= 0) continue; rep = ra; q0 = xa; q1 = shared ? xb : -1; }
        else { if (xb <= 0 || shared) continue; rep = rb; q0 = -1; q1 = xb; }
        FbPick o0, o1;
        fb_decide(fscr + (size_t)(rep * 2) * K * fstride, fstride, bscr + (size_t)(rep * 2) * K * bstride, bstride, K, q0, q1, L, &o0, &o1);
        if (q0 > 0) { if (side) r0 = o0; else l0 = o0; }
        if (q1 > 0) { if (side) r1 = o1; else l1 = o1; }
    }
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int xl = fb_slot_column(g, 2 * half), xr = fb_slot_column(g, 2 * half + 1);
        const FbPick l = half ? l1 : l0, r = half ? r1 : r0;
        const int T = xr > 0 ? r.T : l.T;
        const int v_r = xr > 0 ? r.v : T;          // no right flank inside the window: nothing beyond xr to discount
        FbResult o;
        o.score = T;
        o.flank = l.v + (T - v_r);
        o.mask = l.y + (L - r.y);
        o.tie = l.tie | r.tie | ((xl > 0 && xr > 0 && l.T != r.T) ? 1 : 0);
        if (half) *res1 = o; else *res0 = o;
    }
}

// Both passes and the decision in one call (tests/cpu_emul; the kernels run the passes in two launches: k_flank_fwd / k_flank_bwd).
template <int BAND, bool OGE>
PHMM_HD void dp_flank_fb(const RowEntry* __restrict__ rows, const int L, const ColEntry* __restrict__ t0, const ColEntry* __restrict__ t1,
                         const uint32_t nucp, const int b0, const int b1, const int b2, const int b3,
                         uint32_t* fscr, const size_t fstride, uint32_t* bscr, const size_t bstride, FbResult* res0, FbResult* res1, const uint32_t one = 1u)
{
    const FbBounds g = fb_bounds(b0, b1, b2, b3, L + 2 * BAND - 1);
    dp_flank_fwd<BAND, OGE>(rows, L, t0, t1, nucp, g, [=]() { return fscr; }, fstride, one);
    dp_flank_bwd<BAND>(rows, L, t0, t1, nucp, g, [=]() { return bscr; }, bstride, one);
    fb_finish(2 * BAND, L, g, fscr, fstride, bscr, bstride, res0, res1);
}

// ---------------------------------------------------------------------------------------------------------
// Traceback in registers: HaplotypeLikelihoodModel::align / hmm::align need the alignment itself (CIGAR, first_pos)
// ---------------------------------------------------------------------------------------------------------
//
// Round 1 served these through generic_align<true>: row sweep with the band in LOCAL memory and one read-modify-written back-pointer
// byte per cell in global memory (~64 GCUPS). Here the forward pass is the same register-resident column sweep as dp_flank_acc, on
// labelled values  [31:16] score  [15:14] label (M 0 < I 1 < D 3, compared as whole words: the reference's tie-breaks,
// simd_pair_hmm.hpp:147-163)  [13:0] zero, and every cell writes ONE word holding the three labels a backward walk can ask for:
//   byte 0 = label of S(x, y) << 6          who the match leaving this cell continues (state M at (x+1, y+1) asks its source cell)
//   byte 1 = label picked for D(x+1, y) << 6    (3: extension of a deletion, 0 / 1: opened from M / I)
//   byte 2 = label picked for I(x, y+1) << 6    (1: extension, 0: opened from M)
// (the low 14 bits of every value are zero, so byte 1 of a value IS its label << 6: two PRMTs build the word). Cell (x, k) of a
// thread lives at bp[(x * 2B + k) * bps]; bps = number of threads sharing the scratch (coalesced stores). The walk is
// set_alignments + calculate_flank_score fused, as in generic_align (simd_pair_hmm.hpp:165-231, 352-430).
constexpr uint32_t kTbLabelMask = 3u << 14, kTbLabI = 1u << 14, kTbLabD = 3u << 14;
constexpr uint32_t kTbInf = 0x7000u << 16;
constexpr int kMaxScoreTb = 0x7000 - 1024;       // quality-sum bound of this path (16-bit score field)

// .x = PRMT selector: byte 2 <- cap of the read base (codes 0..3: first operand = the column's four caps; 4 = 'N': byte 0 of the second
// operand), other bytes <- 0 (bytes 1..3 of the second operand); .y = quality << 16
PHMM_HD RowEntry make_row_entry_tb(uint32_t half) { RowEntry r; r.x = 0x5055u | ((half & 7u) << 8); r.y = (half >> 8) << 16; return r; }
PHMM_HD RowEntry pad_row_entry_tb() { RowEntry r; r.x = 0x5055u; r.y = 0u; return r; }

// Row entries of the traceback kernel come as 8-byte RowEntry (tests), packed in 4 bytes (quality << 16 | code << 8) or as the read's
// 2-byte row half-words (TbRows2, what the kernel uses: it stages one read PER THREAD in shared memory, so the footprint decides the
// occupancy) and are decoded at the use.
struct TbRows8 { const RowEntry* p; PHMM_HD RowEntry at(const int i) const { return p[i]; } PHMM_HD TbRows8 shifted(const int x) const { return TbRows8 {p + x}; } };
struct TbRows4
{
    const uint32_t* p;
    PHMM_HD RowEntry at(const int i) const { const uint32_t w = p[i]; RowEntry r; r.x = 0x5055u | (w & 0x700u); r.y = w & 0xFFFF0000u; return r; }
    PHMM_HD TbRows4 shifted(const int x) const { return TbRows4 {p + x}; }
    static PHMM_HD uint32_t pack(const uint32_t half) { return ((half >> 8) << 16) | ((half & 7u) << 8); }     // from the read's row half-word (code | qual << 8)
};

// the read's row half-words themselves (code | qual << 8), 2 bytes per read base: 302 B per 150 bp read and thread
struct TbRows2
{
    const uint16_t* p;
    PHMM_HD RowEntry at(const int i) const { const uint32_t t = (uint32_t)p[i] << 8; RowEntry r; r.x = 0x5055u | (t & 0x700u); r.y = t & 0xFFFF0000u; return r; }
    PHMM_HD TbRows2 shifted(const int x) const { return TbRows2 {p + x}; }
};

template <int BAND, class RowsT>
PHMM_HD void dp_traceback_forward(const RowsT rows, const int L, const ColEntry* __restrict__ tab, const int nuc_prior,
                                  uint32_t* __restrict__ bp, const size_t bps, int* score_out, int* x_end_out, int* state_out)
{
    constexpr int K = 2 * BAND;
    static_assert(K <= 64, "register band limited to 64 diagonals");
    uint32_t M[K], D[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { M[k] = 0u; D[k] = kTbInf | kTbLabD; }
    const int W = L + K - 1;
    ColEntry e = ldg(tab);
    uint32_t go_prev = 0u, ge_prev = 0u;
    const RowEntry w0 = rows.at(0);
    uint32_t best = 0xFFFFFFFFu;
    int x_end = -1;

#define PHMM_TCELL(k, CAPTURE)                                                                          \
    {                                                                                                   \
        const RowEntry w = rp.at(-(k));                                                                    \
        const uint32_t subw = umin32(w.y, prmt(caps, cap_n, w.x));                                      \
        const uint32_t m = M[(k) < K ? (k) : 0], d = D[(k) < K ? (k) : 0];                              \
        const uint32_t S = umin3_32(m, i_run, d);                                                       \
        CAPTURE                                                                                         \
        M[(k) < K ? (k) : 0] = (S & ~kTbLabelMask) + subw;                                              \
        const uint32_t Draw = umin3_32(d + geS, m + goS, i_run + goS);                                  \
        if ((k) + 1 < K) D[((k) + 1) < K ? (k) + 1 : 0] = Draw | kTbLabD;                               \
        const uint32_t Iraw = uaddmin32(i_run, gepS, m + gopS);                                         \
        i_run = Iraw | kTbLabI;                                                                         \
        bcol[(size_t)((k) < K ? (k) : 0) * bps] = prmt(prmt(S, Draw, 0x1151u), Iraw, 0x4510u);          \
    }
#define PHMM_TCASE_PROLOGUE(k) case (k) + 1: if ((k) < K) PHMM_TCELL(k, )
#define PHMM_TCASE_ROW0(k)     case (k): if ((k) < K) M[(k) < K ? (k) : 0] = sub0; break;
#define PHMM_TCAPTURE(k) if (k == klo && (S >> 14) < (best >> 14)) { best = S; x_end = x; }

    for (int x = 0; x <= W; ++x) {
        const int xn = (x + 1 < W) ? x + 1 : W - 1;
        const ColEntry nx = ldg(tab + xn);
        const uint32_t caps = e.x, cap_n = (e.y >> 16) & 0xFFu;
        const uint32_t goS = (e.y & 0xFFu) << 16, geS = ((e.y >> 8) & 0xFFu) << 16;
        const uint32_t gopS = go_prev + ((uint32_t)nuc_prior << 16), gepS = ge_prev + ((uint32_t)nuc_prior << 16);
        const RowsT rp = rows.shifted(x);
        uint32_t* bcol = bp + (size_t)x * K * bps;
        uint32_t i_run = kTbInf | kTbLabI;
        if (x >= K) {
            if (x < L) {
#pragma unroll
                for (int k = K - 1; k >= 0; --k) PHMM_TCELL(k, )
            } else {
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    PHMM_TCELL(k, PHMM_TCAPTURE(k))
                    if (k == klo) break;
                }
            }
        } else {
            const uint32_t sub0 = umin32(w0.y, prmt(caps, cap_n, w0.x));
            i_run = (x & 1) ? (gopS | kTbLabI) : (kTbInf | kTbLabI);
            if (x < L) {
                switch (x) { PHMM_REP64(PHMM_TCASE_PROLOGUE) default: break; }
            } else {
                const int klo = x - L;
#pragma unroll
                for (int k = K - 1; k >= 0; --k) {
                    if (k < x && k >= klo) PHMM_TCELL(k, PHMM_TCAPTURE(k))
                }
            }
            switch (x) { PHMM_REP64(PHMM_TCASE_ROW0) default: break; }
        }
        go_prev = goS; ge_prev = geS;
        const uint32_t z = i_run & 0x8000u;
        e.x = nx.x + z; e.y = nx.y + z;
    }
#undef PHMM_TCELL
#undef PHMM_TCASE_PROLOGUE
#undef PHMM_TCASE_ROW0
#undef PHMM_TCAPTURE
    *score_out = (int)(best >> 16);
    *x_end_out = x_end;
    *state_out = (int)((best >> 14) & 3u);
}

// The backward walk over the words dp_traceback_forward wrote. Same outputs as generic_align<true>: first_pos (-1 if the path
// leaves the band), the flank score and in-flank read bases of the forward replay's rules, optionally the two alignment strings.
struct TbModel { const char* truth; const char* snv_mask; const int8_t* snv_prior; const int8_t* gap_open; const int8_t* gap_extend; int nuc_prior; };
template <int BAND>
PHMM_HD void traceback_walk(const uint32_t* __restrict__ bp, const size_t bps, const TbModel& gm, const char* target, const uint8_t* quals, const int L,
                            int x, int state, const int lhs_flank, const int rhs_flank,
                            int* first_pos, int* flank_score, int* mask_size, char* align1, char* align2)
{
    constexpr int K = 2 * BAND;
    constexpr int LM = 0, LI = 1, LD = 3;
    const int W = L + K - 1, rhs_begin = W - rhs_flank;
    int y = L, fs = 0, ms = 0, n = 0;
    bool ok = x >= 0;
    while (ok && y > 0) {
        int ns;
        if (state == LM) {
            --x; --y;
            const int k = x - y;
            if (k < 0 || k >= K || x < 0) { ok = false; break; }
            ns = (int)((bp[((size_t)x * K + k) * bps] >> 6) & 3u);
            if (align1) { align1[n] = gm.truth[x]; align2[n] = target[y]; }
            if (x < lhs_flank || x >= rhs_begin) {
                const char t = gm.truth[x], r = target[y];
                if (t != r) {
                    if (t != 'N') { int q = quals[y]; if (gm.snv_mask[x] == r && (int)gm.snv_prior[x] < q) q = (int)gm.snv_prior[x]; fs += q; }
                    else fs += 2;
                }
                ++ms;
            }
        } else if (state == LI) {
            --y;
            const int k = x - y;
            if (k < 0 || k >= K) { ok = false; break; }
            ns = (int)((bp[((size_t)x * K + k) * bps] >> 22) & 3u);
            if (align1) { align1[n] = '-'; align2[n] = target[y]; }
            if (x < lhs_flank || x >= rhs_begin) { fs += (ns == LI ? (int)gm.gap_extend[x - 1] : (int)gm.gap_open[x - 1]) + gm.nuc_prior; ++ms; }
        } else {
            --x;
            const int k = x - y;
            if (k < 0 || k >= K || x < 0) { ok = false; break; }
            ns = (int)((bp[((size_t)x * K + k) * bps] >> 14) & 3u);
            if (align1) { align1[n] = gm.truth[x]; align2[n] = '-'; }
            if (x < lhs_flank || x >= rhs_begin) fs += (ns == LD ? (int)gm.gap_extend[x] : (int)gm.gap_open[x]);
        }
        state = ns;
        ++n;
    }
    if (!ok) { *first_pos = -1; *flank_score = 0; *mask_size = 0; if (align1) { align1[0] = 0; align2[0] = 0; } return; }
    if (align1) {
        align1[n] = 0; align2[n] = 0;
        for (int a = 0, b = n - 1; a < b; ++a, --b) {
            char t = align1[a]; align1[a] = align1[b]; align1[b] = t;
            t = align2[a]; align2[a] = align2[b]; align2[b] = t;
        }
    }
    *first_pos = x; *flank_score = fs; *mask_size = ms;
}

// ---------------------------------------------------------------------------------------------------------
// Generic path: int32, any band / alphabet, optional traceback + flank replay (one thread per alignment)
// ---------------------------------------------------------------------------------------------------------

struct GenericModel {
    const char*   truth;       // window start
    const char*   snv_mask;    // window start (never null on this path)
    const int8_t* snv_prior;
    const int8_t* gap_open;
    const int8_t* gap_extend;
    int nuc_prior;
};

PHMM_HD int generic_sub(const GenericModel& m, const char* target, const int8_t* quals, int x, int y)
{
    const char t = m.truth[x], r = target[y];
    if (r == t) return 0;
    int q = quals[y];
    if (m.snv_mask[x] == r && (int)m.snv_prior[x] < q) q = (int)m.snv_prior[x];
    return q < (t == 'N' ? 2 : kInf32) ? q : (t == 'N' ? 2 : kInf32);
}

constexpr int kGenericMaxDiag = 512;   // 2 * 256, the reference's widest band (simd_pair_hmm_wrapper.hpp:207-211)

// Score-only or traceback. State values are (score << 2) | label exactly like the reference (labels only set when TB).
// Row sweep: Mc[k] / Ic[k] hold the match / insertion arrivals of row y at diagonal k and are overwritten in place
// with row y+1's (m moves k → k, i moves k → k-1, whose slot is already consumed); d runs along the row in a scalar.
// bp: TB only — one byte per cell, (L+1) * K bytes at stride bps (cell c lives at bp[c * bps], so a grid of threads
//     can interleave their scratch for coalescing): bits 0-1 / 2-3 / 4-5 = predecessor label of the M / I / D arrival.
//     The M bits are stored first (plain store), the I and D bits are OR-ed in later by the same thread.
// Returns the score; TB additionally returns first_pos, the flank score and the in-flank read-base count
// (simd_pair_hmm.hpp:165-231 set_alignments fused with :352-430 calculate_flank_score_helper).
template <bool TB, int MAXK>
__host__ __device__ inline int generic_align(const int band, const GenericModel& gm, const char* target, const int8_t* quals, const int L,
                             unsigned char* __restrict__ bp, const size_t bps, const int lhs_flank, const int rhs_flank,
                             int* first_pos, int* flank_score, int* mask_size, char* align1 = nullptr, char* align2 = nullptr)
{
    const int K = 2 * band, W = L + K - 1;
    int Mc[MAXK], Ic[MAXK];
    constexpr int LM = 0, LI = 1, LD = 3;
    const int infp = kInf32 << 2;
    for (int k = 0; k < K; ++k) { Mc[k] = infp | (TB ? LM : 0); Ic[k] = infp | (TB ? LI : 0); }
    const int nuc = gm.nuc_prior << 2;
    int best = infp + (1 << 20), best_x = -1;
    for (int y = 0; y <= L; ++y) {
        int dd = infp | (TB ? LD : 0);          // d arrival of (y, y): nothing to the left inside the band
        for (int k = 0; k < K; ++k) {
            const int x = y + k;
            int mm = Mc[k];
            const int ii = Ic[k];
            int mg;
            if (y == 0) { mm = 0; mg = (x & 1) ? 0 : infp; } else mg = mm;
            const int S = min(mm, min(ii, dd));
            if (y == L && S < best) { best = S; best_x = x; }
            int dnext = infp | (TB ? LD : 0);
            if (x < W) {
                if (y < L) {   // match / mismatch → (x+1, y+1), diagonal k of the next row
                    const int v = S + (generic_sub(gm, target, quals, x, y) << 2);
                    if (TB) { bp[((size_t)(y + 1) * K + k) * bps] = (unsigned char)(v & 3); Mc[k] = (v & ~3) | LM; } else Mc[k] = v;
                }
                if (k + 1 < K) {   // deletion → (x+1, y)
                    const int v = min(dd + ((int)gm.gap_extend[x] << 2), min(mg, ii) + ((int)gm.gap_open[x] << 2));
                    if (TB) { bp[((size_t)y * K + (k + 1)) * bps] |= (unsigned char)((v & 3) << 4); dnext = (v & ~3) | LD; } else dnext = v;
                }
            }
            if (k >= 1 && y < L) {   // insertion → (x, y+1), diagonal k-1 of the next row
                const int v = min(ii + ((int)gm.gap_extend[x - 1] << 2), mg + ((int)gm.gap_open[x - 1] << 2)) + nuc;
                if (TB) { bp[((size_t)(y + 1) * K + (k - 1)) * bps] |= (unsigned char)((v & 3) << 2); Ic[k - 1] = (v & ~3) | LI; } else Ic[k - 1] = v;
            }
            dd = dnext;
        }
        Ic[K - 1] = infp | (TB ? LI : 0);   // top diagonal of the next row has no insertion predecessor
    }
    const int score = best >> 2;
    if (TB) {
        if (best_x < 0) { *first_pos = -1; *flank_score = 0; *mask_size = 0; return score; }
        // Walk the path backwards, accumulating the flank score with the forward replay's rules. The replay charges
        // gap OPEN for the first op of a run (prev_state != state, in forward order) and EXTEND otherwise; walking
        // backwards the "first op of a run" is the one whose predecessor state differs, which is ns below.
        const int rhs_begin = W - rhs_flank;
        int x = best_x, y = L, state = best & 3, fs = 0, ms = 0, n = 0;
        bool ok = true;
        while (y > 0) {
            const int k = x - y;
            if (k < 0 || k >= K) { ok = false; break; }
            const unsigned char b = bp[((size_t)y * K + k) * bps];
            int ns;
            if (state == LM) {
                ns = b & 3; --x; --y;
                if (align1) { align1[n] = gm.truth[x]; align2[n] = target[y]; }
                const bool inf = x < lhs_flank || x >= rhs_begin;     // truth_idx of this op == x after the decrement
                if (inf) {
                    const char t = gm.truth[x], r = target[y];
                    if (t != r) {
                        if (t != 'N') { int q = quals[y]; if (gm.snv_mask[x] == r) q = min(q, (int)gm.snv_prior[x]); fs += q; }
                        else fs += 2;
                    }
                    ++ms;
                }
            } else if (state == LI) {
                ns = (b >> 2) & 3; --y;
                if (align1) { align1[n] = '-'; align2[n] = target[y]; }
                const bool inf = x < lhs_flank || x >= rhs_begin;     // truth_idx of an insertion == current x
                if (inf) { fs += (ns == LI ? (int)gm.gap_extend[x - 1] : (int)gm.gap_open[x - 1]) + gm.nuc_prior; ++ms; }
            } else {
                ns = (b >> 4) & 3; --x;
                if (align1) { align1[n] = gm.truth[x]; align2[n] = '-'; }
                const bool inf = x < lhs_flank || x >= rhs_begin;
                if (inf) fs += (ns == LD ? (int)gm.gap_extend[x] : (int)gm.gap_open[x]);
            }
            state = ns;
            ++n;
        }
        if (align1 && ok) {   // the strings were produced end-first: reverse and terminate (simd_pair_hmm.hpp:219-230)
            align1[n] = 0; align2[n] = 0;
            for (int a = 0, b = n - 1; a < b; ++a, --b) {
                char t = align1[a]; align1[a] = align1[b]; align1[b] = t;
                t = align2[a]; align2[a] = align2[b]; align2[b] = t;
            }
        }
        if (!ok) { *first_pos = -1; *flank_score = 0; *mask_size = 0; return score; }
        *first_pos = x; *flank_score = fs; *mask_size = ms;
    }
    return score;
}

// ---------------------------------------------------------------------------------------------------------
// Per-candidate logic above the kernel (shared by the fused populate kernels; __host__ __device__ for CPU tests)
// ---------------------------------------------------------------------------------------------------------

struct HapView {            // one haplotype, strand-selected model arrays (HaplotypeLikelihoodModel::evaluate :269-275)
    const char*   seq;
    const char*   snv_mask;
    const int8_t* snv_prior;
    const int8_t* gap_open;
    const int8_t* gap_extend;
    int len;
};
struct ReadView {
    const char*    bases;
    const uint8_t* quals;
    int len;
};

constexpr int kBestInf = 0x7fffffff;   // "no candidate produced a value" == std::numeric_limits<double>::lowest()

enum CandKind { CAND_VALUE = 0, CAND_DP = 1, CAND_DP_FLANK = 2, CAND_LOWEST = 3 };

// haplotype_likelihood_model.cpp:187-201 num_out_of_range_bases (required pad == band, pair_hmm.hpp:33-38)
PHMM_HD int num_out_of_range_bases(const long long pos, const int read_len, const int hap_len, const int band)
{
    if (pos < band) return (int)(band - pos);
    const long long end = pos + read_len + band;
    if (end > hap_len) return (int)((long long)hap_len - end);
    return 0;
}

// pair_hmm.hpp:275-319 try_naive_evaluate (MutationModel: SNV mask + per-base gap arrays; flanks optional)
PHMM_HD bool naive_evaluate(const HapView& h, const ReadView& r, const int offset, const bool use_flanks,
                            const int lhs_flank, const int rhs_flank, int* phred)
{
    const char* t = h.seq + offset;
    const int L = r.len;
    int i = 0;
    while (i < L && r.bases[i] == t[i]) ++i;
    if (i == L) { *phred = 0; return true; }
    int j = i + 1;
    while (j < L && r.bases[j] == t[j]) ++j;
    if (j != L) return false;
    const int tidx = i + offset;
    if (use_flanks && (tidx < lhs_flank || tidx >= h.len - rhs_flank)) { *phred = 0; return true; }   // :206-214, :298
    int mp = r.quals[i];
    if (h.snv_mask[tidx] == r.bases[i]) { const int cap = (uint8_t)h.snv_prior[tidx]; if (cap < mp) mp = cap; }   // :250-263
    const int go = h.gap_open[tidx];
    if (mp <= go) { *phred = mp; return true; }
    bool eq = true;
    for (int a = i + 1; a < L; ++a) if (r.bases[a] != h.seq[tidx + (a - i - 1)]) { eq = false; break; }   // :305-308
    if (eq) { *phred = go; return true; }
    eq = true;
    for (int a = i; a < L; ++a) if (r.bases[a] != h.seq[tidx + 1 + (a - i)]) { eq = false; break; }       // :309-312
    if (eq) { *phred = go; return true; }
    if (mp <= go + (int)h.gap_extend[tidx]) { *phred = mp; return true; }                                  // :313-315
    return false;
}

// hmm::evaluate for one mapping position up to the point where a DP is needed (pair_hmm.hpp:827-841, :723-766).
//   CAND_VALUE    *out = integer phred penalty (result is -ln10/10 * *out)
//   CAND_DP       *out = window offset a = max(0, p - band); score-only DP suffices
//   CAND_DP_FLANK *out = a; traceback + flank discount needed (read within band of a flank, :123-130)
//   CAND_LOWEST   window does not fit: lowest() (:736-738)
PHMM_HD CandKind classify_candidate(const HapView& h, const ReadView& r, const int band, const int p,
                                    const bool shortcut, const bool use_flanks, const int lhs_flank, const int rhs_flank, int* out)
{
    if (shortcut) {
        int phred;
        if (naive_evaluate(h, r, p, use_flanks, lhs_flank, rhs_flank, &phred)) { *out = phred; return CAND_VALUE; }
    }
    const int W = r.len + 2 * band - 1;
    const int a = p - band > 0 ? p - band : 0;
    if (a + W > h.len) return CAND_LOWEST;
    *out = a;
    const bool near_flank = use_flanks && (p < lhs_flank + band || p + r.len + band > h.len - rhs_flank);
    return near_flank ? CAND_DP_FLANK : CAND_DP;
}

// haplotype_likelihood_model.cpp:211-259 max_score, unrolled into "slots" so that a warp can walk the candidates of
// 32 (haplotype, read) pairs in lock-step: slot c < npos is the c-th listed mapping position, slot npos is the read's
// original position (if it was not listed), slot npos+1 is the shifted fallback (only if nothing was in range).
// Returns 1 with *p set when the slot yields a position to evaluate, 0 when it yields nothing, and -1 for
// ShortHaplotypeError (*p = required extension).
struct EnumState { bool mapped; bool has_in_range; };

PHMM_HD int candidate_slot(const int c, const int npos, const int32_t* pos, const long long orig,
                           const int read_len, const int hap_len, const int band, EnumState& st, int* p)
{
    if (c < npos) {
        const int q = pos[c];
        if (q == orig) st.mapped = true;                                               // :224-226
        if (num_out_of_range_bases(q, read_len, hap_len, band) == 0) { st.has_in_range = true; *p = q; return 1; }
        return 0;
    }
    if (c == npos) {                                                                   // :233-237
        if (!st.mapped && num_out_of_range_bases(orig, read_len, hap_len, band) == 0) { st.has_in_range = true; *p = (int)orig; return 1; }
        return 0;
    }
    if (c == npos + 1 && !st.has_in_range) {                                           // :238-256
        const int min_shift = num_out_of_range_bases(orig, read_len, hap_len, band);
        long long fin = orig;
        if (min_shift > 0) {
            fin += min_shift;
            if (num_out_of_range_bases(fin, read_len, hap_len, band) != 0) { *p = min_shift; return -1; }
        } else {
            const long long left = -(long long)min_shift;
            if (orig >= left) fin -= left;
            else { *p = (int)(left - orig); return -1; }
        }
        *p = (int)fin;
        return 1;
    }
    return 0;
}

// pair_hmm.hpp:755-764: combine the traceback DP's score with the flank replay (window coordinates: :573-588)
PHMM_HD void window_flanks(const int a, const int W, const int hap_len, const int lhs_flank, const int rhs_flank, int* lhs, int* rhs)
{
    *lhs = lhs_flank < a ? 0 : lhs_flank - a;
    if (a + W < hap_len - rhs_flank) *rhs = 0;
    else { const int v = rhs_flank + a + W - hap_len; *rhs = v < 0 ? 0 : v; }
}
PHMM_HD int discount_flank(const int score, int flank, const int read_len, const int mask_size, const int first_pos)
{
    if (first_pos == -1) return kBestInf;               // :750-752 overflow → lowest()
    if (read_len - mask_size < 2) flank = 0;            // :757-759 min_explained_bases
    return flank <= score ? score - flank : score + flank;   // :760-764
}

// haplotype_likelihood_model.cpp:285-303: mapping-quality mixing and the > -1e-15 clamp, from the integer penalty.
__host__ __device__ inline double finish_likelihood(const int best, const bool use_mapq, int mapq, const int mapq_cap, const int mapq_trigger)
{
    const double c = 0.230258509299404568401799145468436420760110148862877297603;   // utils/maths.hpp:41
    const double ln_given_mapped = best == kBestInf ? -1.7976931348623157e308 : -c * (double)best;
    if (use_mapq) {
        // a trigger at or above the cap is dropped when the model is configured (haplotype_likelihood_model.cpp:49-51, 117-119)
        if (mapq_trigger >= 0 && mapq_trigger < mapq_cap && mapq >= mapq_trigger) mapq = mapq_cap;
        const double ln_miss = -c * (double)mapq;
        const double ln_mapped = log(1.0 - exp(ln_miss));
        const double a = ln_mapped + ln_given_mapped, b = ln_miss;
        const double lo = b < a ? b : a, hi = b < a ? a : b;          // std::minmax (utils/maths.hpp:294-298)
        const double r = hi + log1p(exp(lo - hi));
        return r > -1e-15 ? 0.0 : r;
    }
    return ln_given_mapped > -1e-15 ? 0.0 : ln_given_mapped;
}

} // namespace phmm
