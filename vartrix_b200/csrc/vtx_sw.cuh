// vtx_sw.cuh -- Smith-Waterman kernels (sm_100a) of the vartrix read-scoring path.
//
// Replaces bio::alignment::pairwise::banded::Aligner::local x2 per (read, locus) pair
// (/root/reference/src/main.rs:898-901) and fuses evaluate_scores (main.rs:1019-1030) plus the
// count-matrix increment as an epilogue.  Integer DP, no tensor cores:
//
//  * ref and alt haplotype scores travel in the two int16 lanes of one 32-bit word (biased by kBias, see
//    below) and every cell update is 4.5 native DPX instructions -- 2x VIADDMNMX.S16x2 (E, F),
//    VIMNMX3.S16x2 (max(diag + s, F, 0)), VIMNMX.S16x2 (H), half a VIMNMX3 (running maximum) -- plus two
//    ordinary 32-bit adds (diag + s and H + gap_open + gap_extend).
//  * LPP (=8) lanes cooperate on one pair: lane g owns C consecutive haplotype columns whose H/F
//    state lives in registers; rows are skewed by one step per lane (anti-diagonal wavefront) and the
//    boundary column travels to lane g+1 with two __shfl_up_sync per step.  A warp scores 32/LPP pairs
//    of the SAME locus at a time (a "tile").
//  * the substitution scores come from a per-locus profile in shared memory (5 read-base rows x
//    columns, words = {s_ref, s_alt}), built once per locus per warp and read with conflict-free
//    LDS.128; the read itself is turned into a per-row byte offset into that profile.
//  * out-of-range rows/columns are all-mismatch sentinels, which can never raise a local maximum, so the
//    inner loop carries no bounds predicates.
//
// Exactness: biased values stay inside [-300, 16384 + 1024 + 7] for reads up to kFastMaxRead bases, so int16
// never saturates and the low half never borrows/carries other than the one constant carry; longer reads, haplotypes wider than the largest tile class or with
// IUPAC/"=" bytes go to vtx_k_sw_generic (plain per-thread DP with byte equality).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace vtx {

constexpr int kMatch = 1, kMismatch = -5, kGapOpen = -5, kGapExtend = -1;   // main.rs:35-38
constexpr int kGoe = kGapOpen + kGapExtend;                                 // cost of the first gap base

__host__ __device__ constexpr uint32_t pack2(int lo, int hi)
{
    return (uint32_t(uint16_t(int16_t(hi))) << 16) | uint32_t(uint16_t(int16_t(lo)));
}
// Every packed quantity (H, H+gap, E, F, running maximum) is stored with a bias of kBias in both halves.  Max and
// fused add-max instructions are oblivious to a common bias, and it makes plain 32-bit adds of packed words exact:
// adding a small positive pair never carries out of the low half, and adding (gap, gap) with gap < 0 to halves that
// are >= kBias always carries exactly once, which the constant kGoeAdd already contains.  So the two packed adds of
// a cell are ordinary integer adds (VIADD at full rate or IMAD.IADD on the FMA pipe) instead of half-rate VIADD.16x2.
constexpr int kBias = 16384;
constexpr uint32_t kGE2 = pack2(kGapExtend, kGapExtend);
constexpr uint32_t kBIAS2 = pack2(kBias, kBias);                    // biased 0 (the floor of local alignment)
constexpr uint32_t kGOE2 = pack2(kBias + kGoe, kBias + kGoe);       // biased (0 + gap): H = 0 seen through H + go + ge
constexpr uint32_t kNEG2 = pack2(0, 0);                             // biased -16384 ("minus infinity")
constexpr uint32_t kGoeAdd = (uint32_t(uint16_t(int16_t(kGoe - 1))) << 16) | uint32_t(uint16_t(int16_t(kGoe)));   // + (gap, gap) incl. the carry
// Cell update.  1 (default): the diagonal add rides inside VIADDMNMX, x = max(diag + s, F), and the floor of local
// alignment joins the H maximum, h = VIMNMX3(x, E, 0).  0: round-1 form, tf = VIMNMX3(diag + s, F, 0), h = VIMNMX(tf, E).
// Measured on B200 (profiles/r02_dpx_microbench.txt): 3-input DPX instructions hold the ALU pipe for 2 cycles, the 2-input
// VIMNMX for 1, and a plain add next to a DPX instruction is free -- so form 1 costs 12 more ALU cycles per main-pass step
// of the folded kernel (126 instead of 114) but 5 fewer issue slots (117 instead of 122), and the kernel is bound by both
// (ncu: issue slots 81 % busy, ALU pipe 76 %).  Form 1 measured +1.9 %, with the row loop unrolled twice +3.7 %
// (profiles/r02_fold_variants.txt).
#ifndef VTX_SW_FUSE
#define VTX_SW_FUSE 1
#endif
// The remaining plain add of a cell, H + gap.  ptxas places a plain `x + c` on the ALU pipe (VIADD), which the DPX
// instructions already saturate; written as x * one + c with a run-time `one` it is an IMAD on the FMA pipe instead.
// VTX_SW_HADD: 0 = plain add everywhere, 1 = IMAD everywhere, 2 = IMAD on even columns (splits the adds between the pipes).
#ifndef VTX_SW_HADD
#define VTX_SW_HADD 0
#endif
__device__ __forceinline__ uint32_t padd(uint32_t x, uint32_t one, uint32_t c)
{
    (void)one;
    return x + c;
}
__device__ __forceinline__ uint32_t hadd(uint32_t h, uint32_t one, int col)
{
#if VTX_SW_HADD == 1
    (void)col;
    return h * one + kGoeAdd;
#elif VTX_SW_HADD == 2
    return (col & 1) ? h + kGoeAdd : h * one + kGoeAdd;
#else
    (void)one; (void)col;
    return h + kGoeAdd;
#endif
}
// H = max(diag + s, F, E, 0) of one cell (biased halves; `diag` is stored as H + goe and `s` as s - goe)
__device__ __forceinline__ uint32_t sw_h(uint32_t diag, uint32_t one, uint32_t s, uint32_t f, uint32_t e)
{
#if VTX_SW_FUSE
    (void)one;
    return __vimax3_s16x2(__viaddmax_s16x2(diag, s, f), e, kBIAS2);
#else
    return __vmaxs2(__vimax3_s16x2(padd(diag, one, s), f, kBIAS2), e);
#endif
}
// profile entries are biased by -kGoe because the stored state is H + kGoe
constexpr int kProfMatch = kMatch - kGoe, kProfMis = kMismatch - kGoe;     // 7, 1

constexpr int kFastMaxRead = 1024;       // row-code buffer of the single-phase kernels; longer reads are scored in row blocks
constexpr int kMaxRead = 16000;          // biased int16: H + 16384 must stay below 32768
constexpr int kNumFastClasses = 4;                 // single-phase tile classes 0..3
constexpr int kSlowClass = kNumFastClasses;        // 4: generic kernel
constexpr int kNumSplitClasses = 2;                // 5, 6: two-phase kernels (vtx_sw_split.cuh)
constexpr int kSplitClass0 = kSlowClass + 1;
constexpr int kFoldClass = kSplitClass0 + kNumSplitClasses;   // 7: folded kernel (vtx_sw_fold.cuh)
constexpr int kNumClasses = kFoldClass + 1;
constexpr int kTileChunk = 8;            // most tiles grabbed per atomic

// fast tile classes: lanes per pair, columns per lane, storage stride (words; CS % 4 == 0, (CS/4) odd
// so the 8 lanes of an LDS.128 wavefront hit 8 distinct 16-byte bank groups)
template <int CLS> struct TileClass;
// THREADS x MINB = CTA shape / CTAs per SM the register allocator must leave room for (measured on B200,
// profiles/r01_sw_variants.txt: 20 warps/SM at <= 102 registers beats 16 warps at 108 by ~4 %)
template <> struct TileClass<0> { static constexpr int LPP = 8, C = 26, CS = 28, THREADS = 320, MINB = 2; };   // n <= 208 (SNV, pad 100)
template <> struct TileClass<1> { static constexpr int LPP = 8, C = 29, CS = 36, THREADS = 320, MINB = 2; };   // n <= 232 (indels <= 30)
template <> struct TileClass<2> { static constexpr int LPP = 8, C = 32, CS = 36, THREADS = 256, MINB = 2; };   // n <= 256
template <> struct TileClass<3> { static constexpr int LPP = 8, C = 40, CS = 44, THREADS = 384, MINB = 1; };   // n <= 320 per pass
// Class 3 also takes windows wider than 320 columns (e.g. --padding 200) in several passes of 320 columns: the last
// column (H + gap, E) of every row is parked in shared memory between passes, like the two-phase kernels do.
constexpr int kMultiClass = 3;
constexpr int kMultiMaxRead = 256;       // reads longer than this fall back to the generic kernel for wide windows
__host__ __device__ constexpr int class_max_n(int cls)
{
    return cls == 0 ? 208 : cls == 1 ? 232 : cls == 2 ? 256 : cls == 3 ? 320 : 0x7fffffff;
}
constexpr int kSlowPairsPerWarp = 16;    // generic kernel: one thread per (pair, haplotype)

struct SwArgs {
    // staged batch
    const uint8_t* hap_bytes;
    const uint32_t* ref_off; const uint32_t* ref_len; const uint32_t* alt_off; const uint32_t* alt_len;
    const uint8_t* read_nib; const uint64_t* read_off; const uint32_t* read_len;
    // pairs (locus-major) and tiles of this class
    const uint32_t* pair_read;
    const uint32_t* pair_start;     // [n_loci + 1]
    const uint32_t* tile_start;     // [n_loci + 1] exclusive scan of this class's tiles per locus
    uint32_t n_loci;
    uint32_t* tile_counter;         // work-stealing cursor (zeroed before launch)
    // epilogue
    const uint32_t* pair_slot;      // counter slot of each pair (nullptr: no scatter)
    uint32_t* counters;             // [slot][4] = {ref, alt, unk, -}
    uint32_t* pair_scores;          // optional [pair] packed {ref, alt} int16 (nullptr: not kept)
    int32_t min_score;              // MIN_SCORE main.rs:30
    int32_t mcap;                   // row-code capacity (even, >= longest read in the batch)
    uint32_t k64k;                  // 65536 as a run-time value (keeps a shift-add on the FMA pipe, see vtx_sw_split.cuh)
    uint32_t one;                   // 1 as a run-time value (keeps the packed adds on the FMA pipe)
    int32_t multi;                  // class 3 may run several column passes (boundary buffer present in smem)
    int32_t fold_mid_cap;           // folded kernel: allele columns its per-warp table holds (set by launch_sw_fold)
    // generic kernel only
    uint32_t* scratch;              // [warps][max_hap + 1][32]
    uint32_t max_hap;
};

__device__ __forceinline__ uint32_t hap_code(uint8_t b)
{   // haplotype byte -> profile column code; anything but upper-case ACGT can never equal a fast-path read base
    return b == 'A' ? 0u : b == 'C' ? 1u : b == 'G' ? 2u : b == 'T' ? 3u : 5u;
}
__device__ __forceinline__ uint32_t nib_code(uint32_t nib)
{   // BAM nibble -> profile row: A(1) C(2) G(4) T(8) -> 0..3, everything else -> 4 (matches nothing)
    return (0x4444444344424104ull >> (nib * 4)) & 0xF;
}

// largest l in [0, n) with a[l] <= v  (a ascending, a[0] == 0 <= v < a[n])
__device__ __forceinline__ uint32_t upper_locus(const uint32_t* __restrict__ a, uint32_t n, uint32_t v)
{
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

// main.rs:1019-1030 fused with the count increment that main.rs:1032-1039 / 1090-1098 perform later
__device__ __forceinline__ void call_and_scatter(const SwArgs& a, uint32_t pair, uint32_t packed)
{
    const int ref_score = int(int16_t(packed & 0xFFFF)), alt_score = int(int16_t(packed >> 16));
    if (a.pair_scores) a.pair_scores[pair] = pack2(ref_score, alt_score);
    if (!a.pair_slot) return;
    if (ref_score < a.min_score && alt_score < a.min_score) return;            // None
    const uint32_t k = ref_score > alt_score ? 0u : (alt_score > ref_score ? 1u : 2u);
    atomicAdd(a.counters + size_t(a.pair_slot[pair]) * 4 + k, 1u);
}

template <int CLS>
__global__ void __launch_bounds__(TileClass<CLS>::THREADS, TileClass<CLS>::MINB) vtx_k_sw_pairs(const SwArgs a)
{
    using TC = TileClass<CLS>;
    constexpr int LPP = TC::LPP, C = TC::C, CS = TC::CS;
    constexpr int PPW = 32 / LPP;              // pairs per warp tile
    constexpr int RS = LPP * CS;               // profile row stride in words (multiple of 32)
    constexpr int M = LPP;                     // sentinel margin of the row-code buffer
    static_assert(CS % 4 == 0 && ((CS / 4) & 1) == 1 && CS >= C, "bank-conflict-free stride");
    static_assert(RS % 32 == 0, "row stride keeps lanes on their banks");
    constexpr uint32_t kSentinel = 4u * RS * 4u;   // byte offset of the all-mismatch row

    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane % LPP, grp = lane / LPP;
    constexpr bool MULTI = (CLS == kMultiClass);
    const int code_stride = a.mcap + 2 * M;                      // u16 entries per group
    const int bnd_stride = (MULTI && a.multi) ? a.mcap + 8 : 0;  // uint2 entries per group (multi-pass boundary column)
    const size_t codes_bytes = (size_t(PPW) * code_stride * 2 + 7) & ~size_t(7);
    const size_t warp_bytes = size_t(5 * RS) * 4 + codes_bytes + size_t(PPW) * bnd_stride * 8;
    uint8_t* wbase = smem_raw + warp * ((warp_bytes + 15) & ~size_t(15));
    uint32_t* prof = reinterpret_cast<uint32_t*>(wbase);
    uint16_t* codes = reinterpret_cast<uint16_t*>(wbase + size_t(5 * RS) * 4) + grp * code_stride;
    uint2* bnd = reinterpret_cast<uint2*>(wbase + size_t(5 * RS) * 4 + codes_bytes) + grp * bnd_stride;

    const uint32_t n_tiles = __ldg(a.tile_start + a.n_loci);
    uint32_t cached_locus = 0xFFFFFFFFu;
    // tiles grabbed per atomic: up to kTileChunk for locality of the per-locus profile, fewer when the shard is
    // small so that every warp still gets >= ~16 grabs (tail balance)
    const uint32_t tile_chunk = max(1u, min(uint32_t(kTileChunk), n_tiles / (gridDim.x * (blockDim.x >> 5) * 16u)));

    for (;;) {
        uint32_t chunk = 0;
        if (lane == 0) chunk = atomicAdd(a.tile_counter, 1u);
        chunk = __shfl_sync(0xffffffffu, chunk, 0);
        const uint32_t t_begin = chunk * tile_chunk;
        if (t_begin >= n_tiles) break;
        const uint32_t t_end = min(t_begin + tile_chunk, n_tiles);

        uint32_t locus = upper_locus(a.tile_start, a.n_loci, t_begin);
        for (uint32_t tile = t_begin; tile < t_end; ++tile) {
            while (tile >= __ldg(a.tile_start + locus + 1)) ++locus;      // tiles of a chunk are consecutive
            const uint32_t p0 = __ldg(a.pair_start + locus) + PPW * (tile - __ldg(a.tile_start + locus));
            const uint32_t p_end = __ldg(a.pair_start + locus + 1);

            __syncwarp();
            const uint8_t* rh = a.hap_bytes + __ldg(a.ref_off + locus);
            const uint8_t* ah = a.hap_bytes + __ldg(a.alt_off + locus);
            const int n_ref = int(__ldg(a.ref_len + locus)), n_alt = int(__ldg(a.alt_len + locus));
            const int n_pass = MULTI ? max(1, (max(n_ref, n_alt) + LPP * C - 1) / (LPP * C)) : 1;
            // per-locus substitution profile of columns [col0, col0 + LPP*C): rebuilt when the locus (or the pass) changes
            auto build_profile = [&](int col0) {
                for (int idx = lane; idx < RS; idx += 32) {
                    const int gg = idx / CS, k = idx - gg * CS;
                    const int j = col0 + gg * C + k;
                    uint32_t rb = 5, ab = 5;
                    if (k < C) {
                        if (j < n_ref) rb = hap_code(__ldg(rh + j));
                        if (j < n_alt) ab = hap_code(__ldg(ah + j));
                    }
#pragma unroll
                    for (uint32_t r = 0; r < 5; ++r)
                        prof[r * RS + idx] = pack2(r == rb ? kProfMatch : kProfMis, r == ab ? kProfMatch : kProfMis);
                }
            };
            if (n_pass == 1 && locus != cached_locus) { cached_locus = locus; build_profile(0); }
            if (n_pass > 1) cached_locus = 0xFFFFFFFFu;
            // ---- row codes of this group's read: byte offset of the profile row per read base ----
            const uint32_t pair = p0 + grp;
            const bool active = pair < p_end;
            int m = 0;
            const uint8_t* nib = nullptr;
            if (active) {
                const uint32_t r = __ldg(a.pair_read + pair);
                m = int(__ldg(a.read_len + r));
                nib = a.read_nib + __ldg(a.read_off + r);
            }
            // row codes: byte offset of the profile row per read base, for the rows [t0 - M, t0 + R + M) of the current
            // row block (reads longer than the buffer are scored block by block; the DP state stays in registers)
            const int R = a.mcap;
            auto fill_codes = [&](int t0) {
                for (int e = g; e < code_stride; e += LPP) {
                    const int row = t0 - M + e;
                    uint32_t off = kSentinel;
                    if (row >= 0 && row < m) {
                        const uint32_t by = __ldg(nib + (row >> 1));
                        off = nib_code((row & 1) ? (by & 0xF) : (by >> 4)) * (RS * 4);
                    }
                    codes[e] = uint16_t(off);
                }
            };
            int mmax = m;
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) mmax = max(mmax, __shfl_xor_sync(0xffffffffu, mmax, o));

            // ---- anti-diagonal wavefront: lane g works on row (t - g) of its C columns ----
            uint32_t best = kBIAS2;
            const uint8_t* lane_prof = reinterpret_cast<const uint8_t*>(prof) + g * CS * 4;
            const uint16_t* my_codes = codes + M - g;
            const int steps = mmax + LPP - 1;
            const uint32_t one = a.one;
            for (int pass = 0; pass < n_pass; ++pass) {
                if (MULTI && n_pass > 1) { __syncwarp(); build_profile(pass * LPP * C); __syncwarp(); }
                uint32_t hg[C], f[C];
#pragma unroll
                for (int c = 0; c < C; ++c) { hg[c] = kGOE2; f[c] = kNEG2; }
                uint32_t hg_last = kGOE2, e_last = kNEG2, diag_save = kGOE2;
                for (int t0 = 0; t0 < steps; t0 += R) {
                __syncwarp();
                fill_codes(t0);
                __syncwarp();
                const int t_hi = min(steps, t0 + R);
                for (int t = t0; t < t_hi; ++t) {
                    uint32_t hl = __shfl_up_sync(0xffffffffu, hg_last, 1, LPP);
                    uint32_t el = __shfl_up_sync(0xffffffffu, e_last, 1, LPP);
                    if (g == 0) {
                        hl = kGOE2; el = kNEG2;
                        if (MULTI && pass > 0 && t < mmax) { const uint2 b = bnd[t]; hl = b.x; el = b.y; }   // column col0 - 1 of row t
                    }
                    const uint4* prow = reinterpret_cast<const uint4*>(lane_prof + my_codes[t - t0]);
                    uint32_t diag = diag_save;
                    diag_save = hl;
                    // E[i][c] = max(E[i][c-1] + ge, H[i][c-1] + goe)
                    uint32_t e = el, eg = hl, hleft = hl;
#pragma unroll
                    for (int q = 0; q < (C + 3) / 4; ++q) {
                        const uint4 s4 = prow[q];
                        const uint32_t sv[4] = { s4.x, s4.y, s4.z, s4.w };
                        uint32_t hh[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const int c = 4 * q + k;
                            if (c < C) {
                                const uint32_t fc = __viaddmax_s16x2(f[c], kGE2, hg[c]);     // F[i][c]
                                e = __viaddmax_s16x2(e, kGE2, eg);                          // E[i][c]
                                const uint32_t h = sw_h(diag, one, sv[k], fc, e);           // H[i][c]
                                hh[k] = h;
                                diag = hg[c];
                                hleft = hadd(h, one, c);                                    // H + goe
                                eg = hleft;
                                hg[c] = hleft;
                                f[c] = fc;
                            } else {
                                hh[k] = kBIAS2;
                            }
                        }
                        best = __vimax3_s16x2(best, hh[0], hh[1]);
                        if (4 * q + 2 < C) best = __vimax3_s16x2(best, hh[2], hh[3]);
                    }
                    hg_last = hleft;
                    e_last = e;
                    if (MULTI && pass + 1 < n_pass && g == LPP - 1 && t >= LPP - 1) bnd[t - (LPP - 1)] = make_uint2(hleft, e);
                }
                }
            }
            // ---- epilogue: group maximum, call, atomic scatter ----
#pragma unroll
            for (int o = LPP / 2; o >= 1; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(0xffffffffu, best, o));
            if (active && g == 0) call_and_scatter(a, pair, best - kBIAS2);           // un-bias both halves (no borrow: halves >= kBias)
        }
    }
}

// Generic kernel: any read length / haplotype width / byte alphabet.  One thread per (pair, haplotype),
// plain row-by-row Gotoh DP with exact byte equality against "=ACMGRSVTWYHKDBN"[nibble] (main.rs:896-898).
// Rare path (IUPAC bytes in a REF allele, --padding > 150, very long reads): clarity over speed.
__global__ void __launch_bounds__(128) vtx_k_sw_generic(const SwArgs a)
{
    const int lane = threadIdx.x & 31;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t* rowbuf = a.scratch + size_t(gwarp) * (size_t(a.max_hap) + 1) * 32 + lane;   // [(j)*32], {H, F} per column
    const uint32_t n_tiles = __ldg(a.tile_start + a.n_loci);
    const int sub = lane >> 1, which = lane & 1;
    for (;;) {
        uint32_t tile = 0;
        if (lane == 0) tile = atomicAdd(a.tile_counter, 1u);
        tile = __shfl_sync(0xffffffffu, tile, 0);
        if (tile >= n_tiles) break;
        const uint32_t locus = upper_locus(a.tile_start, a.n_loci, tile);
        const uint32_t p0 = __ldg(a.pair_start + locus) + kSlowPairsPerWarp * (tile - __ldg(a.tile_start + locus));
        const uint32_t p_end = __ldg(a.pair_start + locus + 1);
        const uint32_t pair = p0 + sub;
        int score = 0;
        if (pair < p_end) {
            const uint32_t r = __ldg(a.pair_read + pair);
            const int m = int(__ldg(a.read_len + r));
            const uint8_t* nib = a.read_nib + __ldg(a.read_off + r);
            const uint8_t* hap = a.hap_bytes + (which ? __ldg(a.alt_off + locus) : __ldg(a.ref_off + locus));
            const int n = int(which ? __ldg(a.alt_len + locus) : __ldg(a.ref_len + locus));
            for (int j = 0; j <= n; ++j) rowbuf[size_t(j) * 32] = pack2(0, -30000);
            for (int i = 0; i < m; ++i) {
                const uint32_t by = __ldg(nib + (i >> 1));
                const uint8_t xc = uint8_t("=ACMGRSVTWYHKDBN"[(i & 1) ? (by & 0xF) : (by >> 4)]);
                int diag = 0, left = 0, e = -30000;
                for (int j = 1; j <= n; ++j) {
                    const uint32_t w = rowbuf[size_t(j) * 32];
                    const int up = int(int16_t(w & 0xFFFF)), fup = int(int16_t(w >> 16));
                    const int fv = max(fup + kGapExtend, up + kGoe);
                    e = max(e + kGapExtend, left + kGoe);
                    int h = diag + (xc == __ldg(hap + j - 1) ? kMatch : kMismatch);
                    h = max(max(h, fv), max(e, 0));
                    rowbuf[size_t(j) * 32] = pack2(h, max(fv, -30000));
                    diag = up;
                    left = h;
                    e = max(e, -30000);
                    score = max(score, h);
                }
            }
        }
        const int other = __shfl_xor_sync(0xffffffffu, score, 1);
        if (pair < p_end && which == 0) call_and_scatter(a, pair, pack2(score, other));
    }
}

}  // namespace vtx
