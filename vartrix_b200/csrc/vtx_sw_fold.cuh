// vtx_sw_fold.cuh -- "folded" Smith-Waterman: neither shared flank of a locus is computed per haplotype.
//
// construct_haplotypes (/root/reference/src/main.rs:958-994) gives the ref and the alt window the SAME left
// flank and the SAME right flank; only the allele columns in between differ.  The local-alignment maximum
// decomposes exactly (oracle/vtx_oracle.c::vtxo_sw_fold pins this on the CPU against the full matrix):
//
//   best = max( max H over the prefix columns,                                 -- forward DP, shared
//               max Hr over the suffix columns,                                -- DP of the REVERSED read against
//                                                                                 the reversed suffix, shared
//               max H over the allele ("middle") columns,                      -- forward DP continued, per haplotype
//               max_i  H(i, last) + Hr(i + 1),  E(i, last) + Er(i + 1) - go )  -- junction, per haplotype
//
// (E = horizontal-gap state; a gap that runs across the junction was opened on both sides, hence "- go").
// A warp tile is 4 reads of one locus, one read per 8-lane unit:
//
//   main pass   kFoldP = 96 columns, 12 per lane, rows skewed by one step per lane exactly like the other
//               kernels -- but the two int16 halves are (forward DP over hap[0, 96), reversed DP over
//               hap[n - 96, n) reversed) of the SAME read.  Row i of the read meets forward code f = read[i] and reverse
//               code r = read[m - 1 - i], so the profile is pre-merged over the 16 (f, r) pairs of ACGT plus one
//               all-mismatch row: per step a lane loads one code byte (4 f + r) and one profile row (3 LDS.128), used as
//               loaded.  The last column (H + gap, E) of every row goes to shared memory.
//   middle      the n - 192 allele columns (9 for an SNV with --padding 100, up to 40): halves are (ref, alt)
//               again.  Transposed wavefront: lane g owns the 19 read rows [19 g, 19 g + 19), whose (H + gap, E)
//               start from the parked forward boundary, and walks over the columns one step per column,
//               skewed by one column per lane; F travels down the rows (one __shfl_up per step).
//   junction    when a lane has finished the last allele column of a haplotype it adds the parked reverse
//               boundary of the partner rows (reversed row m - 2 - r for forward row r).
//
// Per pair this is 2 x 96 + (n - 192) column-passes in "one read per word" units instead of 96 / 2 + (n - 96):
// ~25 % fewer DPX instructions than vtx_k_sw_split for an SNV window.  Reads up to kFoldMaxRead bases,
// windows with both flanks >= 96 columns in common and at most kFoldMaxMid allele columns.
//
// A tile in which some read has a base other than ACGT (N, IUPAC: nib_code 4, matches nothing) has no pair row for
// it; such tiles (rare: real reads seldom carry an N) run a second instantiation of the main pass whose code byte
// keeps both codes, f << 3 | r, and which assembles each word from the forward half of row 4 f and the reverse half
// of row r, taking the all-mismatch row for a code of 4.
#pragma once
#include "vtx_sw.cuh"

namespace vtx {

constexpr int kFoldP = 96;             // forward-prefix and reversed-suffix columns of the main pass (8 lanes x 12)
constexpr int kFoldC1 = 12;
constexpr int kFoldPPW = 4;            // pairs per warp tile
constexpr int kFoldR = 19;             // read rows per lane in the middle (8 x 19 = 152)
constexpr int kFoldMaxRead = 8 * kFoldR;
constexpr int kFoldMaxMid = 40;        // allele columns: n <= 2 * 96 + 40 = 232
constexpr int kFoldProfRows = 17;      // pre-merged profile: row 4 f + r for f, r in ACGT, row 16 all mismatch
constexpr uint8_t kFoldSentinel = 16;            // code byte of a row outside the read
constexpr uint8_t kFoldSentinelMixed = 4 << 3 | 4;   // the same in the code of the mixed main pass (f << 3 | r)
// boundary rows kept per read; 156 (not 152) so that the four reads of a tile start 8, 16 and 24 banks apart
// (152 rows x 8 bytes put reads 0/2 and 1/3 on the same banks: a 2-way conflict on every boundary store and load)
constexpr int kFoldRows = kFoldMaxRead + 4;
constexpr int kFoldCodeStride = kFoldMaxRead + 16;   // row codes per read (8 sentinels either side)
// 288 threads x 2 CTAs = 18 warps/SM at 96 registers.  Round 1 (unfused cell, no unrolling): 320 x 2 beat 256 x 2 by 5 %;
// with the fused cell and the row loop unrolled twice 288 x 2 is the best of 256 / 288 / 320 by ~1 %
// (profiles/r02_fold_variants.txt): the kernel is bound by issue slots and the ALU pipe, not by latency.  The launch drops to
// kFoldThreadsNarrow when two 288-thread CTAs do not fit an SM with the allele table the batch needs (wide indel windows).
#ifndef VTX_FOLD_UNROLL
#define VTX_FOLD_UNROLL 2
#endif
constexpr int kFoldThreads = 288;
constexpr int kFoldThreadsNarrow = 256;
constexpr int kFoldUnroll = VTX_FOLD_UNROLL;         // row-loop unrolling of the main pass
#ifndef VTX_FOLD_MID_UNROLL
#define VTX_FOLD_MID_UNROLL 1
#endif
constexpr int kFoldMidUnroll = VTX_FOLD_MID_UNROLL;  // column-loop unrolling of the allele pass

// shared memory per warp for allele tables of mid_cap columns (SwArgs::fold_mid_cap, sized at launch from max_hap_len)
__host__ __device__ inline size_t fold_warp_bytes(int mid_cap)
{
    size_t b = size_t(kFoldProfRows * kFoldP) * 4;               // pre-merged (forward | reverse) profile
    b += size_t(mid_cap) * 8 * 4;                                // allele-column table [column][read code]
    b += size_t(kFoldPPW) * kFoldRows * 8 + 32;                  // boundary column (forward | reverse), per read and row
    b += size_t(kFoldPPW) * kFoldCodeStride;                     // row codes, one byte per row
    return (b + 15) & ~size_t(15);
}

// junction constants: (H_f + goe + B) + (H_r + goe + B) -> H_f + H_r + B, and (E_f + B) + (E_r + B) - go -> ... + B;
// the sum of two biased halves is >= 2 * (B + goe), so adding the negative constant always carries exactly once
constexpr int kJuncH = -2 * kGoe - kBias, kJuncE = -kGapOpen - kBias;
constexpr uint32_t kJuncH2 = (uint32_t(uint16_t(int16_t(kJuncH - 1))) << 16) | uint32_t(uint16_t(int16_t(kJuncH)));
constexpr uint32_t kJuncE2 = (uint32_t(uint16_t(int16_t(kJuncE - 1))) << 16) | uint32_t(uint16_t(int16_t(kJuncE)));

// low half of a, high half of b: one LOP3 (a & 0xFFFF | b & ~0xFFFF)
__device__ __forceinline__ uint32_t lop_lo_hi(uint32_t a, uint32_t b)
{
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE2;" : "=r"(d) : "r"(a), "r"(0x0000FFFFu), "r"(b));
    return d;
}

// Main pass of one tile: forward DP over hap[0, P) in the low half, reversed DP over hap[n - P, n) in the high half.
// Returns the running maximum of the unit (not yet reduced over its lanes); parks (H + gap, E) of column P - 1 / n - P.
//   MIXED = false: cA[t] is the profile row (4 f + r, kFoldSentinel outside the read).
//   MIXED = true:  cA[t] = f << 3 | r; the forward half comes from row 4 f (16 for f = 4), the reverse half from row r
//                  (16 for r = 4).
template <bool MIXED>
__device__ __forceinline__ uint32_t fold_main_pass(const uint32_t* __restrict__ prof, const uint8_t* __restrict__ cA, int steps,
                                                   int g, uint32_t one, uint2* __restrict__ my_bnd)
{
    constexpr int C1 = kFoldC1, RS1 = kFoldP;
    uint32_t hg[C1], f[C1];
#pragma unroll
    for (int c = 0; c < C1; ++c) { hg[c] = kGOE2; f[c] = kNEG2; }
    uint32_t hg_last = kGOE2, e_last = kNEG2, diag_save = kGOE2;
    uint32_t best = kBIAS2;
    const uint32_t* lane_p = prof + g * C1;
#pragma unroll kFoldUnroll
    for (int t = 0; t < steps; ++t) {
        uint32_t hl = __shfl_up_sync(0xffffffffu, hg_last, 1, 8);
        uint32_t el = __shfl_up_sync(0xffffffffu, e_last, 1, 8);
        if (g == 0) { hl = kGOE2; el = kNEG2; }
        const uint32_t code = cA[t];
        const uint4* pa = reinterpret_cast<const uint4*>(lane_p + (MIXED ? (code >> 3) * 4 : code) * RS1);
        const uint4* pb = reinterpret_cast<const uint4*>(lane_p + ((code & 7) + 3 * (code & 4)) * RS1);   // MIXED only
        uint32_t diag = diag_save;
        diag_save = hl;
        uint32_t e = el, eg = hl, hleft = hl;
#pragma unroll
        for (int q = 0; q < C1 / 4; ++q) {
            uint32_t sv[4];
            const uint4 a4 = pa[q];
            if (MIXED) {
                const uint4 b4 = pb[q];
                sv[0] = lop_lo_hi(a4.x, b4.x); sv[1] = lop_lo_hi(a4.y, b4.y);
                sv[2] = lop_lo_hi(a4.z, b4.z); sv[3] = lop_lo_hi(a4.w, b4.w);
            } else {
                sv[0] = a4.x; sv[1] = a4.y; sv[2] = a4.z; sv[3] = a4.w;
            }
            uint32_t hh[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c = 4 * q + k;
                const uint32_t fc = __viaddmax_s16x2(f[c], kGE2, hg[c]);
                e = __viaddmax_s16x2(e, kGE2, eg);
                const uint32_t h = sw_h(diag, one, sv[k], fc, e);
                hh[k] = h;
                diag = hg[c];
                hleft = hadd(h, one, c);
                eg = hleft;
                hg[c] = hleft;
                f[c] = fc;
            }
            best = __vimax3_s16x2(best, hh[0], hh[1]);
            best = __vimax3_s16x2(best, hh[2], hh[3]);
        }
        hg_last = hleft;
        e_last = e;
        if (g == 7) my_bnd[t] = make_uint2(hleft, e);                    // columns P-1 (fwd) / n-P (rev) of row t-7
    }
    return best;
}

__global__ void __launch_bounds__(kFoldThreads, 2) vtx_k_sw_fold(const SwArgs a)
{
    constexpr int P = kFoldP, R = kFoldR, M = 8;
    constexpr int RS1 = P;                                       // 96 words: rows stay on their banks

    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int u = lane >> 3, g = lane & 7;                       // unit = read of the tile, lane within the unit
    const int mid_cap = a.fold_mid_cap;                          // allele columns of the widest window of the batch
    uint8_t* wbase = smem_raw + warp * fold_warp_bytes(mid_cap);
    uint32_t* prof = reinterpret_cast<uint32_t*>(wbase);         // [kFoldProfRows][RS1]
    uint32_t* midtab = prof + kFoldProfRows * RS1;               // [mid_cap][8]
    uint2* bnd = reinterpret_cast<uint2*>(midtab + mid_cap * 8);
    uint8_t* codes = reinterpret_cast<uint8_t*>(bnd + kFoldPPW * kFoldRows + 4);

    const uint32_t n_tiles = __ldg(a.tile_start + a.n_loci);
    uint32_t cached_locus = 0xFFFFFFFFu;
    const uint32_t tile_chunk = max(1u, min(uint32_t(kTileChunk), n_tiles / (gridDim.x * (blockDim.x >> 5) * 16u)));
    const uint32_t one = a.one;
    int mid_ref = 0, mid_alt = 0;                                // allele columns of the cached locus

    for (;;) {
        uint32_t chunk = 0;
        if (lane == 0) chunk = atomicAdd(a.tile_counter, 1u);
        chunk = __shfl_sync(0xffffffffu, chunk, 0);
        const uint32_t t_begin = chunk * tile_chunk;
        if (t_begin >= n_tiles) break;
        const uint32_t t_end = min(t_begin + tile_chunk, n_tiles);
        uint32_t locus = upper_locus(a.tile_start, a.n_loci, t_begin);
        for (uint32_t tile = t_begin; tile < t_end; ++tile) {
            while (tile >= __ldg(a.tile_start + locus + 1)) ++locus;
            const uint32_t p0 = __ldg(a.pair_start + locus) + kFoldPPW * (tile - __ldg(a.tile_start + locus));
            const uint32_t p_end = __ldg(a.pair_start + locus + 1);
            __syncwarp();
            // ---- per-locus tables ----
            if (locus != cached_locus) {
                cached_locus = locus;
                const uint8_t* rh = a.hap_bytes + __ldg(a.ref_off + locus);
                const uint8_t* ah = a.hap_bytes + __ldg(a.alt_off + locus);
                const int n_ref = int(__ldg(a.ref_len + locus)), n_alt = int(__ldg(a.alt_len + locus));
                mid_ref = n_ref - 2 * P;
                mid_alt = n_alt - 2 * P;
                for (int j = lane; j < P; j += 32) {             // both flanks are common to ref and alt (vtx_k_locus_prep)
                    const uint32_t fb = hap_code(__ldg(rh + j));
                    const uint32_t sb = hap_code(__ldg(rh + (n_ref - 1 - j)));
#pragma unroll
                    for (uint32_t p = 0; p < 16; ++p)
                        prof[p * RS1 + j] = pack2((p >> 2) == fb ? kProfMatch : kProfMis, (p & 3) == sb ? kProfMatch : kProfMis);
                    prof[16 * RS1 + j] = pack2(kProfMis, kProfMis);
                }
                // lmax <= mid_cap: the batch's max_hap_len bounds every window (vtx_k_locus_prep gives a wider one no tiles)
                const int lmax = max(mid_ref, mid_alt);
                for (int idx = lane; idx < lmax * 8; idx += 32) {
                    const int k = idx >> 3;
                    const uint32_t r = uint32_t(idx & 7);
                    const uint32_t rb = k < mid_ref ? hap_code(__ldg(rh + P + k)) : 5u;      // past the shorter allele: sentinel
                    const uint32_t ab = k < mid_alt ? hap_code(__ldg(ah + P + k)) : 5u;
                    midtab[idx] = pack2(r == rb ? kProfMatch : kProfMis, r == ab ? kProfMatch : kProfMis);
                }
            }
            // ---- row codes: the 8 lanes of a unit fill their read, one byte per row ----
            const uint32_t pair = p0 + u;
            const bool active = pair < p_end;
            int m = 0;
            uint8_t* cw = codes + u * kFoldCodeStride;
            bool mixed;                                          // some read of the tile has a base other than ACGT
            {
                const uint8_t* nib = nullptr;
                if (active) {
                    const uint32_t rd = __ldg(a.pair_read + pair);
                    m = int(__ldg(a.read_len + rd));
                    nib = a.read_nib + __ldg(a.read_off + rd);
                }
                bool other = false;
                for (int b = g; 2 * b < m; b += 8) {             // forward codes 0..4 first
                    const uint32_t by = __ldg(nib + b);
                    const uint32_t c0 = nib_code(by >> 4), c1 = nib_code(by & 0xF);
                    cw[M + 2 * b] = uint8_t(c0);
                    other |= c0 == 4;
                    if (2 * b + 1 < m) { cw[M + 2 * b + 1] = uint8_t(c1); other |= c1 == 4; }
                }
                mixed = __any_sync(0xffffffffu, other);
                __syncwarp();
                for (int i = g; 2 * i < m; i += 8) {             // then row i and its mirror m - 1 - i together, in place
                    const uint32_t x = cw[M + i], y = cw[M + m - 1 - i];
                    cw[M + i] = uint8_t(mixed ? x << 3 | y : 4 * x + y);
                    cw[M + m - 1 - i] = uint8_t(mixed ? y << 3 | x : 4 * y + x);
                }
                for (int e = g; e < kFoldCodeStride; e += 8)
                    if (e < M || e >= M + m) cw[e] = mixed ? kFoldSentinelMixed : kFoldSentinel;
            }
            int mmax = m;
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) mmax = max(mmax, __shfl_xor_sync(0xffffffffu, mmax, o));
            __syncwarp();

            // The boundary of row r lives at entry r + 7: lane 7 stores at entry t in EVERY step (no `t >= 7` test in the
            // loop); its first 7 stores are scratch.  Entries 156..158 of a read (rows 149..151) fall on the scratch entries
            // 0..2 of the next read, which that read wrote 150 steps earlier and nobody reads; the last read has 4 spare.
            uint2* my_bnd = bnd + u * kFoldRows;
            const uint2* row_bnd = my_bnd + 7;
            // =========================== main pass: forward prefix | reversed suffix ===========================
            uint32_t best = mixed ? fold_main_pass<true>(prof, cw + M - g, mmax + 7, g, one, my_bnd)
                                  : fold_main_pass<false>(prof, cw + M - g, mmax + 7, g, one, my_bnd);
#pragma unroll
            for (int o = 4; o >= 1; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(0xffffffffu, best, o));
            best = __vmaxs2(best, __byte_perm(best, 0, 0x1032));                     // both halves: max(prefix, suffix)
            __syncwarp();

            // =========================== middle: (ref, alt) over the allele columns, rows in registers ===========================
            {
                const int lmax = max(mid_ref, mid_alt), lmin = min(mid_ref, mid_alt);
                const uint32_t short_mask = mid_ref < mid_alt ? 0x0000FFFFu : 0xFFFF0000u;   // half whose allele ends first
                uint32_t hg[R], e[R], rc[R];
                const uint8_t* cf = cw + M + R * g;
                const uint32_t fwd_shift = mixed ? 3 : 2;                            // code byte -> forward code
#pragma unroll
                for (int c = 0; c < R; ++c) {
                    const int row = R * g + c;
                    uint2 b = make_uint2(kGOE2, kNEG2);
                    if (row < mmax) b = row_bnd[row];
                    hg[c] = __byte_perm(b.x, 0, 0x1010);                             // forward half, for ref and alt
                    e[c] = __byte_perm(b.y, 0, 0x1010);
                    rc[c] = (uint32_t(cf[c]) >> fwd_shift) * 4u;                     // kFoldSentinel -> 4: matches nothing
                }
                // junction of the halves in `mask`: forward row r meets reversed row m - 2 - r
                auto junction = [&](uint32_t mask) {
                    uint32_t cross = kBIAS2;
#pragma unroll
                    for (int c = 0; c < R; ++c) {
                        const int rr = m - 2 - (R * g + c);
                        uint2 b = make_uint2(kGOE2, kGOE2);                          // Hr = 0; Er such that E + Er - go < H
                        if (rr >= 0) b = row_bnd[rr];
                        const uint32_t ph = __byte_perm(b.x, 0, 0x3232), pe = __byte_perm(b.y, 0, 0x3232);
                        const uint32_t x1 = hg[c] + ph + kJuncH2;
                        const uint32_t x2 = e[c] + pe + kJuncE2;
                        cross = __vimax3_s16x2(cross, x1, x2);
                    }
                    best = __vmaxs2(best, (cross & mask) | (kBIAS2 & ~mask));
                };
                // H(row above the strip, column before the first allele column) + gap: the forward boundary of that row
                uint32_t diag_save = kGOE2;
                if (g > 0 && R * g - 1 < mmax) diag_save = __byte_perm(row_bnd[R * g - 1].x, 0, 0x1010);
                uint32_t hup_last = kGOE2, f_last = kNEG2;
                const uint8_t* tab = reinterpret_cast<const uint8_t*>(midtab) - 32 * g;
                const int steps = lmax + 7;
#pragma unroll kFoldMidUnroll
                for (int s = 0; s < steps; ++s) {
                    uint32_t hup = __shfl_up_sync(0xffffffffu, hup_last, 1, 8);
                    uint32_t fup = __shfl_up_sync(0xffffffffu, f_last, 1, 8);
                    if (g == 0) { hup = kGOE2; fup = kNEG2; }
                    const int k = s - g;                                             // allele column of this lane
                    if (k >= 0 && k < lmax) {
                        const uint8_t* trow = tab + 32 * s;                          // midtab[k][*]
                        uint32_t diag = diag_save;
                        diag_save = hup;
                        uint32_t f = fup, fg = hup, hdown = hup;
                        uint32_t hh[2];
#pragma unroll
                        for (int c = 0; c < R; ++c) {
                            const uint32_t sv = *reinterpret_cast<const uint32_t*>(trow + rc[c]);
                            const uint32_t ec = __viaddmax_s16x2(e[c], kGE2, hg[c]);          // E(r, k)
                            f = __viaddmax_s16x2(f, kGE2, fg);                                // F(r, k)
                            const uint32_t h = sw_h(diag, one, sv, ec, f);
                            hh[c & 1] = h;
                            diag = hg[c];
                            hdown = hadd(h, one, c);
                            fg = hdown;
                            hg[c] = hdown;
                            e[c] = ec;
                            if (c & 1) best = __vimax3_s16x2(best, hh[0], hh[1]);
                        }
                        if (R & 1) best = __vmaxs2(best, hh[0]);
                        hup_last = hdown;
                        f_last = f;
                        if (k == lmin - 1 && lmin != lmax) junction(short_mask);    // the shorter allele ends here (indels only)
                    }
                }
                junction(lmin != lmax ? ~short_mask : 0xFFFFFFFFu);                   // every lane has finished column lmax - 1
#pragma unroll
                for (int o = 4; o >= 1; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(0xffffffffu, best, o));
                if (active && g == 0) call_and_scatter(a, pair, best - kBIAS2);
            }
        }
    }
}

}  // namespace vtx
