// HP-1: all-pairs bit-parallel LCS length on sm_100a.
//
// Replaces CLCSBP::GetLCSBP and its scalar/AVX/AVX2/AVX512/NEON back-ends
// (reference src/lcs/lcsbp.cpp:48-368, src/lcs/lcsbp_classic.h:67-221,
// src/simd/lcsbp_avx2_intr.h:127-395) together with CSequence::ComputeBitMasks
// (src/core/sequence.cpp:190-201) behind the batch drivers of
// src/tree/AbstractTreeGenerator.hpp:131-398.  See DESIGN.md section 3 for the layout.
//
// Design (not a translation of the CPU code):
//   * Sequences are re-ordered by descending length and cut into MASK GROUPS of 32.  A group's
//     per-symbol position bit-vectors are stored lane-interleaved in 32-bit limbs ("blob"), so
//     that lane L of a warp owns sequence L of the group and every mask fetch of the warp is one
//     conflict-free LDS.128/LDS.64/LDS.32.
//   * One CTA = one tile = (mask group, a run of streamed sequences).  The blob is staged to
//     shared memory with one TMA bulk copy (cp.async.bulk + mbarrier).  Each warp streams one
//     sequence at a time: the residue is warp-uniform, each lane advances the Hyyro recurrence
//     for its own (mask sequence, streamed sequence) pair with the bit-vector X[] held in
//     registers and the carry rippling through an add.cc/addc.cc chain.  32 pairs per warp.
//   * The tile kernel computes the TRUE LCS, which is symmetric, so either sequence of a pair may
//     be the mask side.  The reference's result differs from the true LCS only when its row
//     sequence (seq0) owns an all-ones 64-bit mask word (dropped carry, lcsbp_classic.h:55-56);
//     those rows -- and rows too long for the register-resident kernel -- are recomputed by
//     k_lcs_exact, which follows the reference recurrence word for word.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <numeric>
#include <queue>
#include <tuple>

#include <cooperative_groups.h>

#include "ctx.h"

namespace fb {

constexpr int kMaskRows = 21;     // symbols 0..19 + one all-zero row shared by every other code
constexpr int kNoMatch = 20;      // device residue code for "never matches" (B, Z, X, *, padding)
constexpr int kTileWarps = 4;
constexpr int kSeqPerWarp = 8;
constexpr int kTileQ = kTileWarps * kSeqPerWarp;   // streamed sequences per tile
constexpr int kMaxNL = 64;        // limbs the register-resident kernel is instantiated for (2048 aa)

__host__ __device__ inline uint32_t blob_words(uint32_t nl) { return kMaskRows * 32u * nl; }

// word index of (symbol c, limb w, lane) inside a group's blob: limbs are grouped in fours
// (LDS.128), the remaining 1..3 limbs as LDS.32 / LDS.64 / LDS.64+LDS.32.
__host__ __device__ inline uint32_t blob_index(uint32_t nl, uint32_t c, uint32_t w, uint32_t lane)
{
    const uint32_t nq = nl / 4, tail = nl % 4;
    const uint32_t base = c * 32u * nl;
    if (w < 4 * nq) return base + ((w / 4) * 32 + lane) * 4 + (w % 4);
    const uint32_t k = w - 4 * nq;
    const uint32_t tb = base + nq * 128;
    if (tail == 1) return tb + lane;
    if (tail == 2) return tb + lane * 2 + k;
    return k < 2 ? tb + lane * 2 + k : tb + 64 + lane;
}

static uint32_t nl_for_len(uint32_t max_len)
{
    uint32_t req = (max_len + 31) / 32;
    if (req == 0) req = 1;
    if (req <= 32) return req;
    if (req <= kMaxNL) return (req + 3) / 4 * 4;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// upload-time kernels
// ------------------------------------------------------------------------------------------------

// One warp per sequence (sorted position): copy residues into the 16-byte padded device layout,
// mapping every code outside 0..19 to kNoMatch.
__global__ void k_repack(const int8_t* __restrict__ raw, const uint64_t* __restrict__ raw_off,
                         const uint32_t* __restrict__ raw_len, const uint32_t* __restrict__ perm,
                         const uint32_t* __restrict__ code_off, uint8_t* __restrict__ codes,
                         uint32_t n)
{
    const uint32_t p = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    if (p >= n) return;
    const uint32_t lane = threadIdx.x % 32;
    const uint32_t a = perm[p];
    const uint32_t len = raw_len[a];
    const int8_t* src = raw + raw_off[a];
    uint8_t* dst = codes + (size_t)code_off[p] * 16;
    const uint32_t padded = (len + 15) / 16 * 16;
    for (uint32_t i = lane; i < padded; i += 32) {
        int c = i < len ? src[i] : kNoMatch;
        dst[i] = (c >= 0 && c < 20) ? (uint8_t)c : (uint8_t)kNoMatch;
    }
}

// One CTA per mask group: build the lane-interleaved blob in shared memory, write it out.
__global__ void k_build_blob(const uint8_t* __restrict__ codes, const uint32_t* __restrict__ code_off,
                             const uint32_t* __restrict__ len_sorted,
                             const uint64_t* __restrict__ group_blob, const uint32_t* __restrict__ group_nl,
                             uint32_t* __restrict__ blob, uint32_t n)
{
    extern __shared__ uint32_t sm[];
    const uint32_t g = blockIdx.x;
    const uint32_t nl = group_nl[g];
    if (nl == 0) return;
    const uint32_t words = blob_words(nl);
    for (uint32_t i = threadIdx.x; i < words; i += blockDim.x) sm[i] = 0;
    __syncthreads();
    const uint32_t warp = threadIdx.x / 32, lane = threadIdx.x % 32, nwarps = blockDim.x / 32;
    for (uint32_t s = warp; s < 32; s += nwarps) {
        const uint32_t p = g * 32 + s;
        if (p >= n) continue;
        const uint32_t len = len_sorted[p];
        const uint8_t* src = codes + (size_t)code_off[p] * 16;
        for (uint32_t pos = lane; pos < len; pos += 32) {
            const uint32_t c = src[pos];
            if (c < 20) atomicOr(&sm[blob_index(nl, c, pos / 32, s)], 1u << (pos % 32));
        }
    }
    __syncthreads();
    uint32_t* dst = blob + group_blob[g];
    for (uint32_t i = threadIdx.x; i < words; i += blockDim.x) dst[i] = sm[i];
}

// flag[p] = 1 if some 64-bit mask word of sequence p is all ones, i.e. 64 identical matching
// residues starting at a multiple of 64 (the dropped-carry corner needs exactly that).
__global__ void k_quirky(const uint8_t* __restrict__ codes, const uint32_t* __restrict__ code_off,
                         const uint32_t* __restrict__ len_sorted, uint8_t* __restrict__ flag, uint32_t n)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t len = len_sorted[p];
    const uint8_t* src = codes + (size_t)code_off[p] * 16;
    uint8_t f = 0;
    for (uint32_t w = 0; w + 64 <= len; w += 64) {
        const uint8_t c = src[w];
        if (c >= 20) continue;
        bool all = true;
        for (uint32_t k = 1; k < 64; ++k) all &= (src[w + k] == c);
        if (all) f = 1;
    }
    flag[p] = f;
}

// ------------------------------------------------------------------------------------------------
// the tile kernel
// ------------------------------------------------------------------------------------------------

struct TileParams {
    const uint32_t* blob;
    const uint64_t* group_blob;
    const uint3* tiles;            // {group, q_begin, q_end}
    const uint8_t* codes;
    const uint32_t* code_off;
    const uint32_t* len_sorted;
    const uint32_t* perm;
    const uint32_t* refpos;        // rows mode: streamed item q -> sorted position
    void* out;
    uint64_t tri_base;
    uint32_t n;
    uint32_t row_begin, row_end;
    uint32_t ld_res;
    int elem_bytes;
    int rows_mode;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}

// One Hyyro step for 32*NL cells of one pair: X' = (X + (X & M)) | (X & ~M), true carries.
template <int NL>
__device__ __forceinline__ void lcs_step(uint32_t (&X)[NL], const uint32_t* __restrict__ row, uint32_t lane)
{
    constexpr int NQ = NL / 4, TAIL = NL % 4;
    uint32_t m[NL];
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const uint4 v = *reinterpret_cast<const uint4*>(row + (q * 32 + lane) * 4);
        m[4 * q] = v.x; m[4 * q + 1] = v.y; m[4 * q + 2] = v.z; m[4 * q + 3] = v.w;
    }
    const uint32_t* tl = row + NQ * 128;
    if (TAIL == 1) m[4 * NQ] = tl[lane];
    if (TAIL >= 2) {
        const uint2 v = *reinterpret_cast<const uint2*>(tl + lane * 2);
        m[4 * NQ] = v.x; m[4 * NQ + 1] = v.y;
    }
    if (TAIL == 3) m[4 * NQ + 2] = tl[64 + lane];

    uint32_t tb[NL], s[NL];
#pragma unroll
    for (int w = 0; w < NL; ++w) tb[w] = X[w] & m[w];
    // carry chain: one IADD3 + (NL-1) IADD3.X; the carry out of the last limb is discarded
    asm volatile("add.cc.u32 %0, %1, %2;" : "=r"(s[0]) : "r"(X[0]), "r"(tb[0]));
#pragma unroll
    for (int w = 1; w < NL; ++w)
        asm volatile("addc.cc.u32 %0, %1, %2;" : "=r"(s[w]) : "r"(X[w]), "r"(tb[w]));
#pragma unroll
    for (int w = 0; w < NL; ++w) X[w] = s[w] | (X[w] ^ tb[w]);
}

template <int NL>
__global__ void __launch_bounds__(kTileWarps * 32) k_lcs_tile(const TileParams P)
{
    extern __shared__ __align__(128) uint32_t sm[];
    __shared__ __align__(8) uint64_t bar;

    const uint3 tile = P.tiles[blockIdx.x];
    const uint32_t g = tile.x;
    constexpr uint32_t kBlobBytes = kMaskRows * 32u * NL * 4u;

    // stage the group's mask blob: one TMA bulk copy, completion on an mbarrier
    if (threadIdx.x == 0) {
        const uint32_t b = smem_u32(&bar);
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(kBlobBytes) : "memory");
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                smem_u32(sm)),
            "l"(P.blob + P.group_blob[g]), "r"(kBlobBytes), "r"(b)
            : "memory");
    }
    __syncthreads();
    {
        const uint32_t b = smem_u32(&bar);
        uint32_t done = 0;
        while (!done) {
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(b)
                : "memory");
        }
    }

    const uint32_t lane = threadIdx.x % 32, warp = threadIdx.x / 32;
    const uint32_t p = g * 32 + lane;
    const uint32_t a = p < P.n ? P.perm[p] : 0xffffffffu;

    for (uint32_t q = tile.y + warp; q < tile.z; q += kTileWarps) {
        const uint32_t sq = P.rows_mode ? P.refpos[q] : q;
        const uint32_t len = P.len_sorted[sq];
        const uint32_t* sp = reinterpret_cast<const uint32_t*>(P.codes + (size_t)P.code_off[sq] * 16);
        const uint32_t nwords = (len + 3) / 4;

        uint32_t X[NL];
#pragma unroll
        for (int w = 0; w < NL; ++w) X[w] = 0xffffffffu;

        uint32_t word = nwords ? __ldg(sp) : 0;
        for (uint32_t t = 0; t < nwords; ++t) {
            const uint32_t nxt = __ldg(sp + t + 1);    // the code buffer has 16 bytes of slack
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t c = (word >> (8 * k)) & 0xffu;
                lcs_step<NL>(X, sm + c * (32u * NL), lane);
            }
            word = nxt;
        }
        uint32_t lcs = 0;
#pragma unroll
        for (int w = 0; w < NL; ++w) lcs += __popc(~X[w]);

        if (P.rows_mode) {
            const size_t idx = (size_t)q * P.ld_res + p;
            if (P.elem_bytes == 2) static_cast<uint16_t*>(P.out)[idx] = (uint16_t)lcs;
            else static_cast<uint32_t*>(P.out)[idx] = lcs;
        } else if (a != 0xffffffffu && sq < p) {
            const uint32_t b = P.perm[sq];
            const uint32_t i = a > b ? a : b, j = a > b ? b : a;
            if (i >= P.row_begin && i < P.row_end) {
                const size_t idx = (size_t)i * (i - 1) / 2 - P.tri_base + j;
                if (P.elem_bytes == 2) static_cast<uint16_t*>(P.out)[idx] = (uint16_t)lcs;
                else static_cast<uint32_t*>(P.out)[idx] = lcs;
            }
        }
    }
}

// rows mode: res[r][sorted position] -> out[r][k] in the caller's column order
__global__ void k_gather_rows(const void* __restrict__ res, uint32_t ld_res, int res_bytes,
                              const uint32_t* __restrict__ col_ids, const uint32_t* __restrict__ invperm,
                              uint32_t n_col, void* __restrict__ out, int elem_bytes)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t r = blockIdx.y;
    if (k >= n_col) return;
    const uint32_t c = col_ids ? col_ids[k] : k;
    const size_t src = (size_t)r * ld_res + invperm[c];
    const uint32_t v = res_bytes == 2 ? static_cast<const uint16_t*>(res)[src]
                                      : static_cast<const uint32_t*>(res)[src];
    const size_t dst = (size_t)r * n_col + k;
    if (elem_bytes == 2) static_cast<uint16_t*>(out)[dst] = (uint16_t)v;
    else static_cast<uint32_t*>(out)[dst] = v;
}

// ------------------------------------------------------------------------------------------------
// exact path: the reference recurrence word for word (64-bit words, carry = (sum < V))
// ------------------------------------------------------------------------------------------------

// masks[c * nw + w], c in 0..20 (row 20 all zero), for the sequence at sorted position sp
__global__ void k_masks64(const uint8_t* __restrict__ codes, const uint32_t* __restrict__ code_off,
                          const uint32_t* __restrict__ len_sorted, uint32_t sp, uint32_t nw,
                          unsigned long long* __restrict__ masks)
{
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= kMaskRows * nw) return;
    const uint32_t c = idx / nw, w = idx % nw;
    const uint32_t len = len_sorted[sp];
    const uint8_t* src = codes + (size_t)code_off[sp] * 16;
    unsigned long long m = 0;
    if (c < 20)
        for (uint32_t b = 0; b < 64; ++b) {
            const uint32_t pos = w * 64 + b;
            if (pos < len && src[pos] == c) m |= 1ull << b;
        }
    masks[idx] = m;
}

// one thread per column; X lives in global scratch, word-major so the warp's accesses coalesce
__global__ void k_lcs_exact(const uint8_t* __restrict__ codes, const uint32_t* __restrict__ code_off,
                            const uint32_t* __restrict__ len_sorted, const uint32_t* __restrict__ invperm,
                            const unsigned long long* __restrict__ masks, uint32_t nw,
                            const uint32_t* __restrict__ col_ids, uint32_t n_col,
                            const uint32_t* __restrict__ group_nl, int only_long_cols,
                            unsigned long long* __restrict__ xs, void* __restrict__ out,
                            size_t out_base, int elem_bytes)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_col) return;
    const uint32_t col = col_ids ? col_ids[k] : k;
    const uint32_t sq = invperm[col];
    if (only_long_cols && group_nl[sq / 32] != 0) return;
    const uint32_t len = len_sorted[sq];
    const uint8_t* src = codes + (size_t)code_off[sq] * 16;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    unsigned long long* x = xs + k;
    for (uint32_t w = 0; w < nw; ++w) x[w * stride] = ~0ull;
    for (uint32_t t = 0; t < len; ++t) {
        const uint32_t c = src[t];
        if (c >= 20) continue;
        const unsigned long long* m = masks + (size_t)c * nw;
        unsigned long long carry = 0;
        for (uint32_t w = 0; w < nw; ++w) {
            const unsigned long long v = x[w * stride];
            const unsigned long long tb = v & m[w];
            const unsigned long long sum = v + tb + carry;
            carry = sum < v;
            x[w * stride] = sum | (v - tb);
        }
    }
    uint32_t lcs = 0;
    for (uint32_t w = 0; w < nw; ++w) lcs += __popcll(~x[w * stride]);
    const size_t idx = out_base + k;
    if (elem_bytes == 2) static_cast<uint16_t*>(out)[idx] = (uint16_t)lcs;
    else static_cast<uint32_t*>(out)[idx] = lcs;
}

// All special rows of a call in ONE launch: blockIdx.y = the row, its 64-bit masks are built in shared memory by the
// block itself, X[] lives in the thread (local memory, L1-resident) -- for rows of at most kExactWords * 64 residues.
// rows[r] = {sorted position of the row, out_base (element offset of the row's first result), n_col, only_long_cols}.
constexpr int kExactWords = 64;
struct ExactRow { uint32_t sp, n_col, only_long, pad; unsigned long long out_base; };
__global__ void __launch_bounds__(128) k_lcs_exact_batch(const uint8_t* __restrict__ codes, const uint32_t* __restrict__ code_off,
                                                         const uint32_t* __restrict__ len_sorted, const uint32_t* __restrict__ invperm,
                                                         const ExactRow* __restrict__ rows, const uint32_t* __restrict__ col_ids,
                                                         const uint32_t* __restrict__ group_nl, void* __restrict__ out, int elem_bytes)
{
    __shared__ unsigned long long masks[kMaskRows * kExactWords];
    const ExactRow R = rows[blockIdx.y];
    if (blockIdx.x * blockDim.x >= R.n_col) return;
    const uint32_t rlen = len_sorted[R.sp], nw = rlen ? (rlen + 63) / 64 : 1;
    const uint8_t* rsrc = codes + (size_t)code_off[R.sp] * 16;
    for (uint32_t i = threadIdx.x; i < kMaskRows * nw; i += blockDim.x) masks[i] = 0;
    __syncthreads();
    for (uint32_t pos = threadIdx.x; pos < rlen; pos += blockDim.x) {
        const uint32_t c = rsrc[pos];
        if (c < 20) atomicOr(&masks[c * nw + pos / 64], 1ull << (pos % 64));
    }
    __syncthreads();
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= R.n_col) return;
    const uint32_t col = col_ids ? col_ids[k] : k;
    const uint32_t sq = invperm[col];
    if (R.only_long && group_nl[sq / 32] != 0) return;
    const uint32_t len = len_sorted[sq];
    const uint8_t* src = codes + (size_t)code_off[sq] * 16;
    unsigned long long x[kExactWords];
    for (uint32_t w = 0; w < nw; ++w) x[w] = ~0ull;
    for (uint32_t t = 0; t < len; ++t) {
        const uint32_t c = src[t];
        if (c >= 20) continue;
        const unsigned long long* m = masks + c * nw;
        unsigned long long carry = 0;
        for (uint32_t w = 0; w < nw; ++w) {
            const unsigned long long v = x[w];
            const unsigned long long tb = v & m[w];
            const unsigned long long sum = v + tb + carry;
            carry = sum < v;
            x[w] = sum | (v - tb);
        }
    }
    uint32_t lcs = 0;
    for (uint32_t w = 0; w < nw; ++w) lcs += __popcll(~x[w]);
    const size_t idx = R.out_base + k;
    if (elem_bytes == 2) static_cast<uint16_t*>(out)[idx] = (uint16_t)lcs;
    else static_cast<uint32_t*>(out)[idx] = lcs;
}

// ------------------------------------------------------------------------------------------------
// medoid assignment: float Transform + running arg-min over the seed rows (FastTree.cpp:309-324)
// ------------------------------------------------------------------------------------------------

// Transform<float, Distance> (AbstractTreeGenerator.hpp:28-82) with the host-computed (float) pow(i, 0.75) table;
// IEEE division, so the result is the host's bit for bit.
__device__ __forceinline__ float transform_f32(int kind, uint32_t lcs, uint32_t len1, uint32_t len2,
                                               const float* __restrict__ pow075, float never)
{
    if (kind == 2) return __fdiv_rn((float)lcs, (float)(len1 < len2 ? len1 : len2));
    const uint32_t indel_i = len1 + len2 - 2 * lcs;
    if (!lcs) return never;                                  // (float) nextafter((double) FLT_MAX, 0) == FLT_MAX
    if (kind == 0) return __fdiv_rn(pow075[indel_i], (float)lcs);
    return __fdiv_rn((float)indel_i, (float)lcs);
}

__global__ void k_assign(const void* __restrict__ lcs, int elem_bytes, uint32_t n, uint32_t n_seeds,
                         const uint32_t* __restrict__ seed_ids, const uint32_t* __restrict__ lens,
                         const float* __restrict__ pow075, int kind, float never,
                         uint32_t* __restrict__ assign, float* __restrict__ mind)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t lj = lens[j];
    float best = 0.f;
    uint32_t a = 0;
    for (uint32_t k = 0; k < n_seeds; ++k) {
        const size_t at = (size_t)k * n + j;
        const uint32_t l = elem_bytes == 2 ? static_cast<const uint16_t*>(lcs)[at] : static_cast<const uint32_t*>(lcs)[at];
        const float d = transform_f32(kind, l, lens[seed_ids[k]], lj, pow075, never);
        if (k == 0 || d < best) { best = d; a = k; }
    }
    assign[j] = a;
    mind[j] = best;
}

// Sharded form: only the sequences whose mask group lies in [g_begin, g_end) are answered; the result is packed as
// (float bits of the distance << 32) | seed index so that an element-wise MIN over the shards (one all-reduce) assembles
// the complete assignment -- distances are >= 0, so their bit patterns order like the values, and among equal distances
// the lowest seed index wins, which is what the strict < of the sequential loop does.  Unanswered entries hold INT64_MAX.
__global__ void k_assign_packed(const void* __restrict__ lcs, int elem_bytes, uint32_t n, uint32_t n_seeds,
                                const uint32_t* __restrict__ seed_ids, const uint32_t* __restrict__ lens,
                                const float* __restrict__ pow075, int kind, float never,
                                const uint32_t* __restrict__ invperm, uint32_t g_begin, uint32_t g_end,
                                long long* __restrict__ packed)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t g = invperm[j] / 32;
    if (g < g_begin || g >= g_end) { packed[j] = 0x7fffffffffffffffll; return; }
    const uint32_t lj = lens[j];
    float best = 0.f;
    uint32_t a = 0;
    for (uint32_t k = 0; k < n_seeds; ++k) {
        const size_t at = (size_t)k * n + j;
        const uint32_t l = elem_bytes == 2 ? static_cast<const uint16_t*>(lcs)[at] : static_cast<const uint32_t*>(lcs)[at];
        const float d = transform_f32(kind, l, lens[seed_ids[k]], lj, pow075, never);
        if (k == 0 || d < best) { best = d; a = k; }
    }
    packed[j] = (long long)(((unsigned long long)__float_as_uint(best) << 32) | a);
}

// ------------------------------------------------------------------------------------------------
// MST-Prim vertex loop (MSTPrim<>::run_view, MSTPrim.cpp:280-549) on the resident LCS triangle
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ double transform_f64(int kind, uint32_t lcs, uint32_t len1, uint32_t len2,
                                                const double* __restrict__ pow075, double never)
{
    const uint32_t indel_i = len1 + len2 - 2 * lcs;
    if (!lcs) return never;                                  // nextafter(DBL_MAX, 0)
    if (kind == 0) return __ddiv_rn(pow075[indel_i], (double)lcs);
    return __ddiv_rn((double)indel_i, (double)lcs);
}

struct PrimState {                 // per sequence: best known connection to the tree
    double dist;
    unsigned long long key;        // ~ids_to_uint64(from, j)  (MSTPrim.h:432-439)
};

// Cooperative grid (one block per SM, all co-resident): per step every thread relaxes its own unvisited sequences
// against the current vertex (one triangle lookup + one pow-table lookup each, all independent), blocks publish their
// best (dist, key) pair, ONE grid-wide barrier, and every block reduces the published candidates itself, so all
// blocks agree on the next vertex without a second barrier.  Candidate slots are double-buffered by step parity.
// tri: true-LCS triangle in caller order; side rows hold the row-oriented values of the sequences whose LCS is
// orientation dependent (dropped-carry corner): side_idx[v] = row in `side` or -1.
struct PrimCand {
    double dist;
    unsigned long long key;
    int id;
    int pad;
};

__global__ void __launch_bounds__(1024) k_prim(const void* __restrict__ tri, int eb, uint32_t n,
                                               const uint32_t* __restrict__ lens, const double* __restrict__ pow075,
                                               int kind, double never, const int* __restrict__ side_idx,
                                               const uint32_t* __restrict__ side, PrimState* __restrict__ st,
                                               unsigned char* __restrict__ visited, PrimCand* __restrict__ cand,
                                               int* __restrict__ out_from, int* __restrict__ out_to,
                                               double* __restrict__ out_dist, int* __restrict__ order)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double sh_d[32];
    __shared__ unsigned long long sh_k[32];
    __shared__ int sh_id[32];
    __shared__ int sh_v;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t gtid = blockIdx.x * blockDim.x + tid, gthreads = gridDim.x * blockDim.x;
    const uint32_t nblk = gridDim.x;
    auto better = [](double d, unsigned long long k, int id, double bd, unsigned long long bk, int bid) {
        return id >= 0 && (bid < 0 || d < bd || (d == bd && k < bk));
    };
    for (uint32_t j = gtid; j < n; j += gthreads) {
        st[j].dist = 1.7976931348623157e308;        // numeric_limits<double>::max()
        st[j].key = 0;
        visited[j] = j == 0;
        order[j] = j == 0 ? 0 : (int)n;
    }
    // the first sequence a thread owns lives in registers (with n <= gridDim.x * 1024 that is all of them)
    const bool has0 = gtid < n;
    const uint32_t len0 = has0 ? lens[gtid] : 0;
    bool vis0 = gtid == 0;
    double d0 = 1.7976931348623157e308;
    unsigned long long k0 = 0;
    uint32_t v = 0;
    grid.sync();
    for (uint32_t step = 1; step < n; ++step) {
        const uint32_t lv = lens[v];
        const int sv = side_idx[v];
        double bd = 0.0;
        unsigned long long bk = 0;
        int bid = -1;
        auto lookup = [&](uint32_t j) -> uint32_t {
            if (sv >= 0) return side[(size_t)sv * n + j];
            const uint32_t hi = v > j ? v : j, lo = v > j ? j : v;
            const size_t at = (size_t)hi * (hi - 1) / 2 + lo;
            return eb == 2 ? static_cast<const uint16_t*>(tri)[at] : static_cast<const uint32_t*>(tri)[at];
        };
        // MSTPrim.cpp:450-467: a candidate is only computed when the distance it would have with LCS = the shorter length
        // does not exceed its current one.  A no-op for a true LCS (<= the shorter length); with the dropped-carry corner the
        // reference's LCS can be larger, and then the skip decides whether the candidate is relaxed.
        if (has0 && !vis0) {
            const uint32_t j = gtid;
            const bool tried = transform_f64(kind, lv < len0 ? lv : len0, lv, len0, pow075, never) <= d0;
            const double d = tried ? transform_f64(kind, lookup(j), lv, len0, pow075, never) : 1.7976931348623157e308;
            if (tried && d <= d0) {
                const unsigned long long a = v < j ? v : j, b = v < j ? j : v;
                const unsigned long long k = ~((a << 32) + b);
                if (d < d0 || k < k0) { d0 = d; k0 = k; }                                  // pair <, given d <= d0
            }
            bd = d0; bk = k0; bid = (int)j;
        }
        for (uint32_t j = gtid + gthreads; j < n; j += gthreads) {                         // only when n > grid size
            if (visited[j]) continue;
            double cd = st[j].dist;
            unsigned long long ck = st[j].key;
            const uint32_t lj = lens[j];
            const bool tried = transform_f64(kind, lv < lj ? lv : lj, lv, lj, pow075, never) <= cd;
            const double d = tried ? transform_f64(kind, lookup(j), lv, lj, pow075, never) : 1.7976931348623157e308;
            if (tried && d <= cd) {
                const unsigned long long a = v < j ? v : j, b = v < j ? j : v;
                const unsigned long long k = ~((a << 32) + b);
                if (d < cd || k < ck) { cd = d; ck = k; st[j].dist = cd; st[j].key = ck; }
            }
            if (better(cd, ck, (int)j, bd, bk, bid)) { bd = cd; bk = ck; bid = (int)j; }
        }
        // block-wide minimum of (dist, key) ...
        for (int o = 16; o; o >>= 1) {
            const double od = __shfl_xor_sync(0xffffffffu, bd, o);
            const unsigned long long ok = __shfl_xor_sync(0xffffffffu, bk, o);
            const int oid = __shfl_xor_sync(0xffffffffu, bid, o);
            if (better(od, ok, oid, bd, bk, bid)) { bd = od; bk = ok; bid = oid; }
        }
        if (lane == 0) { sh_d[warp] = bd; sh_k[warp] = bk; sh_id[warp] = bid; }
        __syncthreads();
        if (warp == 0) {
            const uint32_t nw = blockDim.x / 32;
            bd = lane < nw ? sh_d[lane] : 0.0; bk = lane < nw ? sh_k[lane] : 0; bid = lane < nw ? sh_id[lane] : -1;
            for (int o = 16; o; o >>= 1) {
                const double od = __shfl_xor_sync(0xffffffffu, bd, o);
                const unsigned long long ok = __shfl_xor_sync(0xffffffffu, bk, o);
                const int oid = __shfl_xor_sync(0xffffffffu, bid, o);
                if (better(od, ok, oid, bd, bk, bid)) { bd = od; bk = ok; bid = oid; }
            }
            if (lane == 0) {
                PrimCand c; c.dist = bd; c.key = bk; c.id = bid; c.pad = 0;
                cand[(step & 1) * nblk + blockIdx.x] = c;
            }
        }
        // ... one grid barrier, then every block reduces the published candidates for itself
        grid.sync();
        if (warp == 0) {
            bd = 0.0; bk = 0; bid = -1;
            for (uint32_t b = lane; b < nblk; b += 32) {
                const PrimCand c = cand[(step & 1) * nblk + b];
                if (better(c.dist, c.key, c.id, bd, bk, bid)) { bd = c.dist; bk = c.key; bid = c.id; }
            }
            for (int o = 16; o; o >>= 1) {
                const double od = __shfl_xor_sync(0xffffffffu, bd, o);
                const unsigned long long ok = __shfl_xor_sync(0xffffffffu, bk, o);
                const int oid = __shfl_xor_sync(0xffffffffu, bid, o);
                if (better(od, ok, oid, bd, bk, bid)) { bd = od; bk = ok; bid = oid; }
            }
            if (lane == 0) {
                sh_v = bid;
                if (blockIdx.x == 0) {
                    const unsigned long long packed = ~bk;             // uint64_to_id (MSTPrim.h:441-450)
                    const int id1 = (int)(packed >> 32), id2 = (int)(packed & 0xffffffffull);
                    out_from[step - 1] = id1 < id2 ? id1 : id2;
                    out_to[step - 1] = id1 < id2 ? id2 : id1;
                    out_dist[step - 1] = bd;
                    order[bid] = (int)step;
                }
                if ((uint32_t)bid >= gthreads && (uint32_t)bid % gthreads / blockDim.x == blockIdx.x) visited[bid] = 1;   // its owner block
            }
        }
        __syncthreads();
        v = (uint32_t)sh_v;
        if (v == gtid) vis0 = true;
    }
}

// ------------------------------------------------------------------------------------------------
// Parallel MST (Boruvka rounds) under MSTPrim's edge order.
//
// MSTPrim relaxes and elects with the pair (distance, ~ids_to_uint64(min id, max id)) compared lexicographically
// (MSTPrim.cpp:366-386, 492-503).  The key is unique per edge, so the pairs are a strict total order and the minimum
// spanning tree under it is unique: any algorithm finds the edges Prim finds.  What Prim adds is the visiting order
// from vertex 0, and that can be replayed on the n-1 tree edges alone (at every step Prim takes the smallest edge
// leaving the visited set, which is a tree edge).  So: distances once into a float64 triangle, then log2(n) rounds in
// which every vertex finds its smallest edge into another component -- two streaming passes over the triangle, rows
// and columns, both coalesced -- while the host merges components (union-find over n entries) and finally replays
// Prim's order with a heap.  Used when no sequence has orientation-dependent LCS values (the dropped-carry corner);
// otherwise the sequential loop above runs.  famsa_b200/mst.py + tests/test_mst_host.py pin the argument on the CPU.
// ------------------------------------------------------------------------------------------------
struct EdgeMin {
    double d;
    unsigned long long k;
};
__device__ __forceinline__ bool edge_less(double d, unsigned long long k, double bd, unsigned long long bk) { return d < bd || (d == bd && k < bk); }
__device__ __forceinline__ unsigned long long edge_key_dev(uint32_t a, uint32_t b)
{
    const unsigned long long lo = a < b ? a : b, hi = a < b ? b : a;
    return ~((lo << 32) + hi);
}
constexpr double kEdgeNone = __builtin_huge_val();      // +inf: no candidate (distances are finite)

// one block per row i: distances of (i, j), j < i  (Transform<double, Distance>, AbstractTreeGenerator.hpp:28-82)
__global__ void __launch_bounds__(256) k_mst_dist(const void* __restrict__ tri, int eb, uint32_t n, const uint32_t* __restrict__ lens,
                                                  const double* __restrict__ pow075, int kind, double never, double* __restrict__ out)
{
    const uint32_t i = blockIdx.x + 1;
    const size_t base = (size_t)i * (i - 1) / 2;
    const uint32_t li = lens[i];
    for (uint32_t j = threadIdx.x; j < i; j += blockDim.x) {
        const uint32_t l = eb == 2 ? static_cast<const uint16_t*>(tri)[base + j] : static_cast<const uint32_t*>(tri)[base + j];
        out[base + j] = transform_f64(kind, l, li, lens[j], pow075, never);
    }
}

__device__ __forceinline__ void block_edge_min(double& d, unsigned long long& k)
{
    __shared__ double sd[32];
    __shared__ unsigned long long sk[32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, d, o);
        const unsigned long long ok = __shfl_xor_sync(0xffffffffu, k, o);
        if (edge_less(od, ok, d, k)) { d = od; k = ok; }
    }
    if (lane == 0) { sd[warp] = d; sk[warp] = k; }
    __syncthreads();
    if (warp == 0) {
        const uint32_t nw = blockDim.x / 32;
        d = lane < nw ? sd[lane] : kEdgeNone; k = lane < nw ? sk[lane] : 0;
        for (int o = 16; o; o >>= 1) {
            const double od = __shfl_xor_sync(0xffffffffu, d, o);
            const unsigned long long ok = __shfl_xor_sync(0xffffffffu, k, o);
            if (edge_less(od, ok, d, k)) { d = od; k = ok; }
        }
    }
}

// row pass: vertex i against its lower neighbours j < i in other components
__global__ void __launch_bounds__(256) k_mst_rows(const double* __restrict__ dtri, uint32_t n, const uint32_t* __restrict__ comp,
                                                  EdgeMin* __restrict__ best)
{
    const uint32_t i = blockIdx.x;
    const size_t base = (size_t)i * (i ? i - 1 : 0) / 2;
    const uint32_t ci = comp[i];
    double d = kEdgeNone;
    unsigned long long k = 0;
    for (uint32_t j = threadIdx.x; j < i; j += blockDim.x) {
        if (comp[j] == ci) continue;
        const double dj = dtri[base + j];
        const unsigned long long kj = edge_key_dev(i, j);
        if (edge_less(dj, kj, d, k)) { d = dj; k = kj; }
    }
    block_edge_min(d, k);
    if (threadIdx.x == 0) { best[i].d = d; best[i].k = k; }
}

// column pass: vertex j against its upper neighbours i > j; block = 32 columns x a chunk of kMstChunk rows, every row
// contributes a coalesced 256-byte segment.  part[chunk][j] receives the chunk's minimum.
constexpr uint32_t kMstChunk = 1024;
__global__ void __launch_bounds__(256) k_mst_cols(const double* __restrict__ dtri, uint32_t n, const uint32_t* __restrict__ comp,
                                                  EdgeMin* __restrict__ part)
{
    __shared__ double sd[8][32];
    __shared__ unsigned long long sk[8][32];
    const uint32_t x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const uint32_t j = blockIdx.x * 32 + x;
    const uint32_t r0 = blockIdx.y * kMstChunk, r1 = r0 + kMstChunk < n ? r0 + kMstChunk : n;
    double d = kEdgeNone;
    unsigned long long k = 0;
    if (j < n) {
        const uint32_t cj = comp[j];
        uint32_t i = r0 + y;
        if (i <= j) i += ((j + 1 - i) + 7) / 8 * 8;                 // first row of this thread's residue class above j
        for (; i < r1; i += 8) {
            if (comp[i] == cj) continue;
            const double di = dtri[(size_t)i * (i - 1) / 2 + j];
            const unsigned long long ki = edge_key_dev(i, j);
            if (edge_less(di, ki, d, k)) { d = di; k = ki; }
        }
    }
    sd[y][x] = d; sk[y][x] = k;
    __syncthreads();
    if (y == 0 && j < n) {
        for (int q = 1; q < 8; ++q)
            if (edge_less(sd[q][x], sk[q][x], d, k)) { d = sd[q][x]; k = sk[q][x]; }
        part[(size_t)blockIdx.y * n + j].d = d;
        part[(size_t)blockIdx.y * n + j].k = k;
    }
}

// best[j] = min(best[j] (row pass), part[*][j])
__global__ void __launch_bounds__(256) k_mst_combine(uint32_t n, uint32_t n_chunks, const EdgeMin* __restrict__ part, EdgeMin* __restrict__ best)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double d = best[j].d;
    unsigned long long k = best[j].k;
    for (uint32_t c = j / kMstChunk; c < n_chunks; ++c) {            // chunks that end at or below row j hold nothing for j
        const EdgeMin e = part[(size_t)c * n + j];
        if (edge_less(e.d, e.k, d, k)) { d = e.d; k = e.k; }
    }
    best[j].d = d; best[j].k = k;
}


// ------------------------------------------------------------------------------------------------
// UPGMA on the resident triangle (UPGMA<>::computeTree, UPGMA.cpp:114-295; SURVEY 8f-1).
//
// The reference's agglomeration is MUSCLE's nearest-neighbour-cache UPGMA: every live row keeps (MinDist, NearestNeighbor);
// an iteration picks the live row with the smallest MinDist (first such row), merges it with its cached neighbour,
// overwrites the row of the left child with the averaged distances and re-labels -- but does not re-evaluate -- the
// caches of the other rows (UPGMA.cpp:229-262: a row whose neighbour was the right child now points at the left child
// and keeps the OLD distance).  Results depend on that, so it is reproduced step for step; what is parallel is the inside
// of a step: both scans (arg-min over the rows, update + arg-min over the new row) are grid-wide reductions of packed
// (float bits, index) words -- distances are >= 0, so unsigned order is value order and ties go to the lowest index,
// exactly what the strict < of the sequential scans does.  One cooperative kernel, two grid barriers per merge.
// ------------------------------------------------------------------------------------------------
constexpr float kUpgmaBig = 1e29f;                                  // UPGMA::BIG_DIST (UPGMA.h:82)
constexpr unsigned long long kNoCand = ~0ull;

// Transform<float, Distance> of every pair: the float triangle computeDistances fills (UPGMA.cpp:75-109)
__global__ void __launch_bounds__(256) k_upgma_dist(const void* __restrict__ tri, int eb, uint32_t n, const uint32_t* __restrict__ lens,
                                                    const float* __restrict__ pow075, int kind, float never, float* __restrict__ out)
{
    const uint32_t i = blockIdx.x + 1;
    const size_t base = (size_t)i * (i - 1) / 2;
    const uint32_t li = lens[i];
    for (uint32_t j = threadIdx.x; j < i; j += blockDim.x) {
        const uint32_t l = eb == 2 ? static_cast<const uint16_t*>(tri)[base + j] : static_cast<const uint32_t*>(tri)[base + j];
        out[base + j] = transform_f32(kind, l, li, lens[j], pow075, never);
    }
}

__device__ __forceinline__ unsigned long long pack_cand(float d, uint32_t j) { return ((unsigned long long)__float_as_uint(d) << 32) | j; }
__device__ __forceinline__ unsigned long long block_min_u64(unsigned long long v, unsigned long long* sh)
{
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o; o >>= 1) { const unsigned long long x = __shfl_xor_sync(0xffffffffu, v, o); v = x < v ? x : v; }
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    if (warp == 0) {
        const uint32_t nw = blockDim.x / 32;
        v = lane < nw ? sh[lane] : kNoCand;
        for (int o = 16; o; o >>= 1) { const unsigned long long x = __shfl_xor_sync(0xffffffffu, v, o); v = x < v ? x : v; }
    }
    return v;                                                        // valid in warp 0
}

// initial (MinDist, NearestNeighbor) of every row (UPGMA.cpp:183-203): partners are met in ascending index order and
// only a strictly smaller distance replaces the cache, so the cache is the arg-min with the lowest partner on ties
__global__ void __launch_bounds__(256) k_upgma_init(const float* __restrict__ dist, uint32_t n, float* __restrict__ mind, uint32_t* __restrict__ nn,
                                                    int* __restrict__ node)
{
    __shared__ unsigned long long sh[32];
    const uint32_t r = blockIdx.x;
    unsigned long long best = kNoCand;
    const size_t base = (size_t)r * (r ? r - 1 : 0) / 2;
    for (uint32_t p = threadIdx.x; p < n; p += blockDim.x) {
        if (p == r) continue;
        const float d = p < r ? dist[base + p] : dist[(size_t)p * (p - 1) / 2 + r];
        if (d < kUpgmaBig) { const unsigned long long c = pack_cand(d, p); best = c < best ? c : best; }
    }
    best = block_min_u64(best, sh);
    if (threadIdx.x == 0) {
        mind[r] = best == kNoCand ? kUpgmaBig : __uint_as_float((unsigned)(best >> 32));
        nn[r] = best == kNoCand ? 0x7fffffffu : (uint32_t)best;
        node[r] = (int)r;
    }
}

template <bool MODIFIED>
__global__ void __launch_bounds__(1024) k_upgma(float* __restrict__ dist, uint32_t n, float* __restrict__ mind, uint32_t* __restrict__ nn,
                                                int* __restrict__ node, unsigned long long* __restrict__ cand, int* __restrict__ out_tree,
                                                int* __restrict__ status)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned long long sh[32];
    __shared__ unsigned long long sh_pick;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t gtid = blockIdx.x * blockDim.x + tid, gthreads = gridDim.x * blockDim.x, nblk = gridDim.x;
    auto tri_at = [](uint32_t a, uint32_t b) -> size_t { const uint32_t hi = a > b ? a : b, lo = a > b ? b : a; return (size_t)hi * (hi - 1) / 2 + lo; };
    // every block reduces the nblk published candidates of buffer `buf` for itself: all agree without a second barrier
    auto gather = [&](uint32_t buf) -> unsigned long long {
        unsigned long long v = kNoCand;
        if (warp == 0) {
            for (uint32_t b = lane; b < nblk; b += 32) { const unsigned long long x = cand[(size_t)buf * nblk + b]; v = x < v ? x : v; }
            for (int o = 16; o; o >>= 1) { const unsigned long long x = __shfl_xor_sync(0xffffffffu, v, o); v = x < v ? x : v; }
            if (lane == 0) sh_pick = v;
        }
        __syncthreads();
        return sh_pick;
    };
    // what the previous merge changed (row L got a new cache, row R died): every thread knows it from the reductions, so the
    // scan below does not have to wait for thread 0's writes to become visible -- two grid barriers per merge, not three
    uint32_t pL = 0xffffffffu, pR = 0xffffffffu;
    unsigned long long pN = kNoCand;
    for (uint32_t it = 0; it + 1 < n; ++it) {
        // ---- the live row with the smallest cached distance (first such row)
        unsigned long long best = kNoCand;
        for (uint32_t j = gtid; j < n; j += gthreads) {
            if (j == pR) continue;
            float d;
            if (j == pL) { if (pN == kNoCand) continue; d = __uint_as_float((unsigned)(pN >> 32)); }
            else { if (node[j] < 0) continue; d = mind[j]; }
            if (d < kUpgmaBig) { const unsigned long long c = pack_cand(d, j); best = c < best ? c : best; }
        }
        best = block_min_u64(best, sh);
        if (tid == 0) cand[(size_t)0 * nblk + blockIdx.x] = best;
        grid.sync();
        const unsigned long long pick = gather(0);
        if (pick == kNoCand) { if (gtid == 0) *status = 1; return; }     // no finite distance left: the reference would index out of range
        const uint32_t L = (uint32_t)pick, R = nn[L];
        // ---- distances to the new node overwrite the row of L; the arg-min of the new row becomes L's cache
        unsigned long long nbest = kNoCand;
        for (uint32_t j = gtid; j < n; j += gthreads) {
            if (j == L || j == R || node[j] < 0) continue;
            const size_t vL = tri_at(L, j), vR = tri_at(R, j);
            const float dL = dist[vL], dR = dist[vR];
            const float nd = MODIFIED ? __fadd_rn(__fmul_rn(0.05f, __fadd_rn(dL, dR)), __fmul_rn(0.9f, dR < dL ? dR : dL))
                                      : __fmul_rn(__fadd_rn(dL, dR), 0.5f);
            if (nn[j] == R) nn[j] = L;
            dist[vL] = nd;
            if (nd < kUpgmaBig) { const unsigned long long c = pack_cand(nd, j); nbest = c < nbest ? c : nbest; }
        }
        nbest = block_min_u64(nbest, sh);
        if (tid == 0) cand[(size_t)1 * nblk + blockIdx.x] = nbest;
        grid.sync();
        const unsigned long long npick = gather(1);
        if (gtid == 0) {
            out_tree[2 * it] = node[L];
            out_tree[2 * it + 1] = node[R];
            node[L] = (int)(n + it);
            nn[L] = npick == kNoCand ? 0x7fffffffu : (uint32_t)npick;
            mind[L] = npick == kNoCand ? kUpgmaBig : __uint_as_float((unsigned)(npick >> 32));
            node[R] = -1;                                                // (visible to everybody after the next barrier)
        }
        pL = L; pR = R; pN = npick;
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------

int DevBuf::reserve(size_t bytes)
{
    if (bytes <= cap) return FAMSA_OK;
    release();
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        p = nullptr;
        set_error(std::string("cudaMalloc(") + std::to_string(want) + ") failed: " + cudaGetErrorString(e));
        return FAMSA_E_NOMEM;
    }
    cap = want;
    return FAMSA_OK;
}
void DevBuf::release()
{
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
}

template <int NL>
static int launch_tile(famsa_ctx* ctx, const TileParams& P, uint32_t n_tiles, cudaStream_t st)
{
    const size_t smem = (size_t)blob_words(NL) * 4;
    if (!(ctx->lcs.tile_configured >> (NL - 1) & 1)) {
        FB_CUDA(cudaFuncSetAttribute(k_lcs_tile<NL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ctx->lcs.tile_configured |= 1ull << (NL - 1);
    }
    k_lcs_tile<NL><<<n_tiles, kTileWarps * 32, smem, st>>>(P);
    FB_CUDA(cudaGetLastError());
    ctx->launches++;
    return FAMSA_OK;
}

static int launch_tile_nl(famsa_ctx* ctx, uint32_t nl, const TileParams& P, uint32_t n_tiles, cudaStream_t st)
{
    switch (nl) {
#define FB_CASE(N) case N: return launch_tile<N>(ctx, P, n_tiles, st);
        FB_CASE(1) FB_CASE(2) FB_CASE(3) FB_CASE(4) FB_CASE(5) FB_CASE(6) FB_CASE(7) FB_CASE(8)
        FB_CASE(9) FB_CASE(10) FB_CASE(11) FB_CASE(12) FB_CASE(13) FB_CASE(14) FB_CASE(15) FB_CASE(16)
        FB_CASE(17) FB_CASE(18) FB_CASE(19) FB_CASE(20) FB_CASE(21) FB_CASE(22) FB_CASE(23) FB_CASE(24)
        FB_CASE(25) FB_CASE(26) FB_CASE(27) FB_CASE(28) FB_CASE(29) FB_CASE(30) FB_CASE(31) FB_CASE(32)
        FB_CASE(36) FB_CASE(40) FB_CASE(44) FB_CASE(48) FB_CASE(52) FB_CASE(56) FB_CASE(60) FB_CASE(64)
#undef FB_CASE
    default:
        set_error("internal: no tile kernel for nl=" + std::to_string(nl));
        return FAMSA_E_INVALID;
    }
}

static int lcs_upload_impl(famsa_ctx* ctx, const int8_t* codes, const uint64_t* offsets, const uint32_t* lens, uint32_t n);

// A failed upload leaves the context without a sequence set (n = 0) rather than with a half-replaced one.
int lcs_upload(famsa_ctx* ctx, const int8_t* codes, const uint64_t* offsets, const uint32_t* lens, uint32_t n)
{
    const int rc = lcs_upload_impl(ctx, codes, offsets, lens, n);
    if (rc != FAMSA_OK) {
        LcsState& S = ctx->lcs;
        S.n = S.n_groups = 0;
        S.max_len = 0;
        S.groups.clear(); S.h_quirky.clear(); S.h_long.clear();
    }
    return rc;
}

static int lcs_upload_impl(famsa_ctx* ctx, const int8_t* codes, const uint64_t* offsets, const uint32_t* lens, uint32_t n)
{
    LcsState& S = ctx->lcs;
    cudaStream_t st = ctx->stream;
    S.n = n;
    S.n_groups = (n + 31) / 32;
    S.h_quirky.clear();
    S.h_long.clear();
    if (n == 0) return FAMSA_OK;
    const uint32_t npad = S.n_groups * 32;

    // length-descending order (stable), as CFAMSA::sortAndExtendSequences leaves it (msa.cpp:245-279)
    S.h_perm.resize(n);
    std::iota(S.h_perm.begin(), S.h_perm.end(), 0u);
    S.identity_perm = std::is_sorted(lens, lens + n, [](uint32_t x, uint32_t y) { return x > y; });
    if (!S.identity_perm)
        std::stable_sort(S.h_perm.begin(), S.h_perm.end(), [&](uint32_t x, uint32_t y) { return lens[x] > lens[y]; });
    S.h_invperm.resize(n);
    for (uint32_t p = 0; p < n; ++p) S.h_invperm[S.h_perm[p]] = p;

    S.h_len_sorted.assign(npad, 0);
    std::vector<uint32_t> code_off(npad + 1, 0);
    uint64_t units = 0, raw_lo = UINT64_MAX, raw_hi = 0;
    S.max_len = 0;
    for (uint32_t p = 0; p < n; ++p) {
        const uint32_t a = S.h_perm[p];
        S.h_len_sorted[p] = lens[a];
        S.max_len = std::max(S.max_len, lens[a]);
        code_off[p] = (uint32_t)units;
        units += (lens[a] + 15) / 16;
        if (units > 0xfffffff0ull) { set_error("sequence set too large (> 64 GiB of residues)"); return FAMSA_E_INVALID; }
        if (lens[a]) { raw_lo = std::min(raw_lo, offsets[a]); raw_hi = std::max(raw_hi, offsets[a] + lens[a]); }
    }
    for (uint32_t p = n; p <= npad; ++p) code_off[p] = (uint32_t)units;
    if (raw_lo == UINT64_MAX) raw_lo = raw_hi = 0;

    S.groups.assign(S.n_groups, LcsGroupInfo{0, 0});
    std::vector<uint64_t> group_blob(S.n_groups);
    std::vector<uint32_t> group_nl(S.n_groups);
    uint64_t words = 0;
    uint32_t max_nl = 1;
    for (uint32_t g = 0; g < S.n_groups; ++g) {
        const uint32_t nl = nl_for_len(S.h_len_sorted[g * 32]);   // first of the group is the longest
        S.groups[g].nl = nl;
        S.groups[g].blob_word = words;
        group_blob[g] = words;
        group_nl[g] = nl;
        words += blob_words(nl);
        max_nl = std::max(max_nl, nl);
        if (nl == 0)
            for (uint32_t p = g * 32; p < std::min(n, g * 32 + 32); ++p) S.h_long.push_back(S.h_perm[p]);
    }

    // shifted offsets so that only the used byte range of the caller's buffer is copied
    std::vector<uint64_t> off_shift(n);
    for (uint32_t a = 0; a < n; ++a) off_shift[a] = lens[a] ? offsets[a] - raw_lo : 0;

    FB_TRY(S.d_perm.reserve(sizeof(uint32_t) * n));
    FB_TRY(S.d_invperm.reserve(sizeof(uint32_t) * n));
    FB_TRY(S.d_len_sorted.reserve(sizeof(uint32_t) * npad));
    FB_TRY(S.d_code_off.reserve(sizeof(uint32_t) * (npad + 1)));
    FB_TRY(S.d_codes.reserve(units * 16 + 64));
    FB_TRY(S.d_blob.reserve(std::max<uint64_t>(words, 1) * 4));
    FB_TRY(S.d_group_blob.reserve(sizeof(uint64_t) * S.n_groups + sizeof(uint32_t) * S.n_groups));
    FB_TRY(S.d_raw_codes.reserve(raw_hi - raw_lo + 16));
    FB_TRY(S.d_raw_off.reserve(sizeof(uint64_t) * n));
    FB_TRY(S.d_raw_len.reserve(sizeof(uint32_t) * n));
    FB_TRY(S.d_flags.reserve(n));

    uint32_t* d_group_nl = reinterpret_cast<uint32_t*>(S.d_group_blob.as<uint64_t>() + S.n_groups);
    FB_CUDA(cudaMemcpyAsync(S.d_perm.p, S.h_perm.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemcpyAsync(S.d_invperm.p, S.h_invperm.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemcpyAsync(S.d_len_sorted.p, S.h_len_sorted.data(), sizeof(uint32_t) * npad, cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemcpyAsync(S.d_code_off.p, code_off.data(), sizeof(uint32_t) * (npad + 1), cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemcpyAsync(S.d_group_blob.p, group_blob.data(), sizeof(uint64_t) * S.n_groups, cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemcpyAsync(d_group_nl, group_nl.data(), sizeof(uint32_t) * S.n_groups, cudaMemcpyHostToDevice, st));
    if (raw_hi > raw_lo)
        FB_CUDA(cudaMemcpyAsync(S.d_raw_codes.p, codes + raw_lo, raw_hi - raw_lo, cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemcpyAsync(S.d_raw_off.p, off_shift.data(), sizeof(uint64_t) * n, cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemcpyAsync(S.d_raw_len.p, lens, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemsetAsync(S.d_codes.p, kNoMatch, units * 16 + 64, st));

    {   // (float) pow(i, 0.75) for every possible indel count, computed by the host libm like the reference's table
        std::vector<float> pw((size_t)2 * S.max_len + 2);
        for (size_t v = 0; v < pw.size(); ++v) pw[v] = (float)pow((double)v, 0.75);
        FB_TRY(S.d_pow075.reserve(sizeof(float) * pw.size()));
        FB_CUDA(cudaMemcpyAsync(S.d_pow075.p, pw.data(), sizeof(float) * pw.size(), cudaMemcpyHostToDevice, st));
        FB_CUDA(cudaStreamSynchronize(st));          // pw goes out of scope
    }
    k_repack<<<(n + 7) / 8, 256, 0, st>>>(S.d_raw_codes.as<int8_t>(), S.d_raw_off.as<uint64_t>(),
                                          S.d_raw_len.as<uint32_t>(), S.d_perm.as<uint32_t>(),
                                          S.d_code_off.as<uint32_t>(), S.d_codes.as<uint8_t>(), n);
    FB_CUDA(cudaGetLastError());
    const size_t build_smem = (size_t)blob_words(max_nl) * 4;
    FB_CUDA(cudaFuncSetAttribute(k_build_blob, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)build_smem));
    k_build_blob<<<S.n_groups, 256, build_smem, st>>>(S.d_codes.as<uint8_t>(), S.d_code_off.as<uint32_t>(),
                                                      S.d_len_sorted.as<uint32_t>(), S.d_group_blob.as<uint64_t>(),
                                                      d_group_nl, S.d_blob.as<uint32_t>(), n);
    FB_CUDA(cudaGetLastError());
    k_quirky<<<(n + 127) / 128, 128, 0, st>>>(S.d_codes.as<uint8_t>(), S.d_code_off.as<uint32_t>(),
                                              S.d_len_sorted.as<uint32_t>(), S.d_flags.as<uint8_t>(), n);
    FB_CUDA(cudaGetLastError());
    ctx->launches += 3;
    std::vector<uint8_t> flags(n);
    FB_CUDA(cudaMemcpyAsync(flags.data(), S.d_flags.p, n, cudaMemcpyDeviceToHost, st));
    FB_CUDA(cudaStreamSynchronize(st));
    for (uint32_t p = 0; p < n; ++p)
        if (flags[p]) S.h_quirky.push_back(S.h_perm[p]);
    std::sort(S.h_quirky.begin(), S.h_quirky.end());
    std::sort(S.h_long.begin(), S.h_long.end());
    return FAMSA_OK;
}

static TileParams base_params(famsa_ctx* ctx)
{
    LcsState& S = ctx->lcs;
    TileParams P{};
    P.blob = S.d_blob.as<uint32_t>();
    P.group_blob = S.d_group_blob.as<uint64_t>();
    P.codes = S.d_codes.as<uint8_t>();
    P.code_off = S.d_code_off.as<uint32_t>();
    P.len_sorted = S.d_len_sorted.as<uint32_t>();
    P.perm = S.d_perm.as<uint32_t>();
    P.n = S.n;
    return P;
}

// exact recomputation of one row (caller id `row`) against a column list
static int exact_row(famsa_ctx* ctx, uint32_t row, const uint32_t* d_col_ids, uint32_t n_col,
                     int only_long_cols, void* d_out, size_t out_base, int elem_bytes, cudaStream_t st)
{
    LcsState& S = ctx->lcs;
    if (n_col == 0) return FAMSA_OK;
    const uint32_t sp = S.h_invperm[row];
    const uint32_t len = S.h_len_sorted[sp];
    const uint32_t nw = std::max(1u, (len + 63) / 64);
    const uint32_t threads = 128, blocks = (n_col + threads - 1) / threads;
    FB_TRY(S.d_masks64.reserve(sizeof(uint64_t) * kMaskRows * nw));
    FB_TRY(S.d_x64.reserve(sizeof(uint64_t) * (size_t)nw * blocks * threads));
    k_masks64<<<(kMaskRows * nw + 127) / 128, 128, 0, st>>>(
        S.d_codes.as<uint8_t>(), S.d_code_off.as<uint32_t>(), S.d_len_sorted.as<uint32_t>(), sp, nw,
        S.d_masks64.as<unsigned long long>());
    FB_CUDA(cudaGetLastError());
    const uint32_t* d_group_nl = reinterpret_cast<const uint32_t*>(S.d_group_blob.as<uint64_t>() + S.n_groups);
    k_lcs_exact<<<blocks, threads, 0, st>>>(
        S.d_codes.as<uint8_t>(), S.d_code_off.as<uint32_t>(), S.d_len_sorted.as<uint32_t>(),
        S.d_invperm.as<uint32_t>(), S.d_masks64.as<unsigned long long>(), nw, d_col_ids, n_col, d_group_nl,
        only_long_cols, S.d_x64.as<unsigned long long>(), d_out, out_base, elem_bytes);
    FB_CUDA(cudaGetLastError());
    ctx->launches += 2;
    return FAMSA_OK;
}

// The exact recomputation of many rows: rows of at most kExactWords * 64 residues go through one launch of
// k_lcs_exact_batch (masks in shared memory, X[] in the thread); longer ones keep the per-row global-memory path.
struct ExactReq { uint32_t row, n_col; int only_long; size_t out_base; };
static int exact_rows(famsa_ctx* ctx, const std::vector<ExactReq>& reqs, const uint32_t* d_col_ids, void* d_out, int elem_bytes, cudaStream_t st)
{
    LcsState& S = ctx->lcs;
    std::vector<ExactRow> batch;
    uint32_t max_cols = 0;
    for (const ExactReq& q : reqs) {
        if (!q.n_col) continue;
        const uint32_t sp = S.h_invperm[q.row];
        if (S.h_len_sorted[sp] <= (uint32_t)kExactWords * 64) {
            batch.push_back(ExactRow{sp, q.n_col, (uint32_t)q.only_long, 0, (unsigned long long)q.out_base});
            max_cols = std::max(max_cols, q.n_col);
        } else FB_TRY(exact_row(ctx, q.row, d_col_ids, q.n_col, q.only_long, d_out, q.out_base, elem_bytes, st));
    }
    if (batch.empty()) return FAMSA_OK;
    const uint32_t* d_group_nl = reinterpret_cast<const uint32_t*>(S.d_group_blob.as<uint64_t>() + S.n_groups);
    for (size_t b0 = 0; b0 < batch.size(); b0 += 65535) {            // gridDim.y limit
        const size_t nb = std::min<size_t>(65535, batch.size() - b0);
        FB_TRY(S.d_masks64.reserve(sizeof(ExactRow) * nb));
        FB_CUDA(cudaMemcpyAsync(S.d_masks64.p, batch.data() + b0, sizeof(ExactRow) * nb, cudaMemcpyHostToDevice, st));
        k_lcs_exact_batch<<<dim3((max_cols + 127) / 128, (unsigned)nb), 128, 0, st>>>(
            S.d_codes.as<uint8_t>(), S.d_code_off.as<uint32_t>(), S.d_len_sorted.as<uint32_t>(), S.d_invperm.as<uint32_t>(),
            S.d_masks64.as<ExactRow>(), d_col_ids, d_group_nl, d_out, elem_bytes);
        FB_CUDA(cudaGetLastError());
        ctx->launches++;
    }
    return FAMSA_OK;
}

// Rows [row_begin, row_end) of the packed triangle.  With `bounds` (n_blocks + 1 ascending row indices spanning the
// range) the work is issued block by block and block_events[b] is recorded after block b, so that a caller can
// start copying finished blocks while later ones are still being computed; every tile list is uploaded up front.
int lcs_triangle(famsa_ctx* ctx, uint32_t row_begin, uint32_t row_end, void* d_out, int elem_bytes, cudaStream_t st,
                 const uint32_t* bounds, int n_blocks, cudaEvent_t* block_events, bool quirk_fixups, bool piece_streams)
{
    LcsState& S = ctx->lcs;
    const uint32_t n = S.n;
    S.last_pairs = (uint64_t)row_end * (row_end ? row_end - 1 : 0) / 2 - (uint64_t)row_begin * (row_begin ? row_begin - 1 : 0) / 2;
    FB_CUDA(cudaEventRecord(ctx->ev[0], st));
    const uint32_t whole[2] = {row_begin, row_end};
    if (!bounds || !S.identity_perm) { bounds = whole; n_blocks = 1; }

    // tiles per (block, limb-count class); one upload for all of them
    std::vector<std::vector<std::vector<uint3>>> tiles(n_blocks, std::vector<std::vector<uint3>>(kMaxNL + 1));
    size_t total = 0;
    for (int b = 0; b < n_blocks; ++b)
        for (uint32_t g = 0; g < S.n_groups; ++g) {
            const uint32_t nl = S.groups[g].nl;
            if (nl == 0) continue;
            if (S.identity_perm && (g * 32 + 32 <= bounds[b] || g * 32 >= bounds[b + 1])) continue;
            const uint32_t q_end = std::min(n, g * 32 + 31);
            for (uint32_t q0 = 0; q0 < q_end; q0 += kTileQ) {
                tiles[b][nl].push_back(make_uint3(g, q0, std::min(q_end, q0 + (uint32_t)kTileQ)));
                ++total;
            }
        }
    S.last_tiles = total;
    std::vector<uint3> flat;
    flat.reserve(total);
    for (auto& blk : tiles)
        for (auto& v : blk) flat.insert(flat.end(), v.begin(), v.end());
    FB_TRY(S.d_tiles.reserve(sizeof(uint3) * std::max<size_t>(total, 1)));
    if (total) FB_CUDA(cudaMemcpyAsync(S.d_tiles.p, flat.data(), sizeof(uint3) * total, cudaMemcpyHostToDevice, st));
    TileParams P = base_params(ctx);
    P.out = d_out;
    P.elem_bytes = elem_bytes;
    P.rows_mode = 0;
    P.tri_base = (uint64_t)row_begin * (row_begin ? row_begin - 1 : 0) / 2;
    std::vector<uint32_t> special;      // rows the tile kernel may not answer for: dropped-carry and over-long rows
    if (quirk_fixups) std::set_union(S.h_quirky.begin(), S.h_quirky.end(), S.h_long.begin(), S.h_long.end(), std::back_inserter(special));
    else special = S.h_long;         // true LCS everywhere: only the rows the tile kernel cannot reach
    FB_CUDA(cudaEventRecord(ctx->ev[1], st));
    // Blocks in one stream would each end with a partly filled last wave (half a wave of tiles per block boundary: 0.4 ms at
    // C2).  Issued round-robin on the auxiliary streams instead, the block scheduler fills the tail of block b with the first
    // tiles of block b+1 and the blocks still finish in order.  (The exact kernels share one scratch: single stream then.)
    constexpr int kAux = sizeof(ctx->aux_stream) / sizeof(ctx->aux_stream[0]);
    const bool fan = piece_streams && n_blocks > 1 && special.empty();
    if (fan) {
        FB_CUDA(cudaEventRecord(ctx->ev_fork, st));
        for (int a = 0; a < std::min(kAux, n_blocks); ++a) FB_CUDA(cudaStreamWaitEvent(ctx->aux_stream[a], ctx->ev_fork, 0));
    }
    size_t at = 0;
    for (int b = 0; b < n_blocks; ++b) {
        const cudaStream_t bst = fan ? ctx->aux_stream[b % kAux] : st;
        P.row_begin = bounds[b];
        P.row_end = bounds[b + 1];
        for (uint32_t nl = 1; nl <= (uint32_t)kMaxNL; ++nl) {
            auto& v = tiles[b][nl];
            if (v.empty()) continue;
            P.tiles = S.d_tiles.as<uint3>() + at;
            FB_TRY(launch_tile_nl(ctx, nl, P, (uint32_t)v.size(), bst));
            at += v.size();
        }
        // rows the tile kernel cannot answer for: dropped-carry rows entirely; over-long rows only against over-long columns
        // (their pairs with shorter sequences were computed with the shorter one as the mask side -- the true LCS is symmetric)
        std::vector<ExactReq> reqs;
        for (uint32_t row : special) {
            if (row < bounds[b] || row >= bounds[b + 1] || row == 0) continue;
            const bool quirky = quirk_fixups && std::binary_search(S.h_quirky.begin(), S.h_quirky.end(), row);
            reqs.push_back(ExactReq{row, row, quirky ? 0 : 1, (size_t)row * (row - 1) / 2 - (size_t)P.tri_base});
        }
        FB_TRY(exact_rows(ctx, reqs, nullptr, d_out, elem_bytes, bst));
        if (block_events) FB_CUDA(cudaEventRecord(block_events[b], bst));
    }
    if (fan)
        for (int a = 0; a < std::min(kAux, n_blocks); ++a) {
            FB_CUDA(cudaEventRecord(ctx->ev_join[a], ctx->aux_stream[a]));
            FB_CUDA(cudaStreamWaitEvent(st, ctx->ev_join[a], 0));
        }
    FB_CUDA(cudaEventRecord(ctx->ev[2], st));
    FB_CUDA(cudaEventRecord(ctx->ev[3], st));
    return FAMSA_OK;
}

int lcs_rows(famsa_ctx* ctx, const uint32_t* d_ref_ids, const uint32_t* h_ref_ids, uint32_t n_ref,
             const uint32_t* d_col_ids, uint32_t n_col, void* d_out, int elem_bytes, cudaStream_t st,
             uint32_t g_begin, uint32_t g_end)
{
    LcsState& S = ctx->lcs;
    const uint32_t n = S.n;
    S.last_pairs = (uint64_t)n_ref * n_col;
    FB_CUDA(cudaEventRecord(ctx->ev[0], st));
    const uint32_t npad = S.n_groups * 32;
    const int res_bytes = S.max_len < 65536 ? 2 : 4;

    // streamed side = the reference rows (true LCS is symmetric); mask side = every group
    std::vector<uint32_t> refpos(n_ref);
    for (uint32_t r = 0; r < n_ref; ++r) refpos[r] = S.h_invperm[h_ref_ids[r]];
    FB_TRY(S.d_refpos.reserve(sizeof(uint32_t) * std::max(1u, n_ref)));
    FB_CUDA(cudaMemcpyAsync(S.d_refpos.p, refpos.data(), sizeof(uint32_t) * n_ref, cudaMemcpyHostToDevice, st));
    FB_TRY(S.d_res.reserve((size_t)res_bytes * npad * std::max(1u, n_ref)));

    std::vector<std::vector<uint3>> by_nl(kMaxNL + 1);
    g_end = std::min(g_end, S.n_groups);
    for (uint32_t g = g_begin; g < g_end; ++g) {                     // the mask groups (= columns) this call answers for
        const uint32_t nl = S.groups[g].nl;
        if (nl == 0) continue;
        for (uint32_t q0 = 0; q0 < n_ref; q0 += kTileQ)
            by_nl[nl].push_back(make_uint3(g, q0, std::min(n_ref, q0 + (uint32_t)kTileQ)));
    }
    size_t total = 0;
    for (auto& v : by_nl) total += v.size();
    FB_TRY(S.d_tiles.reserve(sizeof(uint3) * std::max<size_t>(total, 1)));
    size_t at = 0;
    for (auto& v : by_nl) {
        if (v.empty()) continue;
        FB_CUDA(cudaMemcpyAsync(S.d_tiles.as<uint3>() + at, v.data(), sizeof(uint3) * v.size(), cudaMemcpyHostToDevice, st));
        at += v.size();
    }
    TileParams P = base_params(ctx);
    P.out = S.d_res.p;
    P.elem_bytes = res_bytes;
    P.rows_mode = 1;
    P.refpos = S.d_refpos.as<uint32_t>();
    P.ld_res = npad;
    FB_CUDA(cudaEventRecord(ctx->ev[1], st));
    at = 0;
    for (uint32_t nl = 1; nl <= (uint32_t)kMaxNL; ++nl) {
        auto& v = by_nl[nl];
        if (v.empty()) continue;
        P.tiles = S.d_tiles.as<uint3>() + at;
        FB_TRY(launch_tile_nl(ctx, nl, P, (uint32_t)v.size(), st));
        at += v.size();
    }
    FB_CUDA(cudaEventRecord(ctx->ev[2], st));
    if (n_col && n_ref) {
        dim3 grid((n_col + 255) / 256, n_ref);
        k_gather_rows<<<grid, 256, 0, st>>>(S.d_res.p, npad, res_bytes, d_col_ids, S.d_invperm.as<uint32_t>(),
                                            n_col, d_out, elem_bytes);
        FB_CUDA(cudaGetLastError());
        ctx->launches++;
    }
    // exact fix-ups: dropped-carry / over-long reference rows entirely, over-long columns for the rest
    {
        std::vector<ExactReq> reqs;
        for (uint32_t r = 0; r < n_ref; ++r) {
            const uint32_t row = h_ref_ids[r];
            const bool quirky = std::binary_search(S.h_quirky.begin(), S.h_quirky.end(), row);
            const bool is_long = std::binary_search(S.h_long.begin(), S.h_long.end(), row);
            // (an over-long reference row is the streamed side of the tiles, so only its over-long columns are missing)
            if (quirky) reqs.push_back(ExactReq{row, n_col, 0, (size_t)r * n_col});
            else if (is_long || !S.h_long.empty()) reqs.push_back(ExactReq{row, n_col, 1, (size_t)r * n_col});
        }
        FB_TRY(exact_rows(ctx, reqs, d_col_ids, d_out, elem_bytes, st));
    }
    (void)d_ref_ids;
    (void)n;
    FB_CUDA(cudaEventRecord(ctx->ev[3], st));
    return FAMSA_OK;
}

// Parallel MST + host replay of Prim's visiting order (see the kernels above).  Expects the true-LCS triangle in
// d_prim_tri and the pow table in d_pow075_f64.
static int prim_boruvka(famsa_ctx* ctx, int kind, int eb, int32_t* h_from, int32_t* h_to, double* h_dist, int32_t* h_order)
{
    LcsState& S = ctx->lcs;
    cudaStream_t st = ctx->stream;
    const uint32_t n = S.n;
    const size_t pairs = (size_t)n * (n - 1) / 2;
    const uint32_t n_chunks = (n + kMstChunk - 1) / kMstChunk;
    FB_TRY(S.d_prim_dtri.reserve(pairs * sizeof(double)));
    FB_TRY(S.d_prim_comp.reserve(sizeof(uint32_t) * n));
    FB_TRY(S.d_prim_best.reserve(sizeof(EdgeMin) * n));
    FB_TRY(S.d_prim_part.reserve(sizeof(EdgeMin) * (size_t)n_chunks * n));
    double* d_dtri = S.d_prim_dtri.as<double>();
    uint32_t* d_comp = S.d_prim_comp.as<uint32_t>();
    EdgeMin* d_best = S.d_prim_best.as<EdgeMin>();
    EdgeMin* d_part = S.d_prim_part.as<EdgeMin>();
    k_mst_dist<<<n - 1, 256, 0, st>>>(S.d_prim_tri.p, eb, n, S.d_raw_len.as<uint32_t>(), S.d_pow075_f64.as<double>(), kind,
                                      nextafter(DBL_MAX, 0.0), d_dtri);
    FB_CUDA(cudaGetLastError());
    ctx->launches++;

    std::vector<uint32_t> parent(n), comp(n);
    std::iota(parent.begin(), parent.end(), 0u);
    std::iota(comp.begin(), comp.end(), 0u);
    auto find = [&](uint32_t x) {
        while (parent[x] != x) { parent[x] = parent[parent[x]]; x = parent[x]; }
        return x;
    };
    struct HostEdge { uint32_t a, b; double d; };
    std::vector<HostEdge> edges;
    edges.reserve(n - 1);
    std::vector<EdgeMin> best(n), cbest(n);
    const double none = kEdgeNone;
    uint32_t n_comp = n;
    while (n_comp > 1) {
        FB_CUDA(cudaMemcpyAsync(d_comp, comp.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice, st));
        k_mst_rows<<<n, 256, 0, st>>>(d_dtri, n, d_comp, d_best);
        k_mst_cols<<<dim3((n + 31) / 32, n_chunks), 256, 0, st>>>(d_dtri, n, d_comp, d_part);
        k_mst_combine<<<(n + 255) / 256, 256, 0, st>>>(n, n_chunks, d_part, d_best);
        FB_CUDA(cudaGetLastError());
        ctx->launches += 3;
        FB_CUDA(cudaMemcpyAsync(best.data(), d_best, sizeof(EdgeMin) * n, cudaMemcpyDeviceToHost, st));
        FB_CUDA(cudaStreamSynchronize(st));
        // every component's smallest outgoing edge ...
        for (uint32_t v = 0; v < n; ++v) cbest[v].d = none;
        for (uint32_t v = 0; v < n; ++v) {
            if (!(best[v].d < none)) continue;
            EdgeMin& c = cbest[comp[v]];
            if (best[v].d < c.d || (best[v].d == c.d && best[v].k < c.k)) c = best[v];
        }
        // ... joins two components (the edge order is strict, so no cycle can close)
        const uint32_t before = n_comp;
        for (uint32_t c = 0; c < n; ++c) {
            if (!(cbest[c].d < none)) continue;
            const unsigned long long packed = ~cbest[c].k;         // uint64_to_id (MSTPrim.h:441-450)
            const uint32_t a = (uint32_t)(packed >> 32), b = (uint32_t)(packed & 0xffffffffull);
            const uint32_t ra = find(a), rb = find(b);
            if (ra == rb) continue;                                 // both sides elected the same edge
            parent[ra] = rb;
            edges.push_back(HostEdge{a, b, cbest[c].d});
            --n_comp;
        }
        if (n_comp == before) { set_error("famsa_lcs_prim: no progress in a Boruvka round"); return FAMSA_E_CUDA; }
        for (uint32_t v = 0; v < n; ++v) comp[v] = find(v);
    }
    FB_CUDA(cudaEventRecord(ctx->ev[3], st));
    // Prim's visiting order from vertex 0, replayed on the tree (MSTPrim.cpp:366-386 restricted to tree edges)
    std::vector<std::vector<std::tuple<double, unsigned long long, uint32_t>>> adj(n);
    for (const HostEdge& e : edges) {
        const unsigned long long lo = std::min(e.a, e.b), hi = std::max(e.a, e.b);
        const unsigned long long key = ~((lo << 32) + hi);
        adj[e.a].emplace_back(e.d, key, e.b);
        adj[e.b].emplace_back(e.d, key, e.a);
    }
    using Item = std::tuple<double, unsigned long long, uint32_t>;
    std::priority_queue<Item, std::vector<Item>, std::greater<Item>> heap;
    for (uint32_t v = 0; v < n; ++v) h_order[v] = (int32_t)n;
    h_order[0] = 0;
    for (const Item& it : adj[0]) heap.push(it);
    uint32_t step = 0;
    while (!heap.empty()) {
        const Item it = heap.top();
        heap.pop();
        const uint32_t v = std::get<2>(it);
        if (h_order[v] != (int32_t)n) continue;
        const unsigned long long packed = ~std::get<1>(it);
        h_from[step] = (int32_t)(packed >> 32);
        h_to[step] = (int32_t)(packed & 0xffffffffull);
        h_dist[step] = std::get<0>(it);
        h_order[v] = (int32_t)++step;
        for (const Item& nx : adj[v])
            if (h_order[std::get<2>(nx)] == (int32_t)n) heap.push(nx);
    }
    if (step != n - 1) { set_error("famsa_lcs_prim: the replay did not reach every sequence"); return FAMSA_E_CUDA; }
    return FAMSA_OK;
}

int lcs_prim(famsa_ctx* ctx, int kind, int32_t* h_from, int32_t* h_to, double* h_dist, int32_t* h_order)
{
    LcsState& S = ctx->lcs;
    cudaStream_t st = ctx->stream;
    const uint32_t n = S.n;
    const int eb = S.max_len < 65536 ? 2 : 4;
    const size_t pairs = (size_t)n * (n - 1) / 2;
    FB_TRY(S.d_prim_tri.reserve(std::max<size_t>(pairs, 1) * eb));
    // the true-LCS triangle (orientation-free) ...
    FB_TRY(lcs_triangle(ctx, 0, n, S.d_prim_tri.p, eb, st, nullptr, 1, nullptr, /*quirk_fixups=*/false));
    // ... plus, for the few sequences whose LCS depends on which side is the row, their own rows
    std::vector<int> side_idx(n, -1);
    for (size_t q = 0; q < S.h_quirky.size(); ++q) side_idx[S.h_quirky[q]] = (int)q;
    FB_TRY(S.d_prim_sideidx.reserve(sizeof(int) * n));
    FB_CUDA(cudaMemcpyAsync(S.d_prim_sideidx.p, side_idx.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    const uint32_t nq = (uint32_t)S.h_quirky.size();
    FB_TRY(S.d_prim_side.reserve(std::max<size_t>((size_t)nq * n, 1) * sizeof(uint32_t)));
    if (nq) {
        FB_TRY(S.d_ids_a.reserve(sizeof(uint32_t) * nq));
        FB_CUDA(cudaMemcpyAsync(S.d_ids_a.p, S.h_quirky.data(), sizeof(uint32_t) * nq, cudaMemcpyHostToDevice, st));
        FB_TRY(lcs_rows(ctx, S.d_ids_a.as<uint32_t>(), S.h_quirky.data(), nq, nullptr, n, S.d_prim_side.p, 4, st));
    }
    {   // (double) pow(i, 0.75), host libm, like Transform<double, indel075_div_lcs>'s table
        std::vector<double> pw((size_t)2 * S.max_len + 2);
        for (size_t v = 0; v < pw.size(); ++v) pw[v] = pow((double)v, 0.75);
        FB_TRY(S.d_pow075_f64.reserve(sizeof(double) * pw.size()));
        FB_CUDA(cudaMemcpyAsync(S.d_pow075_f64.p, pw.data(), sizeof(double) * pw.size(), cudaMemcpyHostToDevice, st));
        FB_CUDA(cudaStreamSynchronize(st));
    }
    if (S.h_quirky.empty() && n >= 2 && !getenv("FAMSA_PRIM_SEQUENTIAL")) {
        const int rc = prim_boruvka(ctx, kind, eb, h_from, h_to, h_dist, h_order);
        if (rc != FAMSA_E_NOMEM) return rc;                         // no room for the float64 triangle: sequential loop
    }
    FB_TRY(S.d_prim_state.reserve((sizeof(PrimState) + 1) * (size_t)n + 64));
    FB_TRY(S.d_prim_out.reserve((sizeof(int) * 3 + sizeof(double)) * (size_t)n + 64));
    PrimState* d_state = S.d_prim_state.as<PrimState>();
    unsigned char* d_vis = reinterpret_cast<unsigned char*>(d_state + n);
    double* d_dist = S.d_prim_out.as<double>();
    int* d_from = reinterpret_cast<int*>(d_dist + n);
    int* d_to = d_from + n;
    int* d_order = d_to + n;
    {
        int per_sm = 0;
        FB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_prim, 1024, 0));
        const uint32_t nblk = std::max(1u, std::min((uint32_t)(ctx->sm_count * std::max(per_sm, 1)), (n + 1023) / 1024));
        FB_TRY(S.d_prim_cand.reserve(sizeof(PrimCand) * 2 * nblk));
        const void* a_tri = S.d_prim_tri.p; int a_eb = eb; uint32_t a_n = n;
        const uint32_t* a_len = S.d_raw_len.as<uint32_t>(); const double* a_pow = S.d_pow075_f64.as<double>();
        int a_kind = kind; double a_never = nextafter(DBL_MAX, 0.0);
        const int* a_sidx = S.d_prim_sideidx.as<int>(); const uint32_t* a_side = S.d_prim_side.as<uint32_t>();
        PrimCand* a_cand = S.d_prim_cand.as<PrimCand>();
        void* args[] = {&a_tri, &a_eb, &a_n, &a_len, &a_pow, &a_kind, &a_never, &a_sidx, &a_side, &d_state, &d_vis,
                        &a_cand, &d_from, &d_to, &d_dist, &d_order};
        FB_CUDA(cudaLaunchCooperativeKernel((void*)k_prim, dim3(nblk), dim3(1024), args, 0, st));
    }
    ctx->launches++;
    FB_CUDA(cudaEventRecord(ctx->ev[3], st));
    if (n > 1) {
        FB_CUDA(cudaMemcpyAsync(h_from, d_from, sizeof(int) * (n - 1), cudaMemcpyDeviceToHost, st));
        FB_CUDA(cudaMemcpyAsync(h_to, d_to, sizeof(int) * (n - 1), cudaMemcpyDeviceToHost, st));
        FB_CUDA(cudaMemcpyAsync(h_dist, d_dist, sizeof(double) * (n - 1), cudaMemcpyDeviceToHost, st));
    }
    FB_CUDA(cudaMemcpyAsync(h_order, d_order, sizeof(int) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA(cudaStreamSynchronize(st));
    return FAMSA_OK;
}

int lcs_assign(famsa_ctx* ctx, const uint32_t* h_seed_ids, uint32_t n_seeds, int kind, uint32_t* h_assign, float* h_mind)
{
    LcsState& S = ctx->lcs;
    cudaStream_t st = ctx->stream;
    const uint32_t n = S.n;
    const int eb = S.max_len < 65536 ? 2 : 4;
    FB_TRY(S.d_assign_lcs.reserve((size_t)eb * n * n_seeds));
    FB_TRY(S.d_assign.reserve(sizeof(uint32_t) * n));
    FB_TRY(S.d_mind.reserve(sizeof(float) * n));
    FB_TRY(S.d_ids_a.reserve(sizeof(uint32_t) * n_seeds));
    FB_CUDA(cudaMemcpyAsync(S.d_ids_a.p, h_seed_ids, sizeof(uint32_t) * n_seeds, cudaMemcpyHostToDevice, st));
    // seed k is the row (seq0) of its distance vector, every sequence a column: exactly famsa_lcs_rows
    FB_TRY(lcs_rows(ctx, S.d_ids_a.as<uint32_t>(), h_seed_ids, n_seeds, nullptr, n, S.d_assign_lcs.p, eb, st));
    const float never = (float)nextafter((double)FLT_MAX, 0.0);
    k_assign<<<(n + 255) / 256, 256, 0, st>>>(S.d_assign_lcs.p, eb, n, n_seeds, S.d_ids_a.as<uint32_t>(),
                                             S.d_raw_len.as<uint32_t>(), S.d_pow075.as<float>(), kind, never,
                                             S.d_assign.as<uint32_t>(), S.d_mind.as<float>());
    FB_CUDA(cudaGetLastError());
    ctx->launches++;
    FB_CUDA(cudaEventRecord(ctx->ev[3], st));
    FB_CUDA(cudaMemcpyAsync(h_assign, S.d_assign.p, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA(cudaMemcpyAsync(h_mind, S.d_mind.p, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA(cudaStreamSynchronize(st));
    return FAMSA_OK;
}


// famsa_lcs_upgma: LCS triangle (row = seq0, as calculateDistanceVector builds it) -> float distances -> the agglomeration
int lcs_upgma(famsa_ctx* ctx, int kind, int modified, int32_t* h_tree, const void* d_tri_in, int tri_eb)
{
    LcsState& S = ctx->lcs;
    cudaStream_t st = ctx->stream;
    const uint32_t n = S.n;
    const int eb = d_tri_in ? tri_eb : (S.max_len < 65536 ? 2 : 4);
    const size_t pairs = (size_t)n * (n - 1) / 2;
    const void* d_tri = d_tri_in;
    if (!d_tri) {
        FB_TRY(S.d_prim_tri.reserve(std::max<size_t>(pairs, 1) * eb));
        FB_TRY(lcs_triangle(ctx, 0, n, S.d_prim_tri.p, eb, st));
        d_tri = S.d_prim_tri.p;
    } else {
        S.last_pairs = 0;
        FB_CUDA(cudaEventRecord(ctx->ev[0], st)); FB_CUDA(cudaEventRecord(ctx->ev[1], st)); FB_CUDA(cudaEventRecord(ctx->ev[2], st));
    }
    FB_TRY(S.d_prim_dtri.reserve(std::max<size_t>(pairs, 1) * sizeof(float)));
    FB_TRY(S.d_prim_state.reserve((sizeof(float) + sizeof(uint32_t) + sizeof(int)) * (size_t)n + 64));
    FB_TRY(S.d_prim_out.reserve(sizeof(int) * 2 * (size_t)n + 64));
    float* d_dist = S.d_prim_dtri.as<float>();
    float* d_mind = S.d_prim_state.as<float>();
    uint32_t* d_nn = reinterpret_cast<uint32_t*>(d_mind + n);
    int* d_node = reinterpret_cast<int*>(d_nn + n);
    int* d_tree = S.d_prim_out.as<int>();
    int* d_status = d_tree + 2 * (size_t)(n - 1);
    const float never = (float)nextafter((double)FLT_MAX, 0.0);
    k_upgma_dist<<<n - 1, 256, 0, st>>>(d_tri, eb, n, S.d_raw_len.as<uint32_t>(), S.d_pow075.as<float>(), kind, never, d_dist);
    k_upgma_init<<<n, 256, 0, st>>>(d_dist, n, d_mind, d_nn, d_node);
    FB_CUDA(cudaGetLastError());
    FB_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    ctx->launches += 2;
    {
        void* fn = modified ? (void*)k_upgma<true> : (void*)k_upgma<false>;
        int per_sm = 0;
        FB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, 1024, 0));
        const uint32_t nblk = std::max(1u, std::min((uint32_t)(ctx->sm_count * std::max(per_sm, 1)), (n + 1023) / 1024));
        FB_TRY(S.d_prim_cand.reserve(sizeof(unsigned long long) * 2 * nblk));
        uint32_t a_n = n;
        unsigned long long* a_cand = S.d_prim_cand.as<unsigned long long>();
        void* args[] = {&d_dist, &a_n, &d_mind, &d_nn, &d_node, &a_cand, &d_tree, &d_status};
        FB_CUDA(cudaLaunchCooperativeKernel(fn, dim3(nblk), dim3(1024), args, 0, st));
        ctx->launches++;
    }
    FB_CUDA(cudaEventRecord(ctx->ev[3], st));
    int status = 0;
    FB_CUDA(cudaMemcpyAsync(h_tree, d_tree, sizeof(int) * 2 * (size_t)(n - 1), cudaMemcpyDeviceToHost, st));
    FB_CUDA(cudaMemcpyAsync(&status, d_status, sizeof(int), cudaMemcpyDeviceToHost, st));
    FB_CUDA(cudaStreamSynchronize(st));
    if (status) { set_error("famsa_lcs_upgma: no finite distance left between two clusters (sequences without a common residue)"); return FAMSA_E_INVALID; }
    return FAMSA_OK;
}

// famsa_lcs_assign_shard: the seed rows against this shard's slice of the mask groups only, packed for a MIN all-reduce
int lcs_assign_shard(famsa_ctx* ctx, const uint32_t* h_seed_ids, uint32_t n_seeds, int kind, uint32_t shard, uint32_t n_shards,
                     long long* d_packed, cudaStream_t st)
{
    LcsState& S = ctx->lcs;
    const uint32_t n = S.n;
    const int eb = S.max_len < 65536 ? 2 : 4;
    const uint32_t g_begin = (uint32_t)((unsigned long long)S.n_groups * shard / n_shards);
    const uint32_t g_end = (uint32_t)((unsigned long long)S.n_groups * (shard + 1) / n_shards);
    FB_TRY(S.d_assign_lcs.reserve((size_t)eb * n * n_seeds));
    FB_TRY(S.d_ids_a.reserve(sizeof(uint32_t) * n_seeds));
    FB_CUDA(cudaMemcpyAsync(S.d_ids_a.p, h_seed_ids, sizeof(uint32_t) * n_seeds, cudaMemcpyHostToDevice, st));
    FB_TRY(lcs_rows(ctx, S.d_ids_a.as<uint32_t>(), h_seed_ids, n_seeds, nullptr, n, S.d_assign_lcs.p, eb, st, g_begin, g_end));
    S.last_pairs = 0;
    for (uint32_t g = g_begin; g < g_end; ++g) S.last_pairs += (uint64_t)std::min(32u, n - g * 32) * n_seeds;
    const float never = (float)nextafter((double)FLT_MAX, 0.0);
    k_assign_packed<<<(n + 255) / 256, 256, 0, st>>>(S.d_assign_lcs.p, eb, n, n_seeds, S.d_ids_a.as<uint32_t>(),
                                                    S.d_raw_len.as<uint32_t>(), S.d_pow075.as<float>(), kind, never,
                                                    S.d_invperm.as<uint32_t>(), g_begin, g_end, d_packed);
    FB_CUDA(cudaGetLastError());
    ctx->launches++;
    FB_CUDA(cudaEventRecord(ctx->ev[3], st));
    return FAMSA_OK;
}

} // namespace fb
