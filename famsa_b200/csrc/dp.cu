// HP-2: profile-profile / sequence-profile / sequence-sequence affine-gap DP with position-specific
// gap costs, many independent merges per launch, plus on-device traceback.
//
// Replaces CProfile::Align and its cell loops (reference src/core/profile.cpp:244-305,
// profile_seq.cpp:24-892, profile_par.cpp:26-903), DP_SolveGapsProblemWhenStarting/Continuing
// (profile.cpp:1223-1315) and the traceback of ConstructProfile (profile.cpp:727-782).
// Semantics follow SURVEY.md Appendix B; arithmetic is int64 with NEG = -(1<<62) unsaturated.
//
// Design (two kernels per batch, see DESIGN.md section 4):
//   k_dp_prep  one block per merge: resolves the children's widths (a child may be a merge that is still queued on
//              the stream: its width is read from device memory), variant + orientation (CProfile::Align), the
//              column-side constant records (gap scores + gap-correction counts, 8 x int64 per column, structure of
//              arrays), row 0 of the DP (block-parallel prefix sum) and the ranges that decide which arithmetic the
//              fill may use for the column-pair score.
//   k_dp_fill  the recurrence itself: a team of warps per merge, 32-row stripes, lane L owns row i0+L and at step s
//              computes column s-L (anti-diagonal wavefront); (D,H,V) of the cell above arrives by warp shuffle, the
//              left neighbour stays in registers.  Work proceeds in CHUNKS of 8 columns: the chunk's boundary-row
//              cells, column records and the column profile's scores are staged into the warp's shared memory by
//              cp.async one chunk ahead; from the staged scores the warp builds the 32 x 8 tile of column-pair scores
//              T[i][j] = sum_k counters_row[i][k] * scores_col[j][k]  (profile_par.cpp:695-711) -- on the tensor cores
//              (IMMA, exact byte-digit planes) for ProfProf, a table look-up for the Seq* variants -- into a ring
//              indexed by wavefront step, so the 8 dependent steps that follow read nothing but shared memory and
//              registers.  T never exists in HBM.  Stripes of one merge are DECOUPLED: every stripe publishes how many
//              columns of its last row it has parked in the boundary row (L2) and the stripe below polls that counter
//              once per chunk (the load is issued a whole tile computation before its value is needed); there is no
//              block- or cluster-wide barrier inside the loop.  The direction bytes go out skewed (one 32-byte store
//              per step).  The same kernel then walks the direction matrix back and emits the path.
//   k_dp_unskew only when the caller asks for CDPMatrix bytes: skewed directions -> row-major.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <thread>

#include <cooperative_groups.h>

#include "ctx.h"
#include "dp_dev.h"
#include "prof_dev.cuh"

namespace fb {

constexpr int kDpWarps = 4;               // warps (= merges) per block of the one-warp-per-merge fill kernel
constexpr int kDpTeamWarps = 8;           // warps cooperating on one large merge
constexpr uint32_t kDpTeamMinWidth = 96;  // min(w1, w2) above which a merge gets a team
constexpr int kDpCluster = 8;             // thread blocks per cluster for the widest merges
constexpr uint32_t kDpClusterMinWidth = 1024;   // min(w1, w2) above which a merge gets a whole cluster
constexpr int kTThreads = 256, kTCellsPerThread = 4;

// per column j of the column profile, 64 bytes, meaning depends on the variant:
//   ProfProf: gap scores {S[j][GO], S[j][GE], S[j][TO], S[j][TE]}, chg, b0 = (s_o, s_e), b1 = (s_to, s_te), b2 = (k_e, k_te)
//   SeqProf : same gap scores, chg, b0 = gcv1, b1 = contv1 (profile_par.cpp:204-211)
//   SeqSeq  : unused
struct ColInfo {
    long long cgo, cge, cto, cte;
    long long chg;
    long long b0, b1, b2;
};
static_assert(sizeof(ColInfo) == 64, "ColInfo layout");

struct Cell { long long D, H, V, pad; };   // 32 bytes: two 16-byte cp.async / st.cg.v2 transfers
static_assert(sizeof(Cell) == 32, "Cell layout");

constexpr int kChunk = 8;                   // columns per chunk (= wavefront steps per macro step)
constexpr int kColFields = 8;               // ColInfo as structure-of-arrays: field f of column j at col[f * cstride + j]
constexpr int kRing = 64;                   // shared-memory window of column records per warp (columns mod 64)
constexpr int kTRing = 64;                  // wavefront steps held by the T ring (a chunk's tile spans steps 8m .. 8m+38; a power of two
                                            // that the chunk length divides, so a chunk's eight slots never wrap)
constexpr int kS2Stride = 34;               // int64 per staged score column (272 bytes: conflict-free LDS.128 of the IMMA B fragments)

// Shared memory of one warp of k_dp_fill.
struct __align__(16) WarpShared {
    Cell brow[2][kChunk];                   // boundary-row cells of the current / next chunk
    long long col[kColFields][kRing];       // column records
    long long s2[2][kChunk][kS2Stride];     // the column profile's scores of the current / next chunk
    long long park[kChunk][3];              // (D, H, V) of the stripe's last row, one entry per step of the chunk (written by lane 31)
    long long t[kTRing][32];                // T ring: [wavefront step mod 64][lane]; viewed as int[64][32] when T fits 32 bits.  LAST member:
                                            // k_dp_fill_compact allocates only the half the 4-byte view needs (kCompactStride)
};
// per-warp shared memory of k_dp_fill_compact: everything but the upper half of the T ring (merges whose T needs 8 bytes are left to
// a k_dp_fill launch that follows): 17.3 KB instead of 25.5 KB, i.e. 12 instead of 8 fill warps per SM
constexpr size_t kCompactStride = sizeof(WarpShared) - sizeof(long long) * (kTRing / 2) * 32;
static_assert(offsetof(WarpShared, t) + sizeof(long long) * kTRing * 32 == sizeof(WarpShared) && kCompactStride % 16 == 0, "T ring must end the struct");

// scratch layout of one job (all sections 128-byte aligned); w1, w2 = the layout widths (upper bounds)
struct Scratch {
    unsigned long long col, brow, tmp, lastv, total, cstride;
    __host__ __device__ Scratch(uint32_t w1, uint32_t w2)
    {
        const unsigned long long wm = (w1 > w2 ? w1 : w2) + 1ull;
        cstride = align_up(wm + 1, 16);
        col = 0;
        brow = align_up(col + 8ull * kColFields * cstride, 128);
        tmp = align_up(brow + 48ull * wm, 128);            // kBrowWords tagged words per column
        lastv = align_up(tmp + w1 + w2, 128);
        total = lastv + 128;
    }
};

__device__ __forceinline__ long long pack2(int lo, int hi) { return (long long)(((unsigned long long)(unsigned)hi << 32) | (unsigned)lo); }
__device__ __forceinline__ int lo32(long long v) { return (int)(unsigned long long)v; }
__device__ __forceinline__ int hi32(long long v) { return (int)((unsigned long long)v >> 32); }
// The counts that weight the gap scores (how many sequences open / extend a gap, how many hold a residue) are
// non-negative for every profile CProfile can build; k_dp_prep verifies that (DpMeta::bad) so that the cell loop may
// multiply  int64 score x uint32 count  with two instructions (IMAD.WIDE.U32 + IMAD) instead of the signed 64 x 64 form.
__device__ __forceinline__ unsigned ulo32(long long v) { return (unsigned)(unsigned long long)v; }
__device__ __forceinline__ unsigned uhi32(long long v) { return (unsigned)((unsigned long long)v >> 32); }

__device__ __forceinline__ long long shfl_up_ll(long long v)
{
    int lo = lo32(v), hi = hi32(v);
    lo = __shfl_up_sync(0xffffffffu, lo, 1);
    hi = __shfl_up_sync(0xffffffffu, hi, 1);
    return pack2(lo, hi);
}

__device__ __forceinline__ long long shfl_up_ll_by(long long v, int delta)
{
    int lo = lo32(v), hi = hi32(v);
    lo = __shfl_up_sync(0xffffffffu, lo, delta);
    hi = __shfl_up_sync(0xffffffffu, hi, delta);
    return pack2(lo, hi);
}

// global (L2) -> shared without staging registers: the warp does not wait for the data
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// The boundary row in L2: per column six 8-byte words {D.lo, D.hi, H.lo, H.hi, V.lo, V.hi}; every word carries a
// 32-bit half of the value in its lower half and the writer's tag in its upper half, so a reader can tell from the
// words themselves whether it is looking at the row it waits for (8-byte accesses are single transactions).
constexpr int kBrowWords = 6;
__device__ __forceinline__ void park_cell(unsigned long long* p, const Cell& c, uint32_t tag)
{
    const unsigned long long t = (unsigned long long)tag << 32;
    ulonglong2* q = reinterpret_cast<ulonglong2*>(p);
    __stcg(q, make_ulonglong2(t | (unsigned)(unsigned long long)c.D, t | (unsigned)((unsigned long long)c.D >> 32)));
    __stcg(q + 1, make_ulonglong2(t | (unsigned)(unsigned long long)c.H, t | (unsigned)((unsigned long long)c.H >> 32)));
    __stcg(q + 2, make_ulonglong2(t | (unsigned)(unsigned long long)c.V, t | (unsigned)((unsigned long long)c.V >> 32)));
}
__device__ __forceinline__ ulonglong2 ld_cg_v2(const unsigned long long* p)       // from L2, re-executed on every call
{
    ulonglong2 v;
    asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p) : "memory");
    return v;
}

// a if a>b && a>c; else b if b>c; else c  (strict comparisons, fixed priority)
__device__ __forceinline__ int pick3(long long a, long long b, long long c, int da, int db, int dc, long long& out)
{
    const bool aw = (a > b) & (a > c);
    const bool bw = b > c;
    const long long bc = bw ? b : c;
    const int dbc = bw ? db : dc;
    out = aw ? a : bc;
    return aw ? da : dbc;
}
// a value that can never win a strict comparison: turns a 3-way pick into the reference's 2-way form
constexpr long long kNever = (long long)0x8000000000000000ull;

// DP_SolveGapsProblemWhenStarting / WhenContinuing (profile.cpp:1223-1315) for column c
__device__ __forceinline__ void solve_gaps(const int* __restrict__ cnt, uint32_t c, uint32_t width, int card,
                                           int& s_o, int& s_e, int& s_to, int& s_te, int& k_e, int& k_te)
{
    const int* cc = cnt + (size_t)c * 32;
    if (c >= width) {
        s_te = cc[kGapTO] + cc[kGapTE]; s_to = card - s_te; s_o = 0; s_e = 0;
        k_te = card; k_e = 0;
    } else {
        const int* cn = cc + 32;
        s_to = cn[kGapTO]; s_te = cc[kGapTO] + cc[kGapTE]; s_e = cc[kGapGO] + cc[kGapGE];
        s_o = card - s_e - s_to - s_te;
        k_te = cn[kGapTO] + cc[kGapTO] + cc[kGapTE]; k_e = card - k_te;
    }
}

__device__ __forceinline__ int seq_symbol(const int* __restrict__ cnt, uint32_t c)
{
    const int* cc = cnt + (size_t)c * 32;
    for (int k = 0; k < 24; ++k)
        if (cc[k]) return k;
    return 22;
}

struct DpParams {
    const DpJobDev* jobs;
    DpMeta* meta;
    const uint32_t* order;        // launch slot -> job index
    uint32_t n_jobs;              // jobs of this launch (a sub-batch, or one fill class of it)
    uint32_t job_base;            // first job id of the sub-batch (k_dp_prep indexes jobs as job_base + x)
    long long go, ge, to, te;
    unsigned char* dirs;          // caller-visible row-major direction matrices (CDPMatrix layout) or nullptr
    unsigned char* sdirs;         // internal skewed direction bytes of the sub-batch
    unsigned char* path;          // all paths (forward order)
    unsigned char* scratch;
    const unsigned long long* tblock;   // k_dp_unskew: first block of each job (n_jobs + 1 entries)
    famsa_dp_result* results;
    famsa_dp_result* h_results;   // optional mapped host copies written by the traceback itself (no D2H copy afterwards)
    unsigned char* h_path;
    uint32_t wide_only;           // k_dp_fill: skip merges whose T fits 32 bits (k_dp_fill_compact has done them)
};

// ------------------------------------------------------------------------------------------------
// k_dp_prep: one block per job
// ------------------------------------------------------------------------------------------------
constexpr int kPrepThreads = 512;
// all threads of the block (any multiple of 32 up to kPrepThreads)
__device__ __forceinline__ void prep_body(const DpParams& P, uint32_t jid)
{
    const DpJobDev J = P.jobs[jid];
    const uint32_t tid = threadIdx.x, nthr = blockDim.x;

    // A child that is itself a merge queued earlier on this stream reports its width (and whether it failed) in
    // device memory; the widths in the job are then only upper bounds that size the buffers.
    uint32_t w1 = J.w1, w2 = J.w2;
    int child_bad = 0;
    if (J.w1_src) { const uint32_t v = __ldcg(J.w1_src); child_bad |= v == kWidthBad || v == 0 || v > J.w1; if (!child_bad) w1 = v; }
    if (J.w2_src) { const uint32_t v = __ldcg(J.w2_src); const int b = v == kWidthBad || v == 0 || v > J.w2; child_bad |= b; if (!b) w2 = v; }
    if (child_bad) {
        // nothing below may trust the tables: report the failure and leave a 1 x 1 job behind for the other kernels
        if (tid == 0) {
            DpMeta m;
            m.SR = J.s1; m.CR = J.c1; m.SC = J.s2; m.CC = J.c2; m.WR = 0; m.WC = 0; m.nR = 1; m.nC = 1; m.var = 0; m.sw = 0;
            m.bad = 2; m.tmode = 2; m.t32 = 0;
            P.meta[jid] = m;
        }
        return;
    }

    // variant and orientation (CProfile::Align, profile.cpp:254-304).  Everything the decision and the fill's choice of
    // arithmetic need is gathered in ONE pass over the tables and one reduction: per side the number of non-zero counters
    // (orientation of ProfProf), the largest |score| that can enter T and whether it leaves int32, and -- ProfProf only --
    // whether every count the cell loop multiplies with is >= 0 (see ulo32).
    int var, sw = 0;
    if (J.card1 == 1 && J.card2 == 1) var = 0;
    else if (J.card1 == 1) var = 1;
    else if (J.card2 == 1) { var = 1; sw = 1; }
    else var = 2;
    __shared__ unsigned long long sm_red[2][3];                      // per side: nz, smax, flags (1 wide, 2 bad)
    if (tid < 6) sm_red[tid / 3][tid % 3] = 0;
    __syncthreads();
    for (int side = 0; side < 2; ++side) {
        const bool is_col = var == 2 || (side == 1) != (sw == 1);    // Seq*: only the column side's scores matter
        const long long* sc = side ? J.s2 : J.s1;
        const int* cnt = side ? J.c2 : J.c1;
        const uint32_t w = side ? w2 : w1;
        const int card = (int)(side ? J.card2 : J.card1);
        unsigned long long nz = 0, smax = 0, flags = 0;
        // one thread per column, all loads of a column issued together (the block is small: memory-level parallelism
        // is what makes this pass short)
        for (uint32_t c = tid; c <= w; c += nthr) {
            if (var == 2) {
                const int4* cc = reinterpret_cast<const int4*>(cnt + (size_t)c * 32);
                int4 v[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = cc[q];
                int neg = 0, over = 0;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    nz += (v[q].x != 0) + (v[q].y != 0) + (v[q].z != 0) + (v[q].w != 0);
                    int4 u = v[q];
                    if (q == 7) { u.z = 0; u.w = 0; }                 // rows 30 (GAP) and 31 (GUARD) are not counts of a symbol
                    neg |= u.x | u.y | u.z | u.w;
                    over |= (u.x > card) | (u.y > card) | (u.z > card) | (u.w > card);
                }
                if (c >= 1) {
                    int a2, b2, d2, e2, f2, g2;
                    solve_gaps(cnt, c, w, card, a2, b2, d2, e2, f2, g2);
                    if ((a2 | b2 | d2 | e2 | f2 | g2) < 0 || neg < 0 || over) flags |= 2;
                }
            }
            if (is_col && c >= 1) {                                   // columns 1..w, rows 0..29 feed T
                const longlong2* sp = reinterpret_cast<const longlong2*>(sc + (size_t)c * 32);
                longlong2 v[15];
#pragma unroll
                for (int q = 0; q < 15; ++q) v[q] = sp[q];
#pragma unroll
                for (int q = 0; q < 15; ++q) {
                    flags |= (v[q].x != (long long)(int)v[q].x) | (v[q].y != (long long)(int)v[q].y);
                    const unsigned long long ax = (unsigned long long)(v[q].x < 0 ? -v[q].x : v[q].x);
                    const unsigned long long ay = (unsigned long long)(v[q].y < 0 ? -v[q].y : v[q].y);
                    smax = ax > smax ? ax : smax;
                    smax = ay > smax ? ay : smax;
                }
            }
        }
        for (int o = 16; o; o >>= 1) {
            nz += __shfl_xor_sync(0xffffffffu, nz, o);
            const unsigned long long x = __shfl_xor_sync(0xffffffffu, smax, o);
            smax = x > smax ? x : smax;
            flags |= __shfl_xor_sync(0xffffffffu, flags, o);
        }
        if ((tid & 31) == 0) {
            if (nz) atomicAdd(&sm_red[side][0], nz);
            if (smax) atomicMax(&sm_red[side][1], smax);
            if (flags) atomicOr(&sm_red[side][2], flags);
        }
    }
    __syncthreads();
    if (var == 2 && !(sm_red[0][0] * (unsigned long long)w2 < sm_red[1][0] * (unsigned long long)w1)) sw = 1;
    const long long* SR = sw ? J.s2 : J.s1;  const int* CR = sw ? J.c2 : J.c1;
    const long long* SC = sw ? J.s1 : J.s2;  const int* CC = sw ? J.c1 : J.c2;
    const uint32_t WR = sw ? w2 : w1, WC = sw ? w1 : w2;
    const int nR = (int)(sw ? J.card2 : J.card1), nC = (int)(sw ? J.card1 : J.card2);
    if (tid == 0) {
        const int cs = sw ? 0 : 1;                                    // the column side
        const unsigned long long smax = sm_red[cs][1];
        const int wide = (int)(sm_red[cs][2] & 1);
        DpMeta m;
        m.SR = SR; m.CR = CR; m.SC = SC; m.CC = CC; m.WR = WR; m.WC = WC; m.nR = nR; m.nC = nC; m.var = var; m.sw = sw;
        m.bad = var == 2 && ((sm_red[0][2] | sm_red[1][2]) & 2) ? 1 : 0;
        // column-pair scores: IMMA byte-digit planes need 32-bit scores and counters of one (card <= 127) or two
        // (<= 32767) byte digits; |T| <= max|score| * (sum of the row's counters <= 7 * card) decides the ring's width
        m.tmode = var != 2 ? 2 : (wide ? 2 : (nR <= 127 ? 0 : (nR <= 32767 ? 1 : 2)));
        m.t32 = var == 2 ? smax < (1ull << 31) / (7ull * (unsigned long long)nR) : smax < (1ull << 31);
        P.meta[jid] = m;
    }
    const Scratch L(J.w1, J.w2);
    unsigned char* scratch = P.scratch + J.scratch_off;
    long long* col = reinterpret_cast<long long*>(scratch + L.col);
    unsigned long long* browg = reinterpret_cast<unsigned long long*>(scratch + L.brow);
    const long long go = P.go, ge = P.ge, to = P.to, te = P.te;

    // column records (structure of arrays)
    for (uint32_t j = tid; j <= WC; j += nthr) {
        ColInfo ci = {0, 0, 0, 0, 0, 0, 0, 0};
        if (j >= 1 && var != 0) {
            int s_o, s_e, s_to, s_te, k_e, k_te;
            solve_gaps(CC, j, WC, nC, s_o, s_e, s_to, s_te, k_e, k_te);
            const int* cc = CC + (size_t)j * 32;
            const long long* sc = SC + (size_t)j * 32;
            ci.cgo = sc[kGapGO]; ci.cge = sc[kGapGE]; ci.cto = sc[kGapTO]; ci.cte = sc[kGapTE];
            ci.chg = (long long)cc[kGapGO] * (ge - go) + (long long)cc[kGapTO] * (te - to);
            if (var == 2) { ci.b0 = pack2(s_o, s_e); ci.b1 = pack2(s_to, s_te); ci.b2 = pack2(k_e, k_te); }
            else { ci.b0 = go * s_o + ge * s_e + to * s_to + te * s_te; ci.b1 = ge * k_e + te * k_te; }
        }
        const long long v[kColFields] = {ci.cgo, ci.cge, ci.cto, ci.cte, ci.chg, ci.b0, ci.b1, ci.b2};
#pragma unroll
        for (int f = 0; f < kColFields; ++f) col[(size_t)f * L.cstride + j] = v[f];
    }
    // row 0 (profile_par.cpp:531-555; SeqSeq profile_seq.cpp:48-69): H(0, j) is a running sum over the columns --
    // every thread sums a contiguous segment, the segment totals are combined through shared memory
    {
        __shared__ long long sm_wsum[kPrepThreads / 32];
        auto term = [&](uint32_t j) -> long long {
            const long long* sc = SC + (size_t)j * 32;
            if (var == 0) return j == 1 ? to : te;             // max(H, D = NEG) + te
            if (var == 1) return j == 1 ? sc[kGapTO] : sc[kGapTE];
            return (j == 1 ? sc[kGapTO] : sc[kGapTE]) * nR;
        };
        const uint32_t seg = (WC + nthr - 1) / nthr;
        const uint32_t ja = 1 + tid * seg, jb = ja + seg - 1 < WC ? ja + seg - 1 : WC;
        long long sum = 0;
        for (uint32_t j = ja; j <= jb; ++j) sum += term(j);
        // exclusive prefix of the segment sums: warp scan, then the warp totals
        long long incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long v = shfl_up_ll_by(incl, o);
            if ((int)(tid & 31) >= o) incl += v;
        }
        if ((tid & 31) == 31) sm_wsum[tid >> 5] = incl;
        __syncthreads();
        long long h = incl - sum;
        for (uint32_t u = 0; u < (tid >> 5); ++u) h += sm_wsum[u];
        for (uint32_t j = ja; j <= jb; ++j) {
            h += term(j);
            park_cell(browg + (size_t)j * kBrowWords, Cell{kNegInf, j == WC ? kNegInf : h, kNegInf, 0}, 1);
        }
        if (tid == 0) park_cell(browg, Cell{0, kNegInf, kNegInf, 0}, 1);
    }
}

__global__ void __launch_bounds__(kPrepThreads) k_dp_prep(const DpParams P)
{
    prep_body(P, P.job_base + blockIdx.x);
}

// Caller-visible CDPMatrix bytes (row-major, row 0 all-H, column 0 all-V) from the skewed internal directions.
// Skewed (wavefront-major) storage: stripe k (rows 32k+1 .. 32k+32), wavefront step s, lane l hold cell (32k+1+l, s-l),
// so one warp step of k_dp_fill writes 32 consecutive bytes.
__device__ __forceinline__ unsigned char dir_at(const unsigned char* __restrict__ sdirs, size_t steps, uint32_t i, uint32_t j)
{
    if (i == 0) return j ? (unsigned char)(1 | 1 << 2 | 1 << 4) : 0;
    const uint32_t q = i - 1, l = q & 31;
    return __ldcg(sdirs + ((size_t)(q >> 5) * steps + (j + l)) * 32 + l);
}

__global__ void __launch_bounds__(kTThreads) k_dp_unskew(const DpParams P)
{
    uint32_t lo = 0, hi = P.n_jobs;
    const unsigned long long b = blockIdx.x;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) / 2;
        if (P.tblock[mid] <= b) lo = mid; else hi = mid;
    }
    const uint32_t jid = P.job_base + lo;
    const DpJobDev J = P.jobs[jid];
    const DpMeta M = P.meta[jid];
    if (M.bad == 2) return;
    const size_t ldc = (size_t)M.WC + 1, steps = (size_t)M.WC + 32;
    const size_t cells = ((size_t)M.WR + 1) * ldc;
    const unsigned char* sd = P.sdirs + J.t_off;
    unsigned char* out = P.dirs + J.dirs_off;
    const size_t base = (size_t)(b - P.tblock[lo]) * kTThreads * kTCellsPerThread;
#pragma unroll
    for (int u = 0; u < kTCellsPerThread; ++u) {
        const size_t c = base + (size_t)u * kTThreads + threadIdx.x;
        if (c >= cells) break;
        const uint32_t i = (uint32_t)c / (uint32_t)ldc, j = (uint32_t)c - i * (uint32_t)ldc;
        out[c] = dir_at(sd, steps, i, j);
    }
}

// ------------------------------------------------------------------------------------------------
// k_dp_fill: the recurrence + traceback
// ------------------------------------------------------------------------------------------------

// T tile of one chunk (columns 8m .. 8m+7, the stripe's 32 rows) on the tensor cores: every score fits in int32 and the
// row profile has at most 127 (NDA = 1) or 32767 (NDA = 2) members, so every counter is one or two byte digits and
// T = C x S^T is an exact integer GEMM with K = 32 symbols.  Scores are split into four byte digits (three unsigned, the
// top one signed); IMMA.16832 accumulates each digit plane in int32 (30 x 255 x 255 < 2^21) and the planes are
// recombined with shifts in 64 bits.  The 8 columns are one n-tile, the 32 rows two m-tiles.
template <int NDA, bool T32>
__device__ __forceinline__ void t_tile_mma(const unsigned (&afrag)[2][2][4], const long long (*S2s)[kS2Stride], uint32_t m,
                                           long long (*tring)[32])
{
    const uint32_t lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
    unsigned bfrag[4][2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const longlong2 p = *reinterpret_cast<const longlong2*>(&S2s[g][h * 16 + t4 * 4]);
        const longlong2 q = *reinterpret_cast<const longlong2*>(&S2s[g][h * 16 + t4 * 4 + 2]);
        const unsigned v0 = (unsigned)p.x, v1 = (unsigned)p.y, v2 = (unsigned)q.x, v3 = (unsigned)q.y;
        const unsigned t01 = __byte_perm(v0, v1, 0x5140), t23 = __byte_perm(v2, v3, 0x5140);   // bytes 0,1 interleaved
        const unsigned u01 = __byte_perm(v0, v1, 0x7362), u23 = __byte_perm(v2, v3, 0x7362);   // bytes 2,3 interleaved
        bfrag[0][h] = __byte_perm(t01, t23, 0x5410); bfrag[1][h] = __byte_perm(t01, t23, 0x7632);
        bfrag[2][h] = __byte_perm(u01, u23, 0x5410); bfrag[3][h] = __byte_perm(u01, u23, 0x7632);
    }
    int* tring32 = reinterpret_cast<int*>(tring);
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        long long out[4] = {0, 0, 0, 0};
#pragma unroll
        for (int da = 0; da < NDA; ++da) {
            int acc[4][4];
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                acc[d][0] = acc[d][1] = acc[d][2] = acc[d][3] = 0;
                if (d < 3)
                    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                                 : "+r"(acc[d][0]), "+r"(acc[d][1]), "+r"(acc[d][2]), "+r"(acc[d][3])
                                 : "r"(afrag[da][mt][0]), "r"(afrag[da][mt][1]), "r"(afrag[da][mt][2]), "r"(afrag[da][mt][3]),
                                   "r"(bfrag[d][0]), "r"(bfrag[d][1]));
                else
                    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                                 : "+r"(acc[d][0]), "+r"(acc[d][1]), "+r"(acc[d][2]), "+r"(acc[d][3])
                                 : "r"(afrag[da][mt][0]), "r"(afrag[da][mt][1]), "r"(afrag[da][mt][2]), "r"(afrag[da][mt][3]),
                                   "r"(bfrag[d][0]), "r"(bfrag[d][1]));
            }
#pragma unroll
            for (int c = 0; c < 4; ++c)
                out[c] += ((long long)acc[0][c] + ((long long)acc[1][c] << 8) + ((long long)acc[2][c] << 16) + ((long long)acc[3][c] << 24)) << (8 * da);
        }
        // c0,c1: row g, columns 2*t4, 2*t4+1;  c2,c3: row g+8.  Cell (row r, column j) is consumed at wavefront step j + r.
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const uint32_t r = (uint32_t)mt * 16 + g + (c >> 1) * 8;
            const uint32_t s = m * kChunk + t4 * 2 + (c & 1) + r;
            const uint32_t slot = s % kTRing;
            if (T32) tring32[slot * 32 + r] = (int)out[c];
            else tring[slot][r] = out[c];
        }
    }
}

// One wavefront step of one lane: cell (i, j), j = s - lane.  GUARD = true is the general form (ramp-in: the lane may
// not have reached column 1 yet; tail: it may be past column WC, or on it); GUARD = false is the steady state, where
// every lane is strictly inside the matrix (2 <= j < WC), so nothing has to be protected or special-cased.
struct RowConst {                 // per-lane constants of the stripe
    unsigned s_o, s_e, s_to, s_te, k_e, k_te, g1o, g1t, nongap1;
    long long srgo, srge, srto, srte;
    long long hgo, hge;           // SeqSeq: scalar gap costs of the H update (terminal on the last row)
    const long long* p_gch; const long long* p_conth;   // SeqProf: the column-record fields the H update reads (terminal on the last row)
    bool valid, last_row, row_gt1;
};

template <int VAR, bool T32, bool GUARD>
__device__ __forceinline__ void dp_step(WarpShared& W, const RowConst& R, const Cell* chunk, uint32_t u, uint32_t s, uint32_t lane,
                                        uint32_t WC, uint32_t tslot, Cell& cur, Cell& up, long long go, long long ge, long long to, long long te,
                                        unsigned char* __restrict__ dk, long long* last_out)
{
    const int* tring32 = reinterpret_cast<const int*>(W.t);
    const int j = (int)s - (int)lane;                        // column handled now
    const long long t = T32 ? (long long)tring32[tslot * 32 + lane] : W.t[tslot][lane];
    const uint32_t slot = (uint32_t)j & (kRing - 1);
    // (i-1, j): the lane above computed it one step ago; lane 0 takes it from the boundary row
    Cell U;
    U.D = shfl_up_ll(cur.D); U.H = shfl_up_ll(cur.H); U.V = shfl_up_ll(cur.V);
    if (lane == 0) { const Cell B = chunk[u]; U.D = B.D; U.H = B.H; U.V = B.V; }
    const Cell Pd = up;                                      // (i-1, j-1)
    up = U;
    const Cell L = cur;
    const bool three = GUARD ? (R.row_gt1 && j > 1) : R.row_gt1;
    Cell out;
    out.pad = 0;
    int db;
    if (VAR == 0) {
        // profile_seq.cpp:86-140 (note the >= in the second D test)
        const bool dw = (Pd.D > Pd.H) & (Pd.D > Pd.V), hw = Pd.H >= Pd.V;
        out.D = (dw ? Pd.D : (hw ? Pd.H : Pd.V)) + t;
        db = dw ? 0 : (hw ? 1 : 2);
        long long tD = L.D + R.hgo;
        const long long tH = L.H + R.hge;
        out.H = tD > tH ? tD : tH; db |= tD > tH ? 0 : 1 << 2;
        const bool inner = GUARD ? j < (int)WC : true;
        tD = U.D + (inner ? go : to);
        const long long tV = U.V + (inner ? ge : te);
        out.V = tD > tV ? tD : tV; db |= tD > tV ? 0 : 2 << 4;
    } else if (VAR == 1) {
        // profile_par.cpp:255-421
        db = pick3(Pd.D, Pd.H, Pd.V + W.col[4][slot], 0, 1, 2, out.D);
        out.D += t;
        const long long gcH = R.p_gch[slot];
        long long tD = L.D + gcH;
        const long long tH = L.H + R.p_conth[slot];
        db |= pick3(tD, three ? L.V + gcH : kNever, tH, 0, 2 << 2, 1 << 2, out.H);
        const long long b0 = W.col[5][slot];
        tD = U.D + b0;
        const long long tV = U.V + W.col[6][slot];
        db |= pick3(tD, three ? U.H + b0 : kNever, tV, 0, 1 << 4, 2 << 4, out.V);
    } else {
        // profile_par.cpp:679-886
        const long long cgo = W.col[0][slot], cge = W.col[1][slot], cto = W.col[2][slot], cte = W.col[3][slot];
        const long long b0 = W.col[5][slot], b1 = W.col[6][slot], b2 = W.col[7][slot];
        long long tD = Pd.D + t;
        long long tH = Pd.H + t;
        tH += (cge - cgo) * R.g1o + (cte - cto) * R.g1t;       // == 0 when both counts are 0
        long long tV = Pd.V + t + W.col[4][slot] * R.nongap1;
        db = pick3(tD, tH, tV, 0, 1, 2, out.D);
        const long long gcH = cgo * R.s_o + cge * R.s_e + cto * R.s_to + cte * R.s_te;
        tD = L.D + gcH;
        tH = L.H + cge * R.k_e + cte * R.k_te;
        db |= pick3(tD, three ? L.V + gcH : kNever, tH, 0, 2 << 2, 1 << 2, out.H);
        const long long gcV = R.srgo * ulo32(b0) + R.srge * uhi32(b0) + R.srto * ulo32(b1) + R.srte * uhi32(b1);
        tD = U.D + gcV;
        tV = U.V + R.srge * ulo32(b2) + R.srte * uhi32(b2);
        db |= pick3(tD, three ? U.H + gcV : kNever, tV, 0, 1 << 4, 2 << 4, out.V);
    }
    if (GUARD) {
        // `cur` only has to be protected while the lane still waits for its first column; what it holds past the last
        // column is never read.
        const bool commit = j >= 1;
        const bool active = R.valid && j >= 1 && j <= (int)WC;
        cur.D = commit ? out.D : cur.D; cur.H = commit ? out.H : cur.H; cur.V = commit ? out.V : cur.V;
        if (active) dk[(size_t)s * 32 + lane] = (unsigned char)db;
        if (active && R.last_row && j == (int)WC) { last_out[0] = out.D; last_out[1] = out.H; last_out[2] = out.V; }
    } else {
        cur.D = out.D; cur.H = out.H; cur.V = out.V;
        if (R.valid) dk[(size_t)s * 32 + lane] = (unsigned char)db;
    }
    // the stripe's last row goes to the boundary row once per chunk (see dp_stripes); staged here without a branch
    if (lane == 31) { W.park[u][0] = out.D; W.park[u][1] = out.H; W.park[u][2] = out.V; }
}

// ---- producer / consumer split of a ProfProf stripe (k_dp_fill_duo) ---------------------------------------------
// A warp that runs a stripe alone on its SM sub-partition issues an instruction every 2.2 cycles: the step is one long
// schedule of dependent 64-bit operations.  Roughly two thirds of its instructions do not depend on the DP state at all:
// staging, the tensor-core T tile, and per cell seven int64 terms that combine the column record with the row's counts
// (profile_par.cpp:679-886).  A PRODUCER warp on the same sub-partition computes those into a shared-memory ring, one
// chunk (8 steps x 7 terms x 32 lanes) at a time; the CONSUMER warp is left with the compare / select chain, the
// shuffles and the boundary row.  Two named barriers per buffer (full / empty), two buffers.
constexpr int kTermFields = 7;
struct __align__(16) DuoTerms { long long v[2][kChunk][kTermFields][32]; };
struct __align__(16) DuoShared { WarpShared w; DuoTerms t; };

// Named barriers (bar.sync / bar.arrive, 64 threads = the two warps of a pair): the producer ARRIVES on full[b] after it
// has written buffer b and the consumer SYNCs on it before reading; the consumer arrives on empty[b] when it is done and the
// producer syncs on that before it refills.  Four barrier ids per pair, sixteen per block -- all there are.
__device__ __forceinline__ void pair_sync(uint32_t id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void pair_arrive(uint32_t id) { asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }

// the consumer's step: dp_step<2, ...> with the state-independent terms read from the ring
template <bool GUARD>
__device__ __forceinline__ void dp_step_duo(WarpShared& W, const RowConst& R, const long long* __restrict__ tv, const Cell* chunk, uint32_t u,
                                            uint32_t s, uint32_t lane, uint32_t WC, Cell& cur, Cell& up, unsigned char* __restrict__ dk,
                                            long long* last_out)
{
    const int j = (int)s - (int)lane;
    const long long a1 = tv[0], a2 = tv[32], a3 = tv[64], gcH = tv[96], contH = tv[128], gcV = tv[160], contV = tv[192];
    Cell U;
    U.D = shfl_up_ll(cur.D); U.H = shfl_up_ll(cur.H); U.V = shfl_up_ll(cur.V);
    if (lane == 0) { const Cell B = chunk[u]; U.D = B.D; U.H = B.H; U.V = B.V; }
    const Cell Pd = up;
    up = U;
    const Cell L = cur;
    const bool three = GUARD ? (R.row_gt1 && j > 1) : R.row_gt1;
    Cell out;
    out.pad = 0;
    int db = pick3(Pd.D + a1, Pd.H + a2, Pd.V + a3, 0, 1, 2, out.D);
    long long tD = L.D + gcH;
    const long long tH = L.H + contH;
    db |= pick3(tD, three ? L.V + gcH : kNever, tH, 0, 2 << 2, 1 << 2, out.H);
    tD = U.D + gcV;
    const long long tV = U.V + contV;
    db |= pick3(tD, three ? U.H + gcV : kNever, tV, 0, 1 << 4, 2 << 4, out.V);
    if (GUARD) {
        const bool commit = j >= 1;
        const bool active = R.valid && j >= 1 && j <= (int)WC;
        cur.D = commit ? out.D : cur.D; cur.H = commit ? out.H : cur.H; cur.V = commit ? out.V : cur.V;
        if (active) dk[(size_t)s * 32 + lane] = (unsigned char)db;
        if (active && R.last_row && j == (int)WC) { last_out[0] = out.D; last_out[1] = out.H; last_out[2] = out.V; }
    } else {
        cur.D = out.D; cur.H = out.H; cur.V = out.V;
        if (R.valid) dk[(size_t)s * 32 + lane] = (unsigned char)db;
    }
    if (lane == 31) { W.park[u][0] = out.D; W.park[u][1] = out.H; W.park[u][2] = out.V; }
}

// One team = NW warps (x CL thread blocks of a cluster) working on one merge.  Stripe k (rows 32k+1 .. 32k+32)
// belongs to team warp k % (NW*CL).  A warp works through its stripe chunk by chunk.  The last row of a stripe is parked
// in the job's boundary row (L2) as TAGGED words -- every 8-byte word carries the number of the stripe that wrote it in
// its upper half -- so the stripe below needs neither a flag nor a fence: it loads the next chunk's words one chunk
// ahead (the loads fly during the 8 steps of the current chunk), looks at the tags afterwards and simply reloads until
// all of them are the ones it expects.  Its lane 0 needs column 8c+7 of the stripe above, which that stripe's lane 31
// computes at wavefront step 8c+38: the natural lag between consecutive stripes is about six chunks, self-regulating.
// ROLE 0: one warp does everything; 1: producer, 2: consumer of a duo (VAR == 2 only; DT, bars, gcount: the pair's ring, the first of
// its four barrier ids {full0, full1, empty0, empty1} and the running count of chunks both warps keep)
template <int VAR, bool T32, int ROLE = 0>
__device__ __forceinline__ void dp_stripes(const DpParams& P, const DpMeta& M, const long long* __restrict__ col, uint32_t cstride,
                                           unsigned long long* __restrict__ browg,
                                           unsigned char* __restrict__ dirs, uint32_t team_warp, uint32_t TW,
                                           long long* last_out, WarpShared& W, DuoTerms* DT = nullptr, uint32_t bars = 0,
                                           uint32_t gcount = 0)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t WR = M.WR, WC = M.WC;
    const long long go = P.go, ge = P.ge, to = P.to, te = P.te;
    const uint32_t n_stripes = (WR + 31) / 32;
    const uint32_t steps = WC + 1 + 31;                              // wavefront steps per stripe
    const uint32_t S = (steps + kChunk - 1) / kChunk;                // macro steps per stripe
    int* const tring32 = reinterpret_cast<int*>(W.t);

    for (uint32_t k = team_warp; k < n_stripes; k += TW) {                // TW = warps in the team
        // ---- row-side constants into registers
        const uint32_t i = k * 32 + 1 + lane;
        RowConst R;
        R.valid = i <= WR;
        R.last_row = i == WR;
        R.row_gt1 = i > 1;
        R.s_o = R.s_e = R.s_to = R.s_te = R.k_e = R.k_te = R.g1o = R.g1t = R.nongap1 = 0;
        R.srgo = R.srge = R.srto = R.srte = 0;
        R.hgo = !R.last_row ? go : to; R.hge = !R.last_row ? ge : te;
        R.p_gch = W.col[!R.last_row ? 0 : 2]; R.p_conth = W.col[!R.last_row ? 1 : 3];
        long long col0cost = 0;
        uint32_t residue = 22;
        if (R.valid) {
            if (VAR == 2) {
                const int* rc = M.CR + (size_t)i * 32;
                int a, b, c, d, e, f;
                solve_gaps(M.CR, i, WR, M.nR, a, b, c, d, e, f);
                R.s_o = (unsigned)a; R.s_e = (unsigned)b; R.s_to = (unsigned)c; R.s_te = (unsigned)d; R.k_e = (unsigned)e; R.k_te = (unsigned)f;
                R.g1o = (unsigned)rc[kGapGO]; R.g1t = (unsigned)rc[kGapTO];
                for (int q = 0; q < 24; ++q) R.nongap1 += (unsigned)rc[q];
                const long long* sr = M.SR + (size_t)i * 32;
                R.srgo = sr[kGapGO]; R.srge = sr[kGapGE]; R.srto = sr[kGapTO]; R.srte = sr[kGapTE];
                col0cost = (i == 1 ? R.srto : R.srte) * M.nC;
            } else {
                residue = (uint32_t)seq_symbol(M.CR, i);
                if (VAR == 1) col0cost = (i == 1 ? to : te) * M.nC;
                else col0cost = i == 1 ? to : te;
            }
        }
        // A fragments of the IMMA tile (counters of the stripe's rows as byte digits): h&1 = row +8, h>>1 = symbols 16..31
        unsigned afrag[2][2][4];
        if (VAR == 2 && M.tmode < 2 && ROLE != 2) {
            const uint32_t g = lane >> 2, t4 = lane & 3;
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    const uint32_t row = k * 32 + 1 + (uint32_t)mt * 16 + g + (h & 1) * 8, kk = (h >> 1) * 16 + t4 * 4;
                    unsigned lo = 0, hi = 0;
                    if (row <= WR) {
                        const int4 c = *reinterpret_cast<const int4*>(M.CR + (size_t)row * 32 + kk);
                        const unsigned x = (unsigned)c.x, y = (unsigned)c.y, z = (unsigned)c.z, w = (unsigned)c.w;
                        lo = (x & 0xffu) | (y & 0xffu) << 8 | (z & 0xffu) << 16 | (w & 0xffu) << 24;
                        hi = (x >> 8 & 0xffu) | (y >> 8 & 0xffu) << 8 | (z >> 8 & 0xffu) << 16 | (w >> 8 & 0xffu) << 24;
                        if (kk == 28) { lo &= 0xffffu; hi &= 0xffffu; }     // rows 30 (GAP) and 31 (GUARD) are not part of the sum
                    }
                    afrag[0][mt][h] = lo;
                    afrag[1][mt][h] = hi;
                }
        }
        Cell cur = {kNegInf, kNegInf, kNegInf, 0}, up = {kNegInf, kNegInf, kNegInf, 0};
        unsigned char* dk = dirs + (size_t)k * 32 * steps;           // this stripe's skewed directions: (s, lane) at [s * 32 + lane]
        const uint32_t tag_in = k + 1, tag_out = k + 2;               // k_dp_prep writes row 0 with tag 1
        // columns c0 .. c0+7 of the column records and of the column profile's scores -> this warp's windows
        auto request = [&](uint32_t chunk) {
            const uint32_t c0 = chunk * kChunk, buf = chunk & 1;
            if (VAR != 0) {
                const uint32_t f = lane >> 2, c = c0 + 2u * (lane & 3);
                if (c <= WC) cp_async16(&W.col[f][c & (kRing - 1)], col + (size_t)f * cstride + c);
            }
#pragma unroll
            for (uint32_t q = lane; q < kChunk * 16; q += 32) {
                const uint32_t cc = q >> 4, piece = q & 15;
                if (c0 + cc <= WC) cp_async16(&W.s2[buf][cc][piece * 2], M.SC + (size_t)(c0 + cc) * 32 + piece * 2);
            }
            cp_async_commit();
        };
        // boundary cells of a chunk: lanes 0..23 own one 16-byte unit (two tagged words) each -- value `which` of column c0 + cq
        const uint32_t cq = lane / 3, which = lane - cq * 3;
        ulonglong2 bw = make_ulonglong2(0, 0);
        auto brow_load = [&](uint32_t chunk) {
            const uint32_t c = chunk * kChunk + cq;
            if (lane < 24 && c <= WC) bw = ld_cg_v2(browg + (size_t)c * kBrowWords + which * 2);
        };
        auto brow_land = [&](uint32_t chunk) {                    // waits until the chunk loaded into `bw` is the one parked by the stripe above
            const uint32_t c = chunk * kChunk + cq;
            const bool mine = lane < 24 && c <= WC;
            for (;;) {
                const bool ok = !mine || ((uint32_t)(bw.x >> 32) == tag_in && (uint32_t)(bw.y >> 32) == tag_in);
                if (__all_sync(0xffffffffu, ok)) break;
                __nanosleep(32);
                if (!ok) bw = ld_cg_v2(browg + (size_t)c * kBrowWords + which * 2);
            }
            if (mine) {
                long long* dst = reinterpret_cast<long long*>(&W.brow[chunk & 1][cq]);
                dst[which] = (long long)((bw.x & 0xffffffffull) | (bw.y << 32));
            }
        };
        if (ROLE != 1) brow_load(0);
        if (ROLE != 2) request(0);
        if (ROLE != 1) brow_land(0);
        const bool stripe_parks = k * 32 + 32 < WR;                   // lane 31 holds a row that has a row below it

        for (uint32_t m = 0; m < S; ++m) {
            const bool has_next = (m + 1) * kChunk <= WC;
            if (ROLE != 1 && has_next) brow_load(m + 1);              // in flight during the tile and the 8 steps below
            if (ROLE != 2) {
            cp_async_wait_all();
            __syncwarp();
            }
            // ---- the chunk's tile of column-pair scores into the T ring
            if (ROLE != 2 && m * kChunk <= WC) {
                const long long (*S2s)[kS2Stride] = W.s2[m & 1];
                if (VAR == 2) {
                    if (M.tmode == 0) t_tile_mma<1, T32>(afrag, S2s, m, W.t);
                    else if (M.tmode == 1) t_tile_mma<2, T32>(afrag, S2s, m, W.t);
                    else {
                        // scores beyond int32 or more than 32767 members: 30 multiply-adds per cell, counters >= 0
                        const int4* rc = reinterpret_cast<const int4*>(M.CR + (size_t)(R.valid ? i : 1) * 32);
                        unsigned long long acc[kChunk];
                        unsigned acch[kChunk];
#pragma unroll
                        for (int c = 0; c < kChunk; ++c) { acc[c] = 0; acch[c] = 0; }
#pragma unroll 1
                        for (int k4 = 0; k4 < 8; ++k4) {
                            const int4 cv4 = rc[k4];
                            const unsigned cv[4] = {(unsigned)cv4.x, (unsigned)cv4.y, (unsigned)cv4.z, (unsigned)cv4.w};
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int kk = 4 * k4 + u;
                                if (kk < 30) {
#pragma unroll
                                    for (int c = 0; c < kChunk; ++c) {
                                        const unsigned long long sv = (unsigned long long)S2s[c][kk];
                                        acc[c] += (unsigned long long)cv[u] * (unsigned)sv;
                                        acch[c] += cv[u] * (unsigned)(sv >> 32);
                                    }
                                }
                            }
                        }
#pragma unroll
                        for (int c = 0; c < kChunk; ++c) {
                            const uint32_t slot = (m * kChunk + c + lane) % kTRing;
                            const long long v = (long long)(acc[c] + ((unsigned long long)acch[c] << 32));
                            if (T32) tring32[slot * 32 + lane] = (int)v; else W.t[slot][lane] = v;
                        }
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < kChunk; ++c) {
                        const uint32_t slot = (m * kChunk + c + lane) % kTRing;
                        const long long v = S2s[c][residue];
                        if (T32) tring32[slot * 32 + lane] = (int)v; else W.t[slot][lane] = v;
                    }
                }
            }
            if (ROLE != 2) {
            __syncwarp();
            if (has_next) request(m + 1);                             // static data: no dependence on the stripe above
            }
            const uint32_t s_begin = m * kChunk;
            const uint32_t tb = gcount & 1;                           // duo: buffer and use number of this chunk
            if (ROLE == 1) {
                // ---- producer: the seven state-independent terms of the chunk's 8 x 32 cells into the ring
                if (gcount >= 2) pair_sync(bars + 2 + tb);                // the consumer is done with the buffer's previous chunk
#pragma unroll 2
                for (uint32_t u = 0; u < (uint32_t)kChunk; ++u) {
                    const uint32_t sst = s_begin + u;
                    const uint32_t slot = (sst - lane) & (kRing - 1), tslot = sst & (kTRing - 1);
                    const long long t = T32 ? (long long)tring32[tslot * 32 + lane] : W.t[tslot][lane];
                    const long long cgo = W.col[0][slot], cge = W.col[1][slot], cto = W.col[2][slot], cte = W.col[3][slot];
                    const long long b0 = W.col[5][slot], b1 = W.col[6][slot], b2 = W.col[7][slot];
                    long long* tv = &DT->v[tb][u][0][lane];
                    tv[0] = t;
                    tv[32] = t + ((cge - cgo) * R.g1o + (cte - cto) * R.g1t);
                    tv[64] = t + W.col[4][slot] * R.nongap1;
                    tv[96] = cgo * R.s_o + cge * R.s_e + cto * R.s_to + cte * R.s_te;
                    tv[128] = cge * R.k_e + cte * R.k_te;
                    tv[160] = R.srgo * ulo32(b0) + R.srge * uhi32(b0) + R.srto * ulo32(b1) + R.srte * uhi32(b1);
                    tv[192] = R.srge * ulo32(b2) + R.srte * uhi32(b2);
                }
                pair_arrive(bars + tb);
                ++gcount;
                continue;
            }
            if (ROLE == 2) pair_sync(bars + tb);                      // the chunk's terms are in the ring
            const Cell* chunk = W.brow[m & 1];
            if (m == 0) {
                // Column 0 of the stripe (profile_par.cpp:625-640) in closed form, so that the step below never sees
                // j == 0:  D = H = NEG and V(i, 0) = max(D, V)(i-1, 0) + cost_i, a running sum down the rows (D(i-1, 0)
                // is NEG below row 0).  `cur` starts as that cell, its direction byte (all-V) and, for the stripe's
                // last row, its boundary-row copy are written here -- after this stripe has read the old column 0.
                const Cell B = chunk[0];
                long long pre = col0cost;                               // 0 in lanes past the last row
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const long long v = shfl_up_ll_by(pre, o);
                    if ((int)lane >= o) pre += v;
                }
                cur = Cell{kNegInf, kNegInf, R.last_row ? kNegInf : (B.D > B.V ? B.D : B.V) + pre, 0};
                if (R.valid) {
                    dk[(size_t)lane * 32 + lane] = (unsigned char)(2 | 2 << 2 | 2 << 4);
                    if (lane == 31 && !R.last_row) park_cell(browg, cur, tag_out);
                }
            }
            // steady state: every lane strictly inside the matrix during the whole macro step (j >= 2 and j < WC)
            const uint32_t tbase = s_begin & (kTRing - 1);
            if (ROLE == 2) {
                const long long* tv0 = &DT->v[tb][0][0][lane];
                if (m >= 5 && s_begin + kChunk - 1 < WC) {
#pragma unroll
                    for (uint32_t u = 0; u < (uint32_t)kChunk; ++u)
                        dp_step_duo<false>(W, R, tv0 + u * (kTermFields * 32), chunk, u, s_begin + u, lane, WC, cur, up, dk, last_out);
                } else {
#pragma unroll 2
                    for (uint32_t u = 0; u < (uint32_t)kChunk; ++u)
                        dp_step_duo<true>(W, R, tv0 + u * (kTermFields * 32), chunk, u, s_begin + u, lane, WC, cur, up, dk, last_out);
                }
            } else if (m >= 5 && s_begin + kChunk - 1 < WC) {
#pragma unroll
                for (uint32_t u = 0; u < (uint32_t)kChunk; ++u)
                    dp_step<VAR, T32, false>(W, R, chunk, u, s_begin + u, lane, WC, tbase + u, cur, up, go, ge, to, te, dk, last_out);
            } else {
#pragma unroll 2
                for (uint32_t u = 0; u < (uint32_t)kChunk; ++u)
                    dp_step<VAR, T32, true>(W, R, chunk, u, s_begin + u, lane, WC, tbase + u, cur, up, go, ge, to, te, dk, last_out);
            }
            __syncwarp();
            if (ROLE == 2) { pair_arrive(bars + 2 + tb); ++gcount; }    // the ring buffer may be refilled
            // park the eight cells lane 31 produced: 24 lanes tag and store one 16-byte unit each (value `which` of step cq)
            if (stripe_parks && lane < 24) {
                const int j = (int)(s_begin + cq) - 31;
                if (j >= 1 && j <= (int)WC) {
                    const unsigned long long v = (unsigned long long)W.park[cq][which], t = (unsigned long long)tag_out << 32;
                    __stcg(reinterpret_cast<ulonglong2*>(browg + (size_t)j * kBrowWords + which * 2),
                           make_ulonglong2(t | (unsigned)v, t | (unsigned)(v >> 32)));
                }
            }
            if (has_next) { brow_land(m + 1); __syncwarp(); }
        }
    }
}

// NW == 1: four independent merges per 128-thread block (one warp each).  NW > 1: one merge per block.  CLUSTERED: one
// merge per thread-block CLUSTER (2 .. 16 blocks, chosen per launch): consecutive stripes go to different blocks (stripe
// k -> block k % CL, warp (k / CL) % NW), so that a merge with few stripes has one stripe per SM sub-partition -- two
// active stripes on one sub-partition share its ALU pipe (one warp instruction per two cycles) and both run at half
// speed, which is the wrong trade when a single merge is all there is to do (the top of the guide tree, where the
// reference switches to its multi-threaded ParAlign* variants).  The boundary row travels through L2 either way.  There
// is no barrier anywhere: a warp leaves when its stripes are done, the owner of cell (WR, WC) leaves (D, H, V) in the
// job's scratch for k_dp_trace.
// the stripes of merge `jid` that belong to team warp `team_warp` of `TW`
template <bool ONLY32 = false>
__device__ __forceinline__ void fill_body(const DpParams& P, uint32_t jid, uint32_t team_warp, uint32_t TW, WarpShared& W)
{
    const DpJobDev J = P.jobs[jid];
    const DpMeta M = P.meta[jid];
    if (M.bad == 2) return;                                          // a child failed: k_dp_trace reports it

    const Scratch L(J.w1, J.w2);
    unsigned char* scratch = P.scratch + J.scratch_off;
    const long long* col = reinterpret_cast<const long long*>(scratch + L.col);
    const uint32_t cstride = (uint32_t)L.cstride;
    unsigned long long* browg = reinterpret_cast<unsigned long long*>(scratch + L.brow);
    long long* g_last = reinterpret_cast<long long*>(scratch + L.lastv);
    unsigned char* dirs = P.sdirs + J.t_off;
#define FB_STRIPES(V, T) dp_stripes<V, T>(P, M, col, cstride, browg, dirs, team_warp, TW, g_last, W)
    if (M.var == 0) { if (ONLY32 || M.t32) FB_STRIPES(0, true); else FB_STRIPES(0, false); }
    else if (M.var == 1) { if (ONLY32 || M.t32) FB_STRIPES(1, true); else FB_STRIPES(1, false); }
    else { if (ONLY32 || M.t32) FB_STRIPES(2, true); else FB_STRIPES(2, false); }
#undef FB_STRIPES
}

template <int NW, bool CLUSTERED>
__global__ void __launch_bounds__((NW == 1 ? kDpWarps : NW) * 32, 1) k_dp_fill(const DpParams P)
{
    extern __shared__ __align__(16) unsigned char sm_dyn[];
    const uint32_t warp = threadIdx.x / 32;
    WarpShared& W = reinterpret_cast<WarpShared*>(sm_dyn)[warp];
    uint32_t CL = 1, cta_rank = 0;
    if (CLUSTERED) {
        CL = cooperative_groups::this_cluster().num_blocks();
        cta_rank = cooperative_groups::this_cluster().block_rank();
    }
    const uint32_t team_warp = NW == 1 ? 0 : warp * CL + cta_rank;
    const uint32_t TW = NW == 1 ? 1 : (uint32_t)NW * CL;
    const uint32_t slot = NW == 1 ? blockIdx.x * kDpWarps + warp : blockIdx.x / CL;
    if (slot >= P.n_jobs) return;                                    // whole warp (NW == 1) / whole team otherwise
    if (P.wide_only && P.meta[P.order[slot]].t32) return;            // k_dp_fill_compact has done this one
    fill_body(P, P.order[slot], team_warp, TW, W);
}

// Latency mode with producer / consumer pairs: eight warps per block, warp w < 4 consumes what warp w + 4 (same SM
// sub-partition) produces.  ProfProf merges only; any other merge runs on the four consumer warps with the one-warp code.
constexpr size_t kDuoSmem = 4 * sizeof(DuoShared);
__global__ void __launch_bounds__(256, 1) k_dp_fill_duo(const DpParams P)
{
    extern __shared__ __align__(16) unsigned char sm_dyn[];
    const uint32_t warp = threadIdx.x / 32, pair = warp & 3, producer = warp >> 2;
    DuoShared& DS = reinterpret_cast<DuoShared*>(sm_dyn)[pair];
    const uint32_t bars = pair * 4;                                   // barrier ids of this pair
    const uint32_t CL = cooperative_groups::this_cluster().num_blocks(), cta_rank = cooperative_groups::this_cluster().block_rank();
    const uint32_t team_warp = pair * CL + cta_rank, TW = 4 * CL;
    const uint32_t slot = blockIdx.x / CL;
    if (slot >= P.n_jobs) return;
    const uint32_t jid = P.order[slot];
    const DpJobDev J = P.jobs[jid];
    const DpMeta M = P.meta[jid];
    if (M.bad == 2) return;
    if (M.var != 2) {
        if (!producer) fill_body(P, jid, team_warp, TW, DS.w);
        return;
    }
    const Scratch L(J.w1, J.w2);
    unsigned char* scratch = P.scratch + J.scratch_off;
    const long long* col = reinterpret_cast<const long long*>(scratch + L.col);
    const uint32_t cstride = (uint32_t)L.cstride;
    unsigned long long* browg = reinterpret_cast<unsigned long long*>(scratch + L.brow);
    long long* g_last = reinterpret_cast<long long*>(scratch + L.lastv);
    unsigned char* dirs = P.sdirs + J.t_off;
    if (producer) {
        if (M.t32) dp_stripes<2, true, 1>(P, M, col, cstride, browg, dirs, team_warp, TW, g_last, DS.w, &DS.t, bars);
        else dp_stripes<2, false, 1>(P, M, col, cstride, browg, dirs, team_warp, TW, g_last, DS.w, &DS.t, bars);
    } else {
        if (M.t32) dp_stripes<2, true, 2>(P, M, col, cstride, browg, dirs, team_warp, TW, g_last, DS.w, &DS.t, bars);
        else dp_stripes<2, false, 2>(P, M, col, cstride, browg, dirs, team_warp, TW, g_last, DS.w, &DS.t, bars);
    }
}

// Throughput mode: the same stripes with 12 warps per SM instead of 8.  Two warps per SM sub-partition leave the issue slots
// half empty (the recurrence is a chain of dependent 64-bit compares and selects: ncu smsp__issue_active 53 %); the third
// needs the registers capped at 168 (ptxas spills 24 bytes) and the T ring in its 4-byte form.  One merge per block.
template <int NW>
__global__ void __launch_bounds__(NW * 32, 384 / (NW * 32)) k_dp_fill_compact(const DpParams P)
{
    extern __shared__ __align__(16) unsigned char sm_dyn[];
    const uint32_t warp = threadIdx.x / 32;
    WarpShared& W = *reinterpret_cast<WarpShared*>(sm_dyn + warp * kCompactStride);
    if (blockIdx.x >= P.n_jobs) return;
    const uint32_t jid = P.order[blockIdx.x];
    if (!P.meta[jid].t32) return;                                    // left to the k_dp_fill launch that follows
    fill_body<true>(P, jid, warp, NW, W);
}

// ------------------------------------------------------------------------------------------------
// k_dp_trace: the traceback of ConstructProfile (profile.cpp:727-775), one warp per merge.
// The direction bytes are stored skewed -- inside one 32-row stripe, wavefront step s = j + lane is the major index --
// so the 32 x 32 corner of the matrix that ends at the current cell is ONE contiguous run of at most 63 x 32 bytes when
// its rows are kept inside a stripe: the warp copies it with 16-byte loads, lane 0 walks inside it, repeat.
// ------------------------------------------------------------------------------------------------
constexpr int kTraceWarps = 4;
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned lds_u8(uint32_t a)
{
    unsigned v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
constexpr int kTraceWin = 96;               // wavefront steps per traceback window (3 KB); two windows per warp
constexpr int kSpecSlack = 16;              // columns the speculative window has to spare on either side of the diagonal
// one warp; tile: 2 * kTraceWin x 32 bytes of shared memory; all_dirs: the merge's whole skewed direction matrix already in shared
// memory (small merges in the fused kernel), or NULL
__device__ __forceinline__ void trace_body(const DpParams& P, uint32_t jid, unsigned char* tile, const unsigned char* all_dirs = nullptr)
{
    const uint32_t lane = threadIdx.x % 32;
    const DpJobDev J = P.jobs[jid];
    const DpMeta M = P.meta[jid];
    if (M.bad == 2) {                                                // a child failed: report, touch nothing else
        if (lane == 0) {
            famsa_dp_result r;
            memset(&r, 0, sizeof(r));
            r.path_offset = J.path_off; r.dirs_offset = J.dirs_off;
            r.variant = 0xFF;
            P.results[jid] = r;
            if (P.h_results) P.h_results[jid] = r;
            if (J.w_dst) *J.w_dst = kWidthBad;
        }
        return;
    }
    const Scratch L(J.w1, J.w2);
    unsigned char* scratch = P.scratch + J.scratch_off;
    unsigned char* tmp_path = scratch + L.tmp;
    const long long* g_last = reinterpret_cast<const long long*>(scratch + L.lastv);
    const unsigned char* dirs = P.sdirs + J.t_off;
    const uint32_t WR = M.WR, WC = M.WC;
    const size_t steps = (size_t)WC + 32;
    const long long last[3] = {__ldcg(g_last), __ldcg(g_last + 1), __ldcg(g_last + 2)};

    uint32_t n = 0;
    long long total;
    int dir;
    if (last[0] >= last[1] && last[0] >= last[2]) { dir = 0; total = last[0]; }
    else if (last[1] > last[2]) { dir = 1; total = last[1]; }
    else { dir = 2; total = last[2]; }
    uint32_t ti = WR, tj = WC;
    if (all_dirs && ti) {
        // the whole matrix is at hand: one uninterrupted walk down to row 0 (same index steps as below, D -65, H -32, V -33;
        // leaving a stripe through its first row re-bases the index on the stripe above)
        if (lane == 0) {
            uint32_t ii = ti, jj = tj, stripe = (ii - 1) >> 5;
            int l = (int)((ii - 1) & 31);
            uint32_t idx = (uint32_t)((stripe * steps + jj + l) * 32 + l);
            unsigned b = all_dirs[idx];
            unsigned char* out = tmp_path;
            for (;;) {
                *out++ = (unsigned char)dir;
                const int di = dir != 1, dj = dir != 2;
                if (dj && !jj) { ii = 0; jj = 0; break; }                // cannot happen for a valid matrix
                ii -= di; jj -= dj; l -= di; idx -= 32 * dj + 33 * di;
                if (l < 0) {
                    if (!ii) { dir = (int)((b >> (2 * dir)) & 3); break; }
                    l = 31; --stripe;
                    idx = (uint32_t)((stripe * steps + jj + 31) * 32 + 31);
                }
                const unsigned nb = all_dirs[idx];
                dir = (int)((b >> (2 * dir)) & 3);
                b = nb;
            }
            n = (uint32_t)(out - tmp_path);
            ti = ii; tj = jj;
        }
        ti = __shfl_sync(0xffffffffu, ti, 0);
        tj = __shfl_sync(0xffffffffu, tj, 0);
        dir = __shfl_sync(0xffffffffu, dir, 0);
        n = __shfl_sync(0xffffffffu, n, 0);
    }
    // Window = a run of wavefront steps [wsb, wsb + wn) of one stripe in shared memory; cell (l, j) of the stripe (l = row
    // inside it) sits at ((j + l) - wsb) * 32 + l, so the three moves are constant index steps: D -65, H -32, V -33.  While
    // lane 0 walks in one window, the loads of the NEXT one are already in flight: a path that keeps to the diagonal leaves
    // the stripe through its first row at column p = tj - (l_top + 1), so the steps around (stripe - 1, row 31, p) are fetched
    // into the other buffer with kSpecSlack columns to spare on both sides; a walk that ends elsewhere loads synchronously.
    unsigned char* const buf[2] = {tile, tile + kTraceWin * 32};
    int cur = 0;
    bool spec_ok = false;
    uint32_t ss = 0, ssb = 0, sn = 0;
    while (ti || tj) {
        if (!ti) {
            // row 0 (CDPMatrix::set_dir_all: every byte of row 0 is all-H)
            if (lane == 0) {
                uint32_t jj = tj;
                while (jj) {
                    tmp_path[n++] = (unsigned char)dir;
                    if (dir != 1) { jj = 0; break; }                 // cannot happen for a valid matrix
                    dir = (0x15 >> (2 * dir)) & 3;
                    --jj;
                }
            }
            dir = __shfl_sync(0xffffffffu, dir, 0);
            tj = 0;
            break;
        }
        const uint32_t stripe = (ti - 1) >> 5, l_top = (ti - 1) & 31, row_lo = stripe * 32 + 1;
        const uint32_t st_hi = tj + l_top;
        uint32_t wsb;
        if (spec_ok && ss == stripe && st_hi >= ssb && st_hi < ssb + sn) { cur ^= 1; wsb = ssb; }
        else {
            wsb = st_hi >= 63 ? st_hi - 63 : 0;
            const uint4* src = reinterpret_cast<const uint4*>(dirs + ((size_t)stripe * steps + wsb) * 32);
            const uint32_t n16 = (st_hi - wsb + 1) * 2;              // 16-byte units
            uint4* dst = reinterpret_cast<uint4*>(buf[cur]);
            for (uint32_t q = lane; q < n16; q += 32) dst[q] = __ldcg(src + q);
            __syncwarp();
        }
        // the speculative window of the stripe above: requested now, stored after the walk
        spec_ok = false;
        uint4 r[kTraceWin * 2 / 32];
        uint32_t s16 = 0;
        if (stripe > 0 && tj >= l_top + 1) {
            const uint32_t p = tj - (l_top + 1);
            uint32_t hi = p + 31 + kSpecSlack;
            if (hi > (uint32_t)steps - 1) hi = (uint32_t)steps - 1;
            const uint32_t lo = hi >= (uint32_t)kTraceWin - 1 ? hi - (kTraceWin - 1) : 0;
            ss = stripe - 1; ssb = lo; sn = hi - lo + 1; s16 = sn * 2; spec_ok = true;
            const uint4* src = reinterpret_cast<const uint4*>(dirs + ((size_t)ss * steps + ssb) * 32);
#pragma unroll
            for (uint32_t q = 0; q < kTraceWin * 2 / 32; ++q)
                if (lane + 32 * q < s16) r[q] = __ldcg(src + lane + 32 * q);
        }
        if (lane == 0) {
            // one move = one shared-memory byte load in the dependent chain: the index of the next cell depends only on the
            // current state, the state after that on the current cell's byte.  Per state: index step (D 65, H 32, V 33) and the
            // packed (row, column) decrement, both looked up by shifting constants.
            const uint32_t wbase = smem_addr(tile) + (uint32_t)cur * (kTraceWin * 32);
            int l = (int)l_top, j = (int)tj;
            int idx = (int)(st_hi - wsb) * 32 + l;
            unsigned b = lds_u8(wbase + (uint32_t)idx);
            uint32_t k = n;
            for (;;) {
                tmp_path[k++] = (unsigned char)dir;
                idx -= (int)((0x212041u >> ((unsigned)dir * 8)) & 0xffu);   // index step per state: 0x41 = 65, 0x20 = 32, 0x21 = 33
                l -= dir != 1; j -= dir != 2;
                const bool inside = (l | j | idx) >= 0;              // still in the stripe, in the matrix and in the window
                const unsigned nb = inside ? lds_u8(wbase + (uint32_t)idx) : 0;
                dir = (int)((b >> (2 * dir)) & 3);
                b = nb;
                if (!inside) break;
            }
            n = k;
            ti = l < 0 ? row_lo - 1 : row_lo + (uint32_t)l;
            tj = j < 0 ? 0 : (uint32_t)j;
        }
        if (spec_ok) {
            uint4* dst = reinterpret_cast<uint4*>(buf[cur ^ 1]);
#pragma unroll
            for (uint32_t q = 0; q < kTraceWin * 2 / 32; ++q)
                if (lane + 32 * q < s16) dst[lane + 32 * q] = r[q];
        }
        ti = __shfl_sync(0xffffffffu, ti, 0);
        tj = __shfl_sync(0xffffffffu, tj, 0);
        dir = __shfl_sync(0xffffffffu, dir, 0);
        __syncwarp();
    }
    n = __shfl_sync(0xffffffffu, n, 0);
    __syncwarp();
    unsigned char* path = P.path + J.path_off;
    for (uint32_t k = lane; k < n; k += 32) path[k] = tmp_path[n - 1 - k];
    if (P.h_path) {                                                 // zero-copy: 16 path bytes per store over PCIe
        unsigned char* hp = P.h_path + J.path_off;
        const bool aligned = ((J.path_off | (unsigned long long)(size_t)P.h_path) & 15) == 0;
        if (aligned) {
            for (uint32_t k = lane * 16; k < n; k += 32 * 16) {
                unsigned w[4] = {0, 0, 0, 0};
#pragma unroll
                for (uint32_t b = 0; b < 16; ++b)
                    if (k + b < n) w[b >> 2] |= (unsigned)tmp_path[n - 1 - (k + b)] << (8 * (b & 3));
                *reinterpret_cast<uint4*>(hp + k) = make_uint4(w[0], w[1], w[2], w[3]);     // (the tail may spill up to 15 bytes into this job's own slack)
            }
        } else {
            for (uint32_t k = lane; k < n; k += 32) hp[k] = tmp_path[n - 1 - k];
        }
    }
    if (lane == 0) {
        famsa_dp_result r;
        r.total_score = total;
        r.last[0] = last[0]; r.last[1] = last[1]; r.last[2] = last[2];
        r.path_offset = J.path_off; r.dirs_offset = J.dirs_off;
        r.path_len = n; r.rows_width = WR; r.cols_width = WC;
        r.swapped = (uint8_t)M.sw; r.variant = M.bad ? (uint8_t)0xFF : (uint8_t)M.var; r.pad[0] = r.pad[1] = 0;
        P.results[jid] = r;
        if (P.h_results) P.h_results[jid] = r;
        if (J.w_dst) *J.w_dst = M.bad ? kWidthBad : n;              // the merged profile's width, for merges queued behind this one
    }
}

__global__ void __launch_bounds__(kTraceWarps * 32) k_dp_trace(const DpParams P)
{
    __shared__ __align__(16) unsigned char sm_tile[kTraceWarps][2 * kTraceWin * 32];
    const uint32_t warp = threadIdx.x / 32;
    const uint32_t slot = blockIdx.x * kTraceWarps + warp;
    if (slot >= P.n_jobs) return;
    trace_body(P, P.job_base + slot, sm_tile[warp]);
}

// ------------------------------------------------------------------------------------------------
// k_merge_fused: a whole small merge in ONE block of four warps -- leaf materialisation, prep, the stripes, the
// traceback and the merged tables, phase after phase with block barriers instead of kernel boundaries.  For the
// chain-like parts of a guide tree, where a level is one small merge and five launches cost more than the work.
// ------------------------------------------------------------------------------------------------
constexpr int kFusedWarps = 8;
__device__ unsigned long long g_fused_phase_ns[8];          // development aid (FAMSA_FUSED_TIMING): per phase, the sum over launches of
__device__ unsigned long long g_fused_phase_max[2][8];      // the slowest block's time; [launch parity][phase] collects one launch
__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define FB_PHASE(k)                                                                     \
    do {                                                                                \
        if (F.timing && threadIdx.x == 0 && blockIdx.x == 0) {                          \
            const unsigned long long now__ = globaltimer_ns();                          \
            g_fused_phase_max[F.timing & 1][k] += now__ - t_phase;                      \
            t_phase = now__;                                                            \
        }                                                                               \
    } while (0)
__global__ void __launch_bounds__(kFusedWarps * 32, 1) k_merge_fused(const DpParams P, const FusedParams F)
{
    unsigned long long t_phase = F.timing ? globaltimer_ns() : 0;
    const unsigned long long t_begin = t_phase;
    if (F.timing && blockIdx.x == 0 && threadIdx.x == 0) {           // fold the previous launch (other parity) into the totals
        const int q = (F.timing & 1) ^ 1;
        for (int k = 0; k < 7; ++k) { g_fused_phase_ns[k] += g_fused_phase_max[q][k]; g_fused_phase_max[q][k] = 0; }
        // slot 7 of a launch = when its last block ended (absolute): the idle time before this launch
        if (g_fused_phase_max[q][7] && t_begin > g_fused_phase_max[q][7]) g_fused_phase_ns[7] += t_begin - g_fused_phase_max[q][7];
        g_fused_phase_max[q][7] = 0;
    }
    extern __shared__ __align__(16) unsigned char sm_dyn[];
    __shared__ __align__(16) unsigned char sm_tile[2 * kTraceWin * 32];
    __shared__ ConShared sm_con;
    const uint32_t warp = threadIdx.x / 32;
    uint32_t leaves_ready = 0xffffffffu;                               // job whose leaves are already materialised
    for (uint32_t lv = 0; lv < F.n_levels; ++lv) {
    for (uint32_t jid = F.level_start[lv] + blockIdx.x; jid < F.level_start[lv + 1]; jid += gridDim.x) {
    const FusedJob fj = F.jobs[jid];
    if (jid != leaves_ready)                                          // (else: materialised during the previous level's traceback)
        for (int side = 0; side < 2; ++side)
            if (fj.leaf[side].seq != 0xffffffffu) leaf_body(fj.leaf[side], F.codes, F.off, F.len, F.sm, P.go, P.ge, P.to, P.te);
    __syncthreads();
    FB_PHASE(0);
    prep_body(P, jid);
    __syncthreads();
    FB_PHASE(1);
    fill_body(P, jid, warp, kFusedWarps, reinterpret_cast<WarpShared*>(sm_dyn)[warp]);
    __syncthreads();
    FB_PHASE(2);
    // the traceback walks the direction bytes: bring the whole (skewed) matrix into the shared memory the fill no longer
    // needs when it fits, so that the walk never waits for a tile
    const unsigned char* all_dirs = nullptr;
    {
        const DpMeta M = P.meta[jid];
        const unsigned long long bytes = (unsigned long long)((M.WR + 31) / 32) * ((unsigned long long)M.WC + 32) * 32;
        if (M.bad != 2 && M.WR && bytes <= kFusedWarps * sizeof(WarpShared)) {
            const uint4* src = reinterpret_cast<const uint4*>(P.sdirs + P.jobs[jid].t_off);
            uint4* dst = reinterpret_cast<uint4*>(sm_dyn);
            for (uint32_t q = threadIdx.x; q < bytes / 16; q += blockDim.x) dst[q] = __ldcg(src + q);
            all_dirs = sm_dyn;
        }
    }
    __syncthreads();
    FB_PHASE(3);
    // the seven warps the traceback does not need materialise the leaves of this block's first merge of the next level
    uint32_t nj = 0xffffffffu;
    if (lv + 1 < F.n_levels && jid + gridDim.x >= F.level_start[lv + 1] && F.level_start[lv + 1] + blockIdx.x < F.level_start[lv + 2])
        nj = F.level_start[lv + 1] + blockIdx.x;
    if (warp == 0) trace_body(P, jid, sm_tile, all_dirs);
    else if (nj != 0xffffffffu) {
        const FusedJob nf = F.jobs[nj];
        for (int side = 0; side < 2; ++side)
            if (nf.leaf[side].seq != 0xffffffffu) leaf_body(nf.leaf[side], F.codes, F.off, F.len, F.sm, P.go, P.ge, P.to, P.te, 1);
    }
    leaves_ready = nj;
    __syncthreads();
    FB_PHASE(4);
    ConJob J;
    if (con_resolve(fj.con, P.meta[jid], P.results[jid], P.path, J))
        for (uint32_t k0 = 0; k0 <= J.W; k0 += kConTile) construct_tile(J, k0, sm_con, P.go, P.ge, P.to, P.te);
    FB_PHASE(5);
    __syncthreads();                                                 // the next job of this block reuses the shared memory
    }
    if (lv + 1 < F.n_levels) {
        // grid barrier: the next level reads what this one wrote (merged tables, widths)
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            atomicAdd(F.block_counter + 1, 1u);
            const unsigned target = (lv + 1) * gridDim.x;
            unsigned seen;
            do {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(F.block_counter + 1) : "memory");
                if (seen < target) __nanosleep(40);
            } while (seen < target);
        }
        __syncthreads();
        FB_PHASE(7 - 1);                                             // (slot 6: time spent at the barriers)
    }
    }
    if (!F.h_done && F.n_levels > 1) {
        __syncthreads();
        if (threadIdx.x == 0 && atomicAdd(F.block_counter, 1u) == gridDim.x - 1) { F.block_counter[0] = 0; F.block_counter[1] = 0; }
    }
    if (F.h_done) {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence_system();                                  // this block's records and paths are in host memory
            if (atomicAdd(F.block_counter, 1u) == gridDim.x - 1) {
                F.block_counter[0] = 0;
                F.block_counter[1] = 0;
                __threadfence_system();
                *F.h_done = F.done_seq;
            }
        }
    }
    if (F.timing && threadIdx.x == 0) atomicMax(&g_fused_phase_max[F.timing & 1][7], globaltimer_ns());
}
#undef FB_PHASE

// development aid (not part of the ABI): accumulated nanoseconds of block 0 per phase of k_merge_fused since the last call
// -- leaves, prep, fill, load of the direction bytes, traceback, merged tables; active when FAMSA_FUSED_TIMING is set
extern "C" int famsa_debug_fused_phases(double out_ns[8])
{
    unsigned long long h[8], m[2][8];
    if (cudaMemcpyFromSymbol(h, g_fused_phase_ns, sizeof(h)) != cudaSuccess) return 1;
    if (cudaMemcpyFromSymbol(m, g_fused_phase_max, sizeof(m)) != cudaSuccess) return 1;
    for (int k = 0; k < 7; ++k) out_ns[k] = (double)(h[k] + m[0][k] + m[1][k]);
    out_ns[7] = (double)h[7];
    memset(h, 0, sizeof(h)); memset(m, 0, sizeof(m));
    if (cudaMemcpyToSymbol(g_fused_phase_max, m, sizeof(m)) != cudaSuccess) return 1;
    return cudaMemcpyToSymbol(g_fused_phase_ns, h, sizeof(h)) == cudaSuccess ? 0 : 1;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------

using FillKernel = void (*)(DpParams);

// largest cluster size in {2, 4, 8, 16} that `kernel` can be launched with on this device (1: none)
static uint32_t max_cluster(FillKernel kernel, int block, size_t smem)
{
    uint32_t v = 1;
    for (uint32_t cl : {2u, 4u, 8u, 16u}) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(cl);
        cfg.blockDim = dim3(block);
        cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = cl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess || n == 0) { cudaGetLastError(); break; }
        v = cl;
    }
    return v;
}

// Kernel attributes of every fill shape and of k_merge_fused, and the cluster caps: once per context, on the first DP
// call (an LCS-only caller never loads the DP kernels).
static int configure_dp(famsa_ctx* ctx)
{
    DpState& S = ctx->dp;
    if (S.configured) return FAMSA_OK;
    const auto smem = [](auto kernel, size_t bytes) {
        return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    };
    const auto any_cluster = [](auto kernel) {
        return cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    };
    FB_CUDA(smem(k_dp_fill<1, false>, kDpWarps * sizeof(WarpShared)));
    FB_CUDA(smem(k_dp_fill<2, false>, 2 * sizeof(WarpShared)));
    FB_CUDA(smem(k_dp_fill<4, false>, 4 * sizeof(WarpShared)));
    FB_CUDA(smem(k_dp_fill<kDpTeamWarps, false>, kDpTeamWarps * sizeof(WarpShared)));
    FB_CUDA(smem(k_dp_fill<4, true>, 4 * sizeof(WarpShared)));
    FB_CUDA(any_cluster(k_dp_fill<4, true>));
    FB_CUDA(smem(k_dp_fill<kDpTeamWarps, true>, kDpTeamWarps * sizeof(WarpShared)));
    FB_CUDA(any_cluster(k_dp_fill<kDpTeamWarps, true>));
    FB_CUDA(smem(k_dp_fill_duo, kDuoSmem));
    FB_CUDA(any_cluster(k_dp_fill_duo));
    FB_CUDA(smem(k_dp_fill_compact<2>, 2 * kCompactStride));
    FB_CUDA(smem(k_dp_fill_compact<4>, 4 * kCompactStride));
    FB_CUDA(smem(k_dp_fill_compact<6>, 6 * kCompactStride));
    FB_CUDA(smem(k_merge_fused, kFusedWarps * sizeof(WarpShared)));
    S.cluster4_cap = max_cluster(k_dp_fill<4, true>, 4 * 32, 4 * sizeof(WarpShared));
    S.duo_cap = max_cluster(k_dp_fill_duo, 256, kDuoSmem);
    S.configured = true;
    return FAMSA_OK;
}

// Every fill launch: `grid` blocks, in clusters of `cl` blocks when cl > 1.
static int launch_fill(famsa_ctx* ctx, FillKernel kernel, const DpParams& Q, uint32_t grid, uint32_t block,
                       size_t smem, uint32_t cl, cudaStream_t st)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = cl > 1 ? 1 : 0;
    FB_CUDA(cudaLaunchKernelEx(&cfg, kernel, Q));
    ctx->launches++;
    return FAMSA_OK;
}

// Development knobs of the fill launch policy.  Read on every dp_run_device call: tests change them between calls.
struct DpKnobs {
    unsigned long long max_cells = 1ull << 32;     // FAMSA_DP_MAX_CELLS: matrix cells per sub-batch
    uint32_t team_min = kDpTeamMinWidth;           // FAMSA_DP_TEAM_MIN
    int team_warps = 0;                            // FAMSA_DP_TEAM_WARPS (0: by the number of merges)
    uint32_t cluster_min = kDpClusterMinWidth;     // FAMSA_DP_CLUSTER_MIN
    uint32_t max_cluster = 0xffffffffu;            // FAMSA_DP_MAX_CLUSTER: limits the probed cap
    int latency_mode = -1;                         // FAMSA_DP_LATENCY_MODE (-1: by the batch's demand)
    bool duo = true;                               // FAMSA_DP_DUO=0: one warp per stripe instead of producer / consumer pairs
    int compact = 1;                               // FAMSA_DP_COMPACT: 0 never, 1 from two merges per SM on, 2 always
};

static DpKnobs read_knobs()
{
    DpKnobs K;
    if (const char* e = getenv("FAMSA_DP_MAX_CELLS")) K.max_cells = strtoull(e, nullptr, 10);
    if (const char* e = getenv("FAMSA_DP_TEAM_MIN")) K.team_min = (uint32_t)atoi(e);
    if (const char* e = getenv("FAMSA_DP_TEAM_WARPS")) K.team_warps = atoi(e);
    if (const char* e = getenv("FAMSA_DP_CLUSTER_MIN")) K.cluster_min = (uint32_t)atoi(e);
    if (const char* e = getenv("FAMSA_DP_MAX_CLUSTER")) K.max_cluster = (uint32_t)atoi(e);
    if (const char* e = getenv("FAMSA_DP_LATENCY_MODE")) K.latency_mode = atoi(e) != 0;
    if (const char* e = getenv("FAMSA_DP_DUO")) K.duo = atoi(e) != 0;
    if (const char* e = getenv("FAMSA_DP_COMPACT")) K.compact = atoi(e);
    return K;
}

bool dp_debug()
{
    static const bool debug = getenv("FAMSA_DP_DEBUG") != nullptr;
    return debug;
}

// Job k as the kernels see it, without its buffer offsets.  jobs[k].p1/p2 hold DEVICE pointers; the widths are the
// layout widths (upper bounds when ext->w*_src is set).
static int make_job(const famsa_dp_job& j, const DpJobExt* ext, uint32_t k, DpJobDev& d)
{
    if (j.p1.width == 0 || j.p2.width == 0 || j.p1.card == 0 || j.p2.card == 0) {
        set_error("dp job " + std::to_string(k) + ": empty profile");
        return FAMSA_E_INVALID;
    }
    if (((unsigned long long)j.p1.width + 1) * (j.p2.width + 1) > 0xffffffffull) {
        set_error("dp job " + std::to_string(k) + ": more than 2^32 matrix cells");
        return FAMSA_E_INVALID;
    }
    d.s1 = reinterpret_cast<const long long*>(j.p1.scores); d.c1 = j.p1.counters;
    d.s2 = reinterpret_cast<const long long*>(j.p2.scores); d.c2 = j.p2.counters;
    d.w1 = j.p1.width; d.card1 = j.p1.card; d.w2 = j.p2.width; d.card2 = j.p2.card;
    d.w1_src = ext ? ext->w1_src : nullptr; d.w2_src = ext ? ext->w2_src : nullptr; d.w_dst = ext ? ext->w_dst : nullptr;
    return FAMSA_OK;
}

// what every launch of one batch shares
static DpParams batch_params(const DpJobDev* jobs, DpMeta* meta, const int64_t gaps[4], uint8_t* sdirs, uint8_t* path,
                             uint8_t* scratch, famsa_dp_result* results)
{
    DpParams P{};
    P.jobs = jobs;
    P.meta = meta;
    P.go = gaps[0]; P.ge = gaps[1]; P.to = gaps[2]; P.te = gaps[3];
    P.sdirs = sdirs;
    P.path = path;
    P.scratch = scratch;
    P.results = results;
    return P;
}

unsigned long long dp_scratch_bytes(uint32_t w1, uint32_t w2) { return Scratch(w1, w2).total; }

// ---- the fused path (k_merge_fused): planning and launch are separate so that the caller can place the descriptors in
// mapped host memory and every device buffer in its own ring (no copy, no allocator call per batch)
int dp_fused_plan(const famsa_dp_job* jobs, const DpJobExt* ext, uint32_t n, bool align16, DpJobDev* out, DpFusedPlan* plan)
{
    unsigned long long path_off = 0, scratch_off = 0, t_off = 0, cells = 0;
    for (uint32_t k = 0; k < n; ++k) {
        DpJobDev& d = out[k];
        FB_TRY(make_job(jobs[k], ext ? ext + k : nullptr, k, d));
        d.path_off = path_off; d.dirs_off = 0;
        d.scratch_off = scratch_off; d.t_off = t_off;
        path_off += align16 ? align_up((unsigned long long)d.w1 + d.w2, 16) : (unsigned long long)d.w1 + d.w2;   // 16-byte slots: the traceback
                                                                       // then stores paths to the host in uint4 units
        scratch_off += Scratch(d.w1, d.w2).total;
        t_off += skew_elems(d.w1, d.w2);
        cells += (unsigned long long)d.w1 * d.w2;
    }
    plan->scratch_bytes = scratch_off; plan->skew_bytes = t_off; plan->path_bytes = path_off; plan->cells = cells;
    return FAMSA_OK;
}

int dp_fused_launch(famsa_ctx* ctx, const DpJobDev* jobs, uint32_t n, const int64_t gaps[4], famsa_dp_result* d_results, uint8_t* d_path,
                    DpMeta* d_meta, uint8_t* d_scratch, uint8_t* d_skew, famsa_dp_result* h_results, uint8_t* h_path,
                    const FusedParams& fused, uint32_t grid, uint64_t cells, bool record_events, cudaStream_t st)
{
    FB_TRY(configure_dp(ctx));
    ctx->dp.last_cells = cells;
    DpParams P = batch_params(jobs, d_meta, gaps, d_skew, d_path, d_scratch, d_results);
    P.n_jobs = n;
    P.h_results = h_results;
    P.h_path = h_path;
    if (record_events) { FB_CUDA(cudaEventRecord(ctx->ev[0], st)); FB_CUDA(cudaEventRecord(ctx->ev[1], st)); }
    k_merge_fused<<<grid, kFusedWarps * 32, kFusedWarps * sizeof(WarpShared), st>>>(P, fused);
    FB_CUDA(cudaGetLastError());
    ctx->launches++;
    if (record_events) { FB_CUDA(cudaEventRecord(ctx->ev[2], st)); FB_CUDA(cudaEventRecord(ctx->ev[3], st)); }
    return FAMSA_OK;
}

// Runs a batch of merges on the stream: prep, fill, traceback (and the un-skewed direction matrices when d_dirs is set),
// in sub-batches of consecutive jobs above ~4 Gi cells.
// jobs[k].p1/p2 hold DEVICE pointers here; widths are the layout widths (upper bounds when ext[k].w*_src is set).
int dp_run_device(famsa_ctx* ctx, const famsa_dp_job* jobs, const DpJobExt* ext, uint32_t n, const int64_t gaps[4],
                  famsa_dp_result* d_results, uint8_t* d_path, uint8_t* d_dirs, DpMeta** d_meta_out, void** d_blob_out,
                  cudaStream_t st)
{
    DpState& S = ctx->dp;
    std::vector<DpJobDev> dev(n);
    unsigned long long path_off = 0, dirs_off = 0, cells = 0;
    for (uint32_t k = 0; k < n; ++k) {
        DpJobDev& d = dev[k];
        FB_TRY(make_job(jobs[k], ext ? ext + k : nullptr, k, d));
        d.path_off = path_off; d.dirs_off = dirs_off;           // caller-visible layout: global prefix sums
        path_off += (unsigned long long)d.w1 + d.w2;
        dirs_off += ((unsigned long long)d.w1 + 1) * (d.w2 + 1);
        cells += (unsigned long long)d.w1 * d.w2;
    }
    S.last_cells = cells;
    const DpKnobs K = read_knobs();
    FB_TRY(configure_dp(ctx));

    // Sub-batches of consecutive jobs bound the device scratch (direction bytes are 1 byte per cell): ~4 Gi cells each.
    // Plan them first: one stream-ordered allocation serves all of them.
    struct Sub { uint32_t j0, j1; unsigned long long scratch, skew; std::vector<unsigned long long> tblock; };
    std::vector<Sub> subs;
    unsigned long long max_scratch = 64, max_skew = 64;
    uint32_t max_m = 1;
    for (uint32_t j0 = 0; j0 < n;) {
        Sub sb;
        sb.j0 = j0;
        uint32_t j1 = j0;
        unsigned long long mat_sum = 0, scratch_off = 0, t_off = 0;
        sb.tblock.assign(1, 0);
        while (j1 < n) {
            const unsigned long long mat = ((unsigned long long)dev[j1].w1 + 1) * (dev[j1].w2 + 1);
            if (j1 > j0 && mat_sum + mat > K.max_cells) break;
            dev[j1].scratch_off = scratch_off;
            dev[j1].t_off = t_off;                              // skewed directions are per sub-batch
            scratch_off += Scratch(dev[j1].w1, dev[j1].w2).total;
            t_off += skew_elems(dev[j1].w1, dev[j1].w2);
            mat_sum += mat;
            sb.tblock.push_back(sb.tblock.back() + (mat + kTThreads * kTCellsPerThread - 1) / (kTThreads * kTCellsPerThread));
            ++j1;
        }
        sb.j1 = j1; sb.scratch = scratch_off; sb.skew = t_off;
        if (sb.tblock.back() > 0x7fffffffull) { set_error("dp sub-batch too large for one launch"); return FAMSA_E_INVALID; }
        max_scratch = std::max(max_scratch, scratch_off);
        max_skew = std::max(max_skew, t_off);
        max_m = std::max(max_m, j1 - j0);
        subs.push_back(std::move(sb));
        j0 = j1;
    }
    // blob: [jobs n][meta n][order max_m][tblock max_m+1][scratch][skewed dirs]
    const unsigned long long o_jobs = 0;
    const unsigned long long o_meta = align_up(o_jobs + sizeof(DpJobDev) * (unsigned long long)std::max(n, 1u), 256);
    const unsigned long long o_order = align_up(o_meta + sizeof(DpMeta) * (unsigned long long)std::max(n, 1u), 256);
    const unsigned long long o_tblock = align_up(o_order + sizeof(uint32_t) * (unsigned long long)max_m, 256);
    const unsigned long long o_scratch = align_up(o_tblock + sizeof(unsigned long long) * ((unsigned long long)max_m + 1), 256);
    const unsigned long long o_skew = align_up(o_scratch + max_scratch, 256);
    const unsigned long long blob_bytes = o_skew + max_skew;
    unsigned char* blob = nullptr;
    {
        cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&blob), blob_bytes, st);
        if (e != cudaSuccess) {
            set_error("cudaMallocAsync(" + std::to_string(blob_bytes) + ") for the DP scratch failed: " + cudaGetErrorString(e));
            return FAMSA_E_NOMEM;
        }
    }
    DpJobDev* d_jobs = reinterpret_cast<DpJobDev*>(blob + o_jobs);
    DpMeta* d_meta = reinterpret_cast<DpMeta*>(blob + o_meta);
    FB_CUDA(cudaEventRecord(ctx->ev[0], st));
    FB_CUDA(cudaEventRecord(ctx->ev[1], st));
    if (n) FB_CUDA(cudaMemcpyAsync(d_jobs, dev.data(), sizeof(DpJobDev) * n, cudaMemcpyHostToDevice, st));
    DpParams P = batch_params(d_jobs, d_meta, gaps, blob + o_skew, d_path, blob + o_scratch, d_results);
    P.order = reinterpret_cast<const uint32_t*>(blob + o_order);
    P.dirs = d_dirs;
    P.tblock = reinterpret_cast<const unsigned long long*>(blob + o_tblock);
    const uint32_t sms = (uint32_t)ctx->sm_count;
    std::vector<int> cls(n);                                     // fill class of each merge: larger = launched first
    for (const Sub& sb : subs) {
        const uint32_t j0 = sb.j0, j1 = sb.j1, m = j1 - j0;
        // rows of the DP matrix as far as the host can tell (the orientation of ProfProf merges is decided on the device)
        auto stripes_of = [&](uint32_t a) {
            const DpJobDev& d = dev[a];
            const uint32_t rows = d.card1 == 1 ? d.w1 : (d.card2 == 1 ? d.w2 : std::min(d.w1, d.w2));
            return (rows + 31) / 32;
        };
        // Two regimes.  A batch large enough to fill the device with one warp per stripe-pipeline is THROUGHPUT-bound:
        // wide merges get a block (2, 4 or 8 warps by how many there are), the very widest a cluster of 8 x 8 warps, the
        // rest run one warp per merge.  A small batch (the chain-like parts and the top of a guide tree, where a level is
        // one or a few merges) is LATENCY-bound: every merge with more than one stripe gets a cluster of 4-warp blocks,
        // one stripe per SM sub-partition, as many blocks as its stripes can use (up to 16).
        const uint32_t cl_cap = std::max(1u, std::min(S.cluster4_cap, K.max_cluster));
        // latency mode while the batch's stripes fit one per SM sub-partition
        unsigned long long demand = 0;
        uint32_t n_teamable = 0;
        for (uint32_t a = j0; a < j1; ++a) {
            demand += std::min(stripes_of(a), 4u * cl_cap);
            n_teamable += std::min(dev[a].w1, dev[a].w2) > K.team_min;
        }
        const bool small_batch = K.latency_mode >= 0 ? K.latency_mode != 0 : demand <= 4ull * sms;
        // throughput mode with only a handful of block-sized merges: give every merge with more than 8 stripes a cluster
        uint32_t cl_min = K.cluster_min;
        if (n_teamable * kDpCluster <= 2u * sms) cl_min = std::min(K.cluster_min, std::max(K.team_min, 256u));
        const uint32_t duo_cap = K.duo ? S.duo_cap : 1;
        for (uint32_t a = j0; a < j1; ++a) {
            const uint32_t w = std::min(dev[a].w1, dev[a].w2);
            if (small_batch) {
                const uint32_t stripes = stripes_of(a);
                uint32_t cl = 1;                                 // blocks (of 4 warps) for merge a
                while (cl < (stripes + 3) / 4 && cl < cl_cap) cl *= 2;
                // ProfProf merges wide enough for a cluster: producer / consumer pairs (k_dp_fill_duo)
                if (stripes < 2) cls[a] = 0;
                else if (K.duo && cl >= 2 && dev[a].card1 > 1 && dev[a].card2 > 1) cls[a] = 100 + (int)std::min(cl, duo_cap);
                else cls[a] = 10 + (int)cl;
            } else cls[a] = w > cl_min ? 2 : (w > K.team_min ? 1 : 0);
        }
        std::vector<uint32_t> order(m);
        std::iota(order.begin(), order.end(), j0);
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
            if (cls[a] != cls[b]) return cls[a] > cls[b];
            return (unsigned long long)dev[a].w1 * dev[a].w2 > (unsigned long long)dev[b].w1 * dev[b].w2;
        });
        // one launch per run [q0, q1) of equal class in `order`
        std::vector<std::pair<uint32_t, uint32_t>> runs;
        for (uint32_t q0 = 0, q1 = 0; q0 < m; q0 = q1) {
            while (q1 < m && cls[order[q1]] == cls[order[q0]]) ++q1;
            runs.emplace_back(q0, q1);
        }

        // Throughput mode: the first wave of blocks lands on the SMs in launch order, so deal the merges (sorted by size) in
        // snake rows of one block per SM -- the SM that got the largest merge of a row gets the smallest of the next one.
        if (!small_batch)
            for (const auto& [q0, q1] : runs)
                if (cls[order[q0]] == 1)
                    for (uint32_t r = q0 + sms, row = 1; r < q1; r += sms, ++row)
                        if (row & 1) std::reverse(order.begin() + r, order.begin() + std::min(q1, r + sms));

        // one packed upload: order + tblock
        std::vector<unsigned char> pack(o_scratch - o_order);
        memcpy(pack.data(), order.data(), sizeof(uint32_t) * m);
        memcpy(pack.data() + (o_tblock - o_order), sb.tblock.data(), sizeof(unsigned long long) * (m + 1));
        FB_CUDA(cudaMemcpyAsync(blob + o_order, pack.data(), (o_tblock - o_order) + sizeof(unsigned long long) * (m + 1), cudaMemcpyHostToDevice, st));
        P.n_jobs = m;
        P.job_base = j0;
        k_dp_prep<<<m, kPrepThreads, 0, st>>>(P);
        FB_CUDA(cudaGetLastError());
        ctx->launches += 1;
        // different classes run side by side (fork after prep, join before the traceback) so that a level pays for its
        // slowest merge once, not once per launch shape
        if (runs.size() > 1) FB_CUDA(cudaEventRecord(ctx->ev_fork, st));
        uint32_t aux_used = 0;
        for (size_t r = 0; r < runs.size(); ++r) {
            const uint32_t q0 = runs[r].first, q1 = runs[r].second;
            const int c = cls[order[q0]];
            if (dp_debug()) fprintf(stderr, "[dp] batch of %u: class %d x %u (first %u x %u, %u stripes), demand %llu, cl_cap %u, latency_mode %d\n", m, c, q1 - q0,
                                    dev[order[q0]].w1, dev[order[q0]].w2, stripes_of(order[q0]), demand, cl_cap, (int)small_batch);
            DpParams Q = P;
            Q.order = P.order + q0;
            Q.n_jobs = q1 - q0;
            // class 0 (first in launch order is the heaviest) stays on the main stream, the others go to the aux streams
            cudaStream_t fst = st;
            if (r > 0) {
                const uint32_t a = (uint32_t)(r - 1) % 4;
                fst = ctx->aux_stream[a];
                if (!(aux_used >> a & 1)) { FB_CUDA(cudaStreamWaitEvent(fst, ctx->ev_fork, 0)); aux_used |= 1u << a; }
            }
            if (c == 0) {
                FB_TRY(launch_fill(ctx, k_dp_fill<1, false>, Q, (Q.n_jobs + kDpWarps - 1) / kDpWarps, kDpWarps * 32, kDpWarps * sizeof(WarpShared), 1, fst));
            } else if (c >= 100) {
                const uint32_t cl = (uint32_t)c - 100;
                FB_TRY(launch_fill(ctx, k_dp_fill_duo, Q, Q.n_jobs * cl, 256, kDuoSmem, cl, fst));
            } else if (c >= 10) {
                const uint32_t cl = (uint32_t)c - 10;
                FB_TRY(launch_fill(ctx, cl == 1 ? k_dp_fill<4, false> : k_dp_fill<4, true>, Q, Q.n_jobs * cl, 4 * 32, 4 * sizeof(WarpShared), cl, fst));
            } else if (c == 2) {
                FB_TRY(launch_fill(ctx, k_dp_fill<kDpTeamWarps, true>, Q, Q.n_jobs * kDpCluster, kDpTeamWarps * 32, kDpTeamWarps * sizeof(WarpShared), kDpCluster, fst));
            } else {
                // Team size by how many merges there are: every SM holds 8 fill warps (shared memory), so a level with many
                // block-class merges runs them with smaller teams -- 4 warps from 2 merges per SM on, 2 from 4 -- which lose
                // less to the ramp-up / ramp-down of the stripe pipeline.
                // From two merges per SM on, the compact kernel (12 warps per SM): 6, 4 or 2 warps per merge.
                int nw = kDpTeamWarps;
                bool compact = K.compact == 2 || (K.compact == 1 && Q.n_jobs >= 2u * sms);
                if (compact) nw = Q.n_jobs >= 6u * sms ? 2 : (Q.n_jobs >= 3u * sms ? 4 : 6);
                else if (Q.n_jobs >= 4u * sms) nw = 2;
                else if (Q.n_jobs >= 2u * sms) nw = 4;
                if (K.team_warps) { nw = K.team_warps; compact = compact && (nw == 2 || nw == 4 || nw == 6); }
                if (compact) {
                    const int cw = nw == 2 || nw == 4 ? nw : 6;
                    FB_TRY(launch_fill(ctx, cw == 2 ? k_dp_fill_compact<2> : (cw == 4 ? k_dp_fill_compact<4> : k_dp_fill_compact<6>), Q, Q.n_jobs, cw * 32,
                                       cw * kCompactStride, 1, fst));
                    if (cw == 6) nw = 4;
                    Q.wide_only = 1;                                 // merges whose T needs 8 bytes: the launch below
                }
                const int fw = nw == 2 || nw == 4 ? nw : kDpTeamWarps;
                FB_TRY(launch_fill(ctx, fw == 2 ? k_dp_fill<2, false> : (fw == 4 ? k_dp_fill<4, false> : k_dp_fill<kDpTeamWarps, false>), Q, Q.n_jobs, fw * 32,
                                   fw * sizeof(WarpShared), 1, fst));
            }
        }
        for (uint32_t a = 0; a < 4; ++a)
            if (aux_used >> a & 1) {
                FB_CUDA(cudaEventRecord(ctx->ev_join[a], ctx->aux_stream[a]));
                FB_CUDA(cudaStreamWaitEvent(st, ctx->ev_join[a], 0));
            }
        k_dp_trace<<<(m + kTraceWarps - 1) / kTraceWarps, kTraceWarps * 32, 0, st>>>(P);
        FB_CUDA(cudaGetLastError());
        ctx->launches++;
        if (d_dirs) {                                            // caller wants CDPMatrix bytes: un-skew
            k_dp_unskew<<<(unsigned)sb.tblock[m], kTThreads, 0, st>>>(P);
            FB_CUDA(cudaGetLastError());
            ctx->launches++;
        }
    }
    FB_CUDA(cudaEventRecord(ctx->ev[2], st));
    FB_CUDA(cudaEventRecord(ctx->ev[3], st));
    if (d_meta_out) { *d_meta_out = d_meta; *d_blob_out = blob; }    // the caller still reads meta / paths: it frees the blob
    else FB_CUDA(cudaFreeAsync(blob, st));
    return FAMSA_OK;
}

// variant 0xFF: k_dp_prep found a negative count in the tables (see ulo32) -- fail loudly rather than return a
// result that could differ from the reference's signed arithmetic
int dp_check_results(const famsa_dp_result* results, uint32_t n)
{
    for (uint32_t k = 0; k < n; ++k)
        if (results[k].variant == 0xFF) {
            set_error("dp job " + std::to_string(k) + ": a profile holds negative residue / gap counts");
            return FAMSA_E_INVALID;
        }
    return FAMSA_OK;
}

int dp_run_host(famsa_ctx* ctx, const famsa_dp_job* jobs, uint32_t n, const int64_t gaps[4], famsa_dp_result* results,
                uint8_t* path_buf, uint8_t* dirs_buf)
{
    DpState& S = ctx->dp;
    cudaStream_t st = ctx->stream;
    // pack every table into one staging buffer -> one H2D
    unsigned long long bytes = 0, path_total = 0, dirs_total = 0;
    for (uint32_t k = 0; k < n; ++k) {
        const famsa_dp_job& j = jobs[k];
        if (!j.p1.scores || !j.p1.counters || !j.p2.scores || !j.p2.counters) {
            set_error("dp job " + std::to_string(k) + ": NULL table");
            return FAMSA_E_INVALID;
        }
        bytes += ((unsigned long long)j.p1.width + 1 + j.p2.width + 1) * 32 * (8 + 4);
        path_total += (unsigned long long)j.p1.width + j.p2.width;
        dirs_total += ((unsigned long long)j.p1.width + 1) * (j.p2.width + 1);
    }
    // pinned staging buffer; tables are packed and shipped in ~8 MB slices so that packing slice k+1 overlaps the
    // H2D of slice k
    if (bytes > S.h_pinned_cap) {
        if (S.h_pinned) cudaFreeHost(S.h_pinned);
        S.h_pinned = nullptr;
        S.h_pinned_cap = 0;
        FB_CUDA(cudaHostAlloc(&S.h_pinned, bytes + bytes / 4 + 4096, cudaHostAllocDefault));
        S.h_pinned_cap = bytes + bytes / 4 + 4096;
    }
    FB_TRY(S.d_tables.reserve(std::max<unsigned long long>(bytes, 64)));
    std::vector<famsa_dp_job> dj(jobs, jobs + n);
    unsigned long long at = 0;
    uint8_t* hb = static_cast<uint8_t*>(S.h_pinned);
    uint8_t* db = S.d_tables.as<uint8_t>();
    // device addresses first (cheap), then the copies: the staging buffer is filled by a few host threads, each
    // shipping its own contiguous slice as soon as it is packed
    std::vector<unsigned long long> job_at(n + 1, 0);
    for (uint32_t k = 0; k < n; ++k) {      // every table size is a multiple of 128 bytes, so alignment is kept
        famsa_dp_job& j = dj[k];
        const size_t s1 = ((size_t)jobs[k].p1.width + 1) * 32 * 8, s2 = ((size_t)jobs[k].p2.width + 1) * 32 * 8;
        j.p1.scores = reinterpret_cast<const int64_t*>(db + at);
        j.p2.scores = reinterpret_cast<const int64_t*>(db + at + s1);
        j.p1.counters = reinterpret_cast<const int32_t*>(db + at + s1 + s2);
        j.p2.counters = reinterpret_cast<const int32_t*>(db + at + s1 + s2 + s1 / 2);
        at += (s1 + s2) * 3 / 2;
        job_at[k + 1] = at;
    }
    {
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const unsigned n_thr = bytes > (16u << 20) ? std::min(8u, hw) : 1;
        std::vector<std::thread> workers;
        std::vector<cudaError_t> errs(n_thr, cudaSuccess);
        for (unsigned t = 0; t < n_thr; ++t)
            workers.emplace_back([&, t] {
                cudaSetDevice(ctx->device);
                const uint32_t k0 = (uint32_t)((unsigned long long)n * t / n_thr), k1 = (uint32_t)((unsigned long long)n * (t + 1) / n_thr);
                unsigned long long sent = job_at[k0];
                for (uint32_t k = k0; k < k1; ++k) {
                    const size_t s1 = ((size_t)jobs[k].p1.width + 1) * 32 * 8, s2 = ((size_t)jobs[k].p2.width + 1) * 32 * 8;
                    uint8_t* h = hb + job_at[k];
                    memcpy(h, jobs[k].p1.scores, s1);
                    memcpy(h + s1, jobs[k].p2.scores, s2);
                    memcpy(h + s1 + s2, jobs[k].p1.counters, s1 / 2);
                    memcpy(h + s1 + s2 + s1 / 2, jobs[k].p2.counters, s2 / 2);
                    if (job_at[k + 1] - sent >= (8u << 20) || k + 1 == k1) {
                        cudaError_t e = cudaMemcpyAsync(db + sent, hb + sent, job_at[k + 1] - sent, cudaMemcpyHostToDevice, st);
                        if (e != cudaSuccess) errs[t] = e;
                        sent = job_at[k + 1];
                    }
                }
            });
        for (auto& w : workers) w.join();
        for (cudaError_t e : errs) FB_CUDA(e);
    }
    FB_TRY(S.d_results.reserve(sizeof(famsa_dp_result) * std::max(1u, n)));
    FB_TRY(S.d_path.reserve(std::max<unsigned long long>(path_total, 64)));
    uint8_t* d_dirs = nullptr;
    if (dirs_buf) {
        FB_TRY(S.d_dirs_out.reserve(std::max<unsigned long long>(dirs_total, 64)));   // row-major copy for the caller
        d_dirs = S.d_dirs_out.as<uint8_t>();
    }
    FB_TRY(dp_run_device(ctx, dj.data(), nullptr, n, gaps, S.d_results.as<famsa_dp_result>(), S.d_path.as<uint8_t>(), d_dirs, nullptr, nullptr, st));
    if (n) FB_CUDA(cudaMemcpyAsync(results, S.d_results.p, sizeof(famsa_dp_result) * n, cudaMemcpyDeviceToHost, st));
    if (path_total) FB_CUDA(cudaMemcpyAsync(path_buf, S.d_path.p, path_total, cudaMemcpyDeviceToHost, st));
    if (dirs_buf && dirs_total) FB_CUDA(cudaMemcpyAsync(dirs_buf, d_dirs, dirs_total, cudaMemcpyDeviceToHost, st));
    FB_CUDA(cudaStreamSynchronize(st));
    return dp_check_results(results, n);
}

} // namespace fb
