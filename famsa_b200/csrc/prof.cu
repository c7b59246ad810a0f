// Resident profiles: leaf materialisation and ConstructProfile's merge part on the device (SURVEY 8f-2).
//
// What the reference does per merge (src/core/profile.cpp:784-1002) is one sequential walk over the traceback
// path that (a) adds the children's columns into the merged profile (InsertColumn :1107-1111), (b) for an H / V
// step inserts a column of gaps into the row / column child (InsertGaps :1005-1050) whose open / ext / term_open /
// term_ext split comes from SolveGapsProblemWhenStarting / WhenContinuing (:1146-1220 / :1114-1143), and (c) turns
// "open" into "ext" in the child column right of a freshly started gap run (the n_gap_to_transfer bookkeeping).
//
// None of that carries state further than one run of equal directions, so here every merged column is built
// independently (one warp per column, lane = one of the 32 rows of CProfileValues):
//   * i_k / j_k, the child columns consumed up to merged column k, are prefix counts over the path;
//   * a gap column's split depends only on whether it starts its run (path[k-2] != path[k-1]) and on the child's
//     counters at src and src+1.  For a continued run the reference's "values at left" recurrence collapses after
//     one step to  term_ext = TO[src+1] + TO[src] + TE[src],  ext = card - term_ext,  open = term_open = 0
//     (interior) or term_ext = card (src == 0 or src == width);
//   * the transfer into a consumed child column is pending exactly when the previous step was a gap in that child:
//     term_transfer = TO[col], transfer = GO[col] (0 when the run sat before the child's first column);
//     it moves GO->GE, TO->TE and adds transfer*(ge-go) + term_transfer*(te-to) to the 24 residue scores.
//   The sums GO+GE and TO+TE that later gap starts read from an already adjusted column are invariant under (c),
//   which is what makes the columns independent.
// tests/test_prof_gpu.py compares this kernel with a CPU restatement of the reference's sequential walk and with the
// reference's own ConstructProfile.
#include <algorithm>
#include <cstring>
#include <numeric>

#include <atomic>
#include <chrono>
#include <cstdio>
#include <deque>

#include "ctx.h"
#include "prof_dev.cuh"

namespace fb {

namespace {

__global__ void __launch_bounds__(256) k_prof_leaf(const LeafDesc* __restrict__ leaves, const int8_t* __restrict__ codes,
                                                   const uint64_t* __restrict__ off, const uint32_t* __restrict__ len,
                                                   const long long* __restrict__ sm, long long go, long long ge,
                                                   long long to, long long te)
{
    leaf_body(leaves[blockIdx.x], codes, off, len, sm, go, ge, to, te);
}

__global__ void __launch_bounds__(kConThreads) k_prof_construct(const ConJobDev* __restrict__ jobs, uint32_t n_jobs,
                                                                const DpMeta* __restrict__ meta,
                                                                const famsa_dp_result* __restrict__ results,
                                                                const uint8_t* __restrict__ path_base,
                                                                long long go, long long ge, long long to, long long te)
{
    __shared__ ConShared S;
    // block -> (job, tile of kConTile merged columns)
    uint32_t lo = 0, hi = n_jobs;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (jobs[mid].tile0 <= blockIdx.x) lo = mid; else hi = mid;
    }
    ConJob J;
    const ConJobDev D = jobs[lo];
    if (!con_resolve(D, meta[D.job], results[D.job], path_base, J)) return;
    const uint32_t k0 = (blockIdx.x - J.tile0) * kConTile;          // first merged column of the tile (0 = column 0)
    if (k0 > J.W) return;                                           // the tiles were counted with the upper bound
    construct_tile(J, k0, S, go, ge, to, te);
}

size_t table_bytes(uint32_t width) { return ((size_t)width + 1) * kColBytes; }

} // namespace

void* DevArena::alloc(size_t n)
{
    n = (n + 511) & ~(size_t)511;
    auto it = free_by_size.lower_bound(n);
    if (it == free_by_size.end()) {
        const size_t want = std::max(n, chunk_bytes);
        char* base = nullptr;
        if (cudaMalloc(reinterpret_cast<void**>(&base), want) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        chunks.push_back(Chunk{base, want});
        free_by_addr[base] = {want, (int)chunks.size() - 1};
        it = free_by_size.emplace(want, base);
    }
    char* p = it->second;
    const size_t have = it->first;
    free_by_size.erase(it);
    const int chunk = free_by_addr[p].second;
    free_by_addr.erase(p);
    if (have > n) {
        free_by_addr[p + n] = {have - n, chunk};
        free_by_size.emplace(have - n, p + n);
    }
    return p;
}

void DevArena::free(void* ptr, size_t n)
{
    if (defer) { deferred.emplace_back(ptr, n); return; }
    n = (std::max<size_t>(n, 256) + 511) & ~(size_t)511;
    char* p = static_cast<char*>(ptr);
    int chunk = -1;
    for (size_t c = 0; c < chunks.size(); ++c)
        if (p >= chunks[c].base && p < chunks[c].base + chunks[c].bytes) { chunk = (int)c; break; }
    // merge with the free neighbours of the same chunk
    auto nx = free_by_addr.lower_bound(p);
    if (nx != free_by_addr.end() && nx->first == p + n && nx->second.second == chunk) {
        erase_size(nx->second.first, nx->first);
        n += nx->second.first;
        nx = free_by_addr.erase(nx);
    }
    if (nx != free_by_addr.begin()) {
        auto pv = std::prev(nx);
        if (pv->first + pv->second.first == p && pv->second.second == chunk) {
            erase_size(pv->second.first, pv->first);
            p = pv->first;
            n += pv->second.first;
            free_by_addr.erase(pv);
        }
    }
    free_by_addr[p] = {n, chunk};
    free_by_size.emplace(n, p);
}

void DevArena::release_all()
{
    for (Chunk& c : chunks) cudaFree(c.base);
    chunks.clear(); free_by_addr.clear(); free_by_size.clear();
}

namespace {

int ensure_pool(famsa_ctx* ctx)
{
    ProfState& P = ctx->prof;
    if (P.pool_ready) return FAMSA_OK;
    cudaMemPool_t pool;
    FB_CUDA(cudaDeviceGetDefaultMemPool(&pool, ctx->device));
    unsigned long long keep = ~0ull;                                // slabs are recycled by the pool, never trimmed
    FB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    for (auto& e : P.ev) FB_CUDA(cudaEventCreate(&e));
    for (auto& e : P.ev_tree) FB_CUDA(cudaEventCreate(&e));
    P.pool_ready = true;
    return FAMSA_OK;
}

int new_slab(famsa_ctx* ctx, size_t bytes, int* out)
{
    ProfState& P = ctx->prof;
    bytes = std::max<size_t>(bytes, 256);
    void* p = P.arena.alloc(bytes);
    if (!p) {
        set_error("no device memory for " + std::to_string(bytes) + " bytes of resident profiles");
        return FAMSA_E_NOMEM;
    }
    int id;
    if (!P.free_slabs.empty()) { id = P.free_slabs.back(); P.free_slabs.pop_back(); }
    else { id = (int)P.slabs.size(); P.slabs.emplace_back(); }
    P.slabs[id].p = p; P.slabs[id].bytes = bytes; P.slabs[id].live = 0;
    P.resident_bytes += bytes;
    *out = id;
    return FAMSA_OK;
}

uint32_t new_entry(ProfState& P)
{
    if (!P.free_ids.empty()) { const uint32_t id = P.free_ids.back(); P.free_ids.pop_back(); ++P.entries[id].gen; return id; }
    P.entries.emplace_back();
    return (uint32_t)P.entries.size() - 1;
}

// Carves one profile out of slab `slab` at *cursor.
void place(ProfState& P, uint32_t id, int slab, size_t* cursor, uint32_t width, uint32_t card)
{
    ProfEntry& e = P.entries[id];
    char* base = static_cast<char*>(P.slabs[slab].p) + *cursor;
    e.scores = reinterpret_cast<long long*>(base);
    e.counters = reinterpret_cast<int*>(base + ((size_t)width + 1) * kRows * sizeof(long long));
    e.width = width; e.card = card; e.slab = slab; e.live = true; e.pending = false;
    *cursor += table_bytes(width);                                  // multiple of 384: keeps 128-byte alignment
    ++P.slabs[slab].live;
    ++P.n_live;
}

// Carves the scratch tables of leaf `ld` (width `width`) out of `base` at *cursor.
void place_leaf(LeafDesc& ld, unsigned char* base, size_t* cursor, uint32_t width)
{
    char* at = reinterpret_cast<char*>(base) + *cursor;
    ld.scores = reinterpret_cast<long long*>(at);
    ld.counters = reinterpret_cast<int*>(at + ((size_t)width + 1) * kRows * sizeof(long long));
    *cursor += table_bytes(width);
}

int release_entry(famsa_ctx* ctx, uint32_t id)
{
    ProfState& P = ctx->prof;
    ProfEntry& e = P.entries[id];
    e.live = false;
    --P.n_live;
    ProfSlab& s = P.slabs[e.slab];
    if (--s.live == 0) {
        P.arena.free(s.p, s.bytes);                                  // reusable by batches queued from now on (stream order)
        P.resident_bytes -= s.bytes;
        s.p = nullptr; s.bytes = 0;
        P.free_slabs.push_back(e.slab);
    }
    e.slab = -1;
    P.free_ids.push_back(id);
    return FAMSA_OK;
}

int check_id(const ProfState& P, uint32_t id, const char* what)
{
    if (id >= P.entries.size() || !P.entries[id].live) {
        set_error(std::string(what) + ": " + std::to_string(id) + " is not a resident profile");
        return FAMSA_E_INVALID;
    }
    return FAMSA_OK;
}

} // namespace

int prof_set_scoring(famsa_ctx* ctx, const int64_t* sm)
{
    ProfState& P = ctx->prof;
    FB_TRY(ensure_pool(ctx));
    FB_TRY(P.d_sm.reserve(sizeof(long long) * kNAA * kNAA));
    FB_CUDA(cudaMemcpyAsync(P.d_sm.p, sm, sizeof(long long) * kNAA * kNAA, cudaMemcpyHostToDevice, ctx->stream));
    FB_CUDA(cudaStreamSynchronize(ctx->stream));
    P.has_scoring = true;
    return FAMSA_OK;
}

int prof_put(famsa_ctx* ctx, const famsa_dp_profile* profs, uint32_t n, uint32_t* ids)
{
    ProfState& P = ctx->prof;
    FB_TRY(ensure_pool(ctx));
    if (!n) return FAMSA_OK;
    size_t bytes = 0;
    for (uint32_t k = 0; k < n; ++k) {
        if (!profs[k].scores || !profs[k].counters || !profs[k].width || !profs[k].card) {
            set_error("famsa_prof_put: profile " + std::to_string(k) + " is empty");
            return FAMSA_E_INVALID;
        }
        bytes += table_bytes(profs[k].width);
    }
    int slab;
    FB_TRY(new_slab(ctx, bytes, &slab));
    size_t cur = 0;
    for (uint32_t k = 0; k < n; ++k) {
        const uint32_t id = new_entry(P);
        place(P, id, slab, &cur, profs[k].width, profs[k].card);
        const size_t cols = (size_t)profs[k].width + 1;
        FB_CUDA(cudaMemcpyAsync(P.entries[id].scores, profs[k].scores, cols * kRows * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        FB_CUDA(cudaMemcpyAsync(P.entries[id].counters, profs[k].counters, cols * kRows * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        ids[k] = id;
    }
    FB_CUDA(cudaStreamSynchronize(ctx->stream));
    return FAMSA_OK;
}

// d_widths[id]: the slot a pending profile's width is published to (see ProfEntry::pending)
static int ensure_widths(famsa_ctx* ctx, size_t n_ids)
{
    ProfState& P = ctx->prof;
    if (n_ids * sizeof(uint32_t) <= P.d_widths.cap) return FAMSA_OK;
    // growing moves the array: nothing may be in flight that still points into the old one
    for (const ProfEntry& e : P.entries)
        if (e.live && e.pending) { set_error("internal: width table cannot grow while merges are queued"); return FAMSA_E_STATE; }
    return P.d_widths.reserve(std::max<size_t>(n_ids * 2, 4096) * sizeof(uint32_t));
}

static cudaEvent_t take_event(ProfState& P)
{
    if (!P.free_events.empty()) { cudaEvent_t e = P.free_events.back(); P.free_events.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    return e;
}

// Queues one batch of independent merges on the context's stream and returns without waiting: leaves, DP + traceback
// (dp.cu), merged tables (k_prof_construct), then one copy of the result records and paths into h_results / h_paths
// (pinned memory makes that copy asynchronous too).  Children may be profiles of batches that are still queued -- their
// widths are then upper bounds on the host and are resolved on the device.  The merged profiles are sized for w1 + w2.
// Children of a batch of merges -> DP jobs: resident profiles by their tables (and, while they are still queued, the device
// slot their width will appear in), leaves by a descriptor for later materialisation.
static int prof_resolve(famsa_ctx* ctx, const famsa_prof_merge* merges, uint32_t n, std::vector<famsa_dp_job>& jobs, std::vector<DpJobExt>& ext,
                        std::vector<LeafDesc>& leaves, std::vector<std::pair<uint32_t, int>>& leaf_slot, size_t& leaf_bytes,
                        uint64_t& path_need, uint64_t& cells)
{
    ProfState& P = ctx->prof;
    LcsState& L = ctx->lcs;
    jobs.assign(n, famsa_dp_job{});
    ext.assign(n, DpJobExt{nullptr, nullptr, nullptr});
    std::vector<uint8_t> seen(P.entries.size(), 0);
    for (uint32_t k = 0; k < n; ++k) {
        for (int side = 0; side < 2; ++side) {
            const uint32_t c = side ? merges[k].child2 : merges[k].child1;
            famsa_dp_profile& p = side ? jobs[k].p2 : jobs[k].p1;
            const uint32_t*& src = side ? ext[k].w2_src : ext[k].w1_src;
            src = nullptr;
            if (c & FAMSA_PROF_LEAF) {
                const uint32_t seq = c & ~FAMSA_PROF_LEAF;
                if (seq >= L.n) { set_error("famsa_prof_merge_batch: leaf " + std::to_string(seq) + " was not uploaded (famsa_lcs_upload)"); return FAMSA_E_INVALID; }
                if (!P.has_scoring) { set_error("famsa_prof_merge_batch: leaves need famsa_prof_set_scoring first"); return FAMSA_E_INVALID; }
                p.width = L.h_len_sorted[L.h_invperm[seq]];
                p.card = 1;
                if (!p.width) { set_error("famsa_prof_merge_batch: leaf " + std::to_string(seq) + " is empty"); return FAMSA_E_INVALID; }
                leaves.push_back(LeafDesc{seq, nullptr, nullptr});
                leaf_slot.emplace_back(k, side);
                leaf_bytes += table_bytes(p.width);
            } else {
                FB_TRY(check_id(P, c, "famsa_prof_merge_batch"));
                if (seen[c]) { set_error("famsa_prof_merge_batch: profile " + std::to_string(c) + " is used twice"); return FAMSA_E_INVALID; }
                seen[c] = 1;
                const ProfEntry& e = P.entries[c];
                p.scores = reinterpret_cast<const int64_t*>(e.scores); p.counters = e.counters; p.width = e.width; p.card = e.card;
                if (e.pending) src = P.d_widths.as<uint32_t>() + c;
            }
        }
        path_need += (uint64_t)jobs[k].p1.width + jobs[k].p2.width;
        cells += (uint64_t)jobs[k].p1.width * jobs[k].p2.width;
    }
    return FAMSA_OK;
}

// The merged profiles of a batch: one slab, every profile pending and sized for the widest alignment possible (w1 + w2
// columns); the fill publishes the real width to d_widths[id].  Appends their ids and generations, and one construct job
// per merge (job index base + k).
static int new_merged(famsa_ctx* ctx, const std::vector<famsa_dp_job>& jobs, std::vector<DpJobExt>& ext, uint32_t base,
                      std::vector<uint32_t>& ids, std::vector<uint32_t>& gens, std::vector<ConJobDev>& con)
{
    ProfState& P = ctx->prof;
    size_t slab_bytes = 0;
    for (const famsa_dp_job& j : jobs) slab_bytes += table_bytes(j.p1.width + j.p2.width);
    int slab;
    FB_TRY(new_slab(ctx, slab_bytes, &slab));
    size_t cur = 0;
    for (uint32_t k = 0; k < (uint32_t)jobs.size(); ++k) {
        const uint32_t ub = jobs[k].p1.width + jobs[k].p2.width;
        const uint32_t id = new_entry(P);
        place(P, id, slab, &cur, ub, jobs[k].p1.card + jobs[k].p2.card);
        P.entries[id].pending = true;
        ids.push_back(id);
        gens.push_back(P.entries[id].gen);
        ext[k].w_dst = P.d_widths.as<uint32_t>() + id;
        con.push_back(ConJobDev{P.entries[id].scores, P.entries[id].counters, base + k, 0});
    }
    return FAMSA_OK;
}

static bool fused_eligible(const std::vector<famsa_dp_job>& jobs)
{
    if (jobs.size() > 4096) return false;
    for (const famsa_dp_job& j : jobs) {
        const uint32_t rows = j.p1.card == 1 ? j.p1.width : (j.p2.card == 1 ? j.p2.width : std::min(j.p1.width, j.p2.width));
        if (rows > 512 || std::max(j.p1.width, j.p2.width) > 8192) return false;
    }
    if (const char* e = getenv("FAMSA_PROF_FUSED")) return atoi(e) != 0;                            // development knob
    return true;
}

// Dependency levels of small merges accumulated for ONE launch of k_merge_fused (every merge whole in one block: leaves,
// prep, fill, traceback, merged tables; a grid barrier between the levels).  add() does the host bookkeeping of a level
// right away -- merged profiles get their ids and (upper-bound sized) tables, consumed children are released -- so that
// the next level can name them; flush() places everything and launches.
struct FusedAccum {
    std::vector<famsa_dp_job> jobs;
    std::vector<DpJobExt> ext;
    std::vector<LeafDesc> leaves;
    std::vector<std::pair<uint32_t, int>> leaf_slot;                 // (job, side), job index over the whole accumulation
    std::vector<uint32_t> level_start{0};
    std::vector<uint32_t> merged_ids, merged_gen;
    std::vector<ConJobDev> con;
    size_t leaf_bytes = 0, dev_bytes_est = 0;
    uint64_t path_bytes = 0;                                         // host path slots used (16-byte aligned when host_mapped)
    uint32_t max_level = 0;
    bool empty() const { return jobs.empty(); }
};

static size_t fused_dev_estimate(const famsa_dp_job& j)
{
    return sizeof(famsa_dp_result) + sizeof(DpMeta) + align_up((uint64_t)j.p1.width + j.p2.width, 16) + 2 * 384ull * (std::max(j.p1.width, j.p2.width) + 2) +
           dp_scratch_bytes(j.p1.width, j.p2.width) + skew_elems(j.p1.width, j.p2.width) + 1024;
}

// may the level (already resolved into `jobs`) join the accumulation?  Checks the rings conservatively.
static bool fused_fits(famsa_ctx* ctx, const FusedAccum& A, const std::vector<famsa_dp_job>& jobs)
{
    ProfState& P = ctx->prof;
    size_t dev = A.dev_bytes_est;
    for (const famsa_dp_job& j : jobs) dev += fused_dev_estimate(j);
    const size_t host = (A.jobs.size() + jobs.size()) * (sizeof(DpJobDev) + sizeof(FusedJob)) + (A.level_start.size() + 2) * sizeof(uint32_t) + 1024;
    return P.d_ring.fits(dev + 4096) && P.h_ring.fits(host);
}

static int fused_add(famsa_ctx* ctx, FusedAccum& A, const famsa_prof_merge* merges, uint32_t n, std::vector<famsa_dp_job>& jobs, std::vector<DpJobExt>& ext,
                     std::vector<LeafDesc>& leaves, std::vector<std::pair<uint32_t, int>>& leaf_slot, size_t leaf_bytes, bool align16)
{
    ProfState& P = ctx->prof;
    const uint32_t base = (uint32_t)A.jobs.size();
    FB_TRY(new_merged(ctx, jobs, ext, base, A.merged_ids, A.merged_gen, A.con));
    for (uint32_t k = 0; k < n; ++k) {
        A.dev_bytes_est += fused_dev_estimate(jobs[k]);
        A.path_bytes += align16 ? align_up((uint64_t)jobs[k].p1.width + jobs[k].p2.width, 16) : (uint64_t)jobs[k].p1.width + jobs[k].p2.width;
    }
    for (auto& ls : leaf_slot) ls.first += base;
    A.jobs.insert(A.jobs.end(), jobs.begin(), jobs.end());
    A.ext.insert(A.ext.end(), ext.begin(), ext.end());
    A.leaves.insert(A.leaves.end(), leaves.begin(), leaves.end());
    A.leaf_slot.insert(A.leaf_slot.end(), leaf_slot.begin(), leaf_slot.end());
    A.leaf_bytes += leaf_bytes;
    A.level_start.push_back((uint32_t)A.jobs.size());
    A.max_level = std::max(A.max_level, n);
    // the children are consumed (msa.cpp:406-407).  Their storage must not be handed out again before this launch has
    // been queued: inside one launch there is no kernel boundary that would invalidate a stale L1 line
    P.arena.defer = true;
    for (uint32_t k = 0; k < n; ++k)
        for (uint32_t c : {merges[k].child1, merges[k].child2})
            if (!(c & FAMSA_PROF_LEAF)) FB_TRY(release_entry(ctx, c));
    return FAMSA_OK;
}

static int fused_flush(famsa_ctx* ctx, FusedAccum& A, const int64_t gaps[4], famsa_dp_result* h_results, uint8_t* h_paths, bool host_mapped, ProfTicket* T)
{
    ProfState& P = ctx->prof;
    LcsState& L = ctx->lcs;
    cudaStream_t st = ctx->stream;
    const uint32_t n = (uint32_t)A.jobs.size(), n_levels = (uint32_t)A.level_start.size() - 1;
    std::vector<DpJobDev> plan_jobs(n);
    DpFusedPlan plan;
    FB_TRY(dp_fused_plan(A.jobs.data(), A.ext.data(), n, host_mapped, plan_jobs.data(), &plan));
    const size_t ho_fj = align_up(sizeof(DpJobDev) * n, 256);
    const size_t ho_lv = align_up(ho_fj + sizeof(FusedJob) * n, 256);
    const size_t h_bytes = ho_lv + sizeof(uint32_t) * (n_levels + 1);
    const size_t o_res = 0;
    const size_t o_meta = align_up(o_res + sizeof(famsa_dp_result) * n, 256);
    const size_t o_path = align_up(o_meta + sizeof(DpMeta) * n, 256);
    const size_t o_leaf = align_up(o_path + std::max<uint64_t>(plan.path_bytes, 1), 256);
    const size_t o_scr = align_up(o_leaf + A.leaf_bytes, 256);
    const size_t o_skew = align_up(o_scr + plan.scratch_bytes, 256);
    const size_t d_bytes = o_skew + plan.skew_bytes;
    const size_t h_off = P.h_ring.alloc(h_bytes), d_off = P.d_ring.alloc(d_bytes);
    if (h_off == (size_t)-1 || d_off == (size_t)-1) { set_error("internal: the fused batch does not fit its rings"); return FAMSA_E_NOMEM; }
    unsigned char* hb = P.h_ring_mem + h_off;
    unsigned char* db = P.d_ring_mem.as<unsigned char>() + d_off;
    DpJobDev* hj = reinterpret_cast<DpJobDev*>(hb);
    FusedJob* fj = reinterpret_cast<FusedJob*>(hb + ho_fj);
    uint32_t* hl = reinterpret_cast<uint32_t*>(hb + ho_lv);
    famsa_dp_result* d_results = reinterpret_cast<famsa_dp_result*>(db + o_res);
    for (uint32_t k = 0; k < n; ++k) { fj[k].leaf[0].seq = fj[k].leaf[1].seq = 0xffffffffu; fj[k].con = A.con[k]; }
    size_t cur = 0;
    for (size_t a = 0; a < A.leaves.size(); ++a) {
        const auto [k, side] = A.leaf_slot[a];
        LeafDesc& ld = A.leaves[a];
        place_leaf(ld, db + o_leaf, &cur, side ? A.jobs[k].p2.width : A.jobs[k].p1.width);
        (side ? plan_jobs[k].s2 : plan_jobs[k].s1) = ld.scores;
        (side ? plan_jobs[k].c2 : plan_jobs[k].c1) = ld.counters;
        fj[k].leaf[side] = ld;
    }
    memcpy(hj, plan_jobs.data(), sizeof(DpJobDev) * n);
    memcpy(hl, A.level_start.data(), sizeof(uint32_t) * (n_levels + 1));
    FusedParams FP{fj, hl, n_levels, L.d_raw_codes.as<int8_t>(), L.d_raw_off.as<uint64_t>(), L.d_raw_len.as<uint32_t>(), P.d_sm.as<long long>(),
                   0, P.d_block_counter.as<unsigned>(), nullptr, 0};
    if (host_mapped) { FP.h_done = P.h_done; FP.done_seq = ++P.done_seq; }
    if (getenv("FAMSA_FUSED_TIMING")) { static int launch_no = 0; FP.timing = 2 + (++launch_no & 1); }   // development aid
    if (!host_mapped) { FB_CUDA(cudaEventRecord(P.ev[0], st)); FB_CUDA(cudaEventRecord(P.ev[1], st)); }
    const uint32_t grid = std::max(1u, std::min(A.max_level, (uint32_t)ctx->sm_count));      // co-resident: the levels meet at a spin barrier
    FB_TRY(dp_fused_launch(ctx, hj, n, gaps, d_results, db + o_path, reinterpret_cast<DpMeta*>(db + o_meta), db + o_scr, db + o_skew,
                           host_mapped ? h_results : nullptr, host_mapped ? h_paths : nullptr, FP, grid, plan.cells, !host_mapped, st));
    if (!host_mapped) {
        FB_CUDA(cudaEventRecord(P.ev[2], st));
        P.timing_valid = true;
        FB_CUDA(cudaMemcpyAsync(h_results, d_results, sizeof(famsa_dp_result) * n, cudaMemcpyDeviceToHost, st));
        if (plan.path_bytes) FB_CUDA(cudaMemcpyAsync(h_paths, db + o_path, plan.path_bytes, cudaMemcpyDeviceToHost, st));
        T->done = take_event(P);
        FB_CUDA(cudaEventRecord(T->done, st));
    } else T->done_seq = FP.done_seq;
    // storage of the consumed children may be handed out again from here on (everything later is behind this launch)
    P.arena.flush_deferred();
    T->merged_ids = A.merged_ids; T->merged_gen = A.merged_gen;
    T->n = n; T->h_results = h_results; T->h_paths = h_paths; T->path_bytes = plan.path_bytes; T->cells_bound = plan.cells;
    T->ring_host_end = P.h_ring.head; T->ring_dev_end = P.d_ring.head;
    A = FusedAccum();
    return FAMSA_OK;
}

static int ensure_rings(famsa_ctx* ctx)
{
    ProfState& P = ctx->prof;
    if (P.h_ring_mem) return FAMSA_OK;
    const size_t hcap = 8u << 20, dcap = 512u << 20;
    FB_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&P.h_ring_mem), hcap, cudaHostAllocMapped));
    P.h_ring.cap = hcap;
    FB_TRY(P.d_ring_mem.reserve(dcap));
    P.d_ring.cap = dcap;
    FB_CUDA(cudaHostAlloc(reinterpret_cast<void**>(const_cast<unsigned long long**>(&P.h_done)), 64, cudaHostAllocMapped));
    *P.h_done = 0;
    FB_TRY(P.d_block_counter.reserve(64));
    FB_CUDA(cudaMemsetAsync(P.d_block_counter.p, 0, 64, ctx->stream));
    return FAMSA_OK;
}

// host_mapped: h_results / h_paths are mapped pinned memory the device may write to directly (and path slots are 16-byte
// aligned: job k's path at the running sum of align16(w1 + w2))
static int prof_launch(famsa_ctx* ctx, const famsa_prof_merge* merges, uint32_t n, const int64_t gaps[4],
                       famsa_dp_result* h_results, uint8_t* h_paths, uint64_t path_cap, bool host_mapped, ProfTicket* T)
{
    ProfState& P = ctx->prof;
    LcsState& L = ctx->lcs;
    cudaStream_t st = ctx->stream;

    // resolve the children; leaves get scratch tables for the duration of the batch
    std::vector<famsa_dp_job> jobs;
    std::vector<DpJobExt> ext;
    std::vector<LeafDesc> leaves;
    std::vector<std::pair<uint32_t, int>> leaf_slot;                 // (job, side) per leaf, in `leaves` order
    size_t leaf_bytes = 0;
    uint64_t path_need = 0, cells = 0;
    FB_TRY(prof_resolve(ctx, merges, n, jobs, ext, leaves, leaf_slot, leaf_bytes, path_need, cells));
    if (host_mapped) {
        path_need = 0;
        for (uint32_t k = 0; k < n; ++k) path_need += align_up((uint64_t)jobs[k].p1.width + jobs[k].p2.width, 16);
    }
    if (path_need > path_cap) {
        set_error("famsa_prof_merge_batch: path_buf holds " + std::to_string(path_cap) + " bytes, " + std::to_string(path_need) + " needed");
        return FAMSA_E_INVALID;
    }
    FB_TRY(ensure_widths(ctx, P.entries.size() + n));
    // A batch of small merges only (the chain-like parts of a guide tree: every level one or a few short merges) runs
    // every merge whole in one block of k_merge_fused instead of five launches.
    if (fused_eligible(jobs)) {
        FB_TRY(ensure_rings(ctx));
        FusedAccum A;
        if (fused_fits(ctx, A, jobs)) {
            FB_TRY(fused_add(ctx, A, merges, n, jobs, ext, leaves, leaf_slot, leaf_bytes, host_mapped));
            return fused_flush(ctx, A, gaps, h_results, h_paths, host_mapped, T);
        }
    }
    T->merged_ids.clear();
    T->merged_gen.clear();
    std::vector<ConJobDev> con;
    FB_TRY(new_merged(ctx, jobs, ext, 0, T->merged_ids, T->merged_gen, con));
    uint32_t tiles = 0;
    for (uint32_t k = 0; k < n; ++k) {
        con[k].tile0 = tiles;
        tiles += (jobs[k].p1.width + jobs[k].p2.width + 1 + kConTile - 1) / kConTile;
    }
    // batch blob: [results][con jobs][leaf descs][paths][leaf tables]
    const size_t o_res = 0;
    const size_t o_con = align_up(o_res + sizeof(famsa_dp_result) * n, 256);
    const size_t o_leafd = align_up(o_con + sizeof(ConJobDev) * n, 256);
    const size_t o_path = align_up(o_leafd + sizeof(LeafDesc) * leaves.size(), 256);
    const size_t o_leaf = align_up(o_path + std::max<uint64_t>(path_need, 1), 256);
    const size_t blob_bytes = o_leaf + leaf_bytes;
    unsigned char* blob = nullptr;
    {
        cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&blob), blob_bytes, st);
        if (e != cudaSuccess) { set_error(std::string("cudaMallocAsync for a merge batch failed: ") + cudaGetErrorString(e)); return FAMSA_E_NOMEM; }
    }
    famsa_dp_result* d_results = reinterpret_cast<famsa_dp_result*>(blob + o_res);
    uint8_t* d_path = blob + o_path;

    // one upload: [con jobs][leaf descs]
    std::vector<unsigned char> pack(o_path - o_con);
    memcpy(pack.data(), con.data(), sizeof(ConJobDev) * n);
    LeafDesc* ld = reinterpret_cast<LeafDesc*>(pack.data() + (o_leafd - o_con));
    size_t cur = 0;
    for (size_t a = 0; a < leaves.size(); ++a) {
        famsa_dp_profile& p = leaf_slot[a].second ? jobs[leaf_slot[a].first].p2 : jobs[leaf_slot[a].first].p1;
        place_leaf(leaves[a], blob + o_leaf, &cur, p.width);
        p.scores = reinterpret_cast<const int64_t*>(leaves[a].scores);
        p.counters = leaves[a].counters;
        ld[a] = leaves[a];
    }
    FB_CUDA(cudaEventRecord(P.ev[0], st));
    FB_CUDA(cudaMemcpyAsync(blob + o_con, pack.data(), pack.size(), cudaMemcpyHostToDevice, st));
    if (!leaves.empty()) {
        k_prof_leaf<<<(unsigned)leaves.size(), 256, 0, st>>>(reinterpret_cast<const LeafDesc*>(blob + o_leafd), L.d_raw_codes.as<int8_t>(),
                                                             L.d_raw_off.as<uint64_t>(), L.d_raw_len.as<uint32_t>(),
                                                             P.d_sm.as<long long>(), gaps[0], gaps[1], gaps[2], gaps[3]);
        FB_CUDA(cudaGetLastError());
        ++ctx->launches;
    }
    // DP + traceback on the resident tables (dp.cu)
    DpMeta* d_meta = nullptr;
    void* dp_blob = nullptr;
    FB_TRY(dp_run_device(ctx, jobs.data(), ext.data(), n, gaps, d_results, d_path, nullptr, &d_meta, &dp_blob, st));
    FB_CUDA(cudaEventRecord(P.ev[1], st));
    k_prof_construct<<<tiles, kConThreads, 0, st>>>(reinterpret_cast<const ConJobDev*>(blob + o_con), n, d_meta, d_results, d_path,
                                                    gaps[0], gaps[1], gaps[2], gaps[3]);
    FB_CUDA(cudaGetLastError());
    ++ctx->launches;
    FB_CUDA(cudaEventRecord(P.ev[2], st));
    P.timing_valid = true;
    FB_CUDA(cudaMemcpyAsync(h_results, d_results, sizeof(famsa_dp_result) * n, cudaMemcpyDeviceToHost, st));
    if (path_need) FB_CUDA(cudaMemcpyAsync(h_paths, d_path, path_need, cudaMemcpyDeviceToHost, st));
    FB_CUDA(cudaFreeAsync(dp_blob, st));
    FB_CUDA(cudaFreeAsync(blob, st));
    // the children are consumed (msa.cpp:406-407); frees are ordered after the construct kernel
    for (uint32_t k = 0; k < n; ++k)
        for (uint32_t c : {merges[k].child1, merges[k].child2})
            if (!(c & FAMSA_PROF_LEAF)) FB_TRY(release_entry(ctx, c));
    T->done = take_event(P);
    FB_CUDA(cudaEventRecord(T->done, st));
    T->n = n; T->h_results = h_results; T->h_paths = h_paths; T->path_bytes = path_need; T->cells_bound = cells;
    return FAMSA_OK;
}

// Waits for a queued batch and takes note of the merged widths.
static int prof_collect(famsa_ctx* ctx, ProfTicket* T)
{
    ProfState& P = ctx->prof;
    if (T->done_seq) {
        // flag-tracked batch: the kernel's last block published its sequence number after fencing every block's results
        unsigned spins = 0;
        while (*P.h_done < T->done_seq) {
            if (++spins > 2000000u) {                                // ~ seconds: make sure the device is still alive
                const cudaError_t e = cudaStreamQuery(ctx->stream);
                if (e != cudaSuccess && e != cudaErrorNotReady) { FB_CUDA(e); }
                if (e == cudaSuccess && *P.h_done < T->done_seq) { set_error("internal: a flag-tracked batch finished without publishing"); return FAMSA_E_CUDA; }
                spins = 0;
            }
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        std::atomic_thread_fence(std::memory_order_acquire);
        T->done_seq = 0;
    } else if (T->done) {
        FB_CUDA(cudaEventSynchronize(T->done));
        P.free_events.push_back(T->done);
        T->done = nullptr;
    }
    if (T->ring_host_end != (size_t)-1) { P.h_ring.release_to(T->ring_host_end); T->ring_host_end = (size_t)-1; }
    if (T->ring_dev_end != (size_t)-1) { P.d_ring.release_to(T->ring_dev_end); T->ring_dev_end = (size_t)-1; }
    int rc = FAMSA_OK;
    for (uint32_t k = 0; k < T->n; ++k) {
        ProfEntry& e = P.entries[T->merged_ids[k]];
        const famsa_dp_result& r = T->h_results[k];
        if (e.live && e.pending && e.gen == T->merged_gen[k]) {     // (a later batch may already have consumed it)
            e.pending = false;
            if (r.variant != 0xFF) e.width = r.path_len;
        }
        if (r.variant == 0xFF && rc == FAMSA_OK) {
            set_error("merge " + std::to_string(k) + " of the batch: a profile holds negative residue / gap counts");
            rc = FAMSA_E_INVALID;
        }
    }
    return rc;
}

int prof_merge_batch(famsa_ctx* ctx, const famsa_prof_merge* merges, uint32_t n, const int64_t gaps[4], uint32_t* merged_ids,
                     famsa_dp_result* results, uint8_t* path_buf, uint64_t path_cap)
{
    ProfState& P = ctx->prof;
    FB_TRY(ensure_pool(ctx));
    P.timing_valid = false;
    if (!n) return FAMSA_OK;
    ProfTicket T;
    FB_TRY(prof_launch(ctx, merges, n, gaps, results, path_buf, path_cap, false, &T));
    const int rc = prof_collect(ctx, &T);
    for (uint32_t k = 0; k < n; ++k) merged_ids[k] = T.merged_ids[k];
    return rc;
}

// ------------------------------------------------------------------------------------------------
// The whole progressive alignment (CFAMSA::ComputeAlignment, msa.cpp:360-438) as one call.
//
// The reference hands a merge to a worker thread as soon as both children are finished, deepest node first
// (CProfileQueue, queues.cpp:27-40, 127-187).  Here the unit of submission is "every merge that is ready", and the host
// does not wait for a batch before it queues the next one: all a parent needs from its children on the host side is an
// upper bound of their widths (to size buffers); the real widths travel on the device.  Several batches are therefore in
// flight on the stream while the host collects finished ones in the background to tighten its bounds; it only drains
// the queue when the bounds of the next batch would inflate its scratch beyond what the real widths would need.
// ------------------------------------------------------------------------------------------------
static int pinned_reserve(void** p, size_t* cap, size_t bytes)
{
    if (bytes <= *cap) return FAMSA_OK;
    if (*p) cudaFreeHost(*p);
    *p = nullptr; *cap = 0;
    const size_t want = bytes + bytes / 4 + 4096;
    FB_CUDA(cudaHostAlloc(p, want, cudaHostAllocMapped));
    *cap = want;
    return FAMSA_OK;
}

int prof_align_tree(famsa_ctx* ctx, const int32_t* tree, uint32_t n_leaves, const int64_t gaps[4], famsa_dp_result* results,
                    uint32_t* root_id, uint64_t* path_bytes, famsa_tree_stats* stats)
{
    ProfState& P = ctx->prof;
    LcsState& L = ctx->lcs;
    FB_TRY(ensure_pool(ctx));
    const auto t_begin = std::chrono::steady_clock::now();
    if (n_leaves != L.n) { set_error("famsa_prof_align_tree: the tree has " + std::to_string(n_leaves) + " leaves, " + std::to_string(L.n) + " sequences are uploaded"); return FAMSA_E_INVALID; }
    if (!P.has_scoring) { set_error("famsa_prof_align_tree: famsa_prof_set_scoring first"); return FAMSA_E_STATE; }
    if (n_leaves < 2) { set_error("famsa_prof_align_tree: fewer than two sequences"); return FAMSA_E_INVALID; }
    const uint32_t n_merges = n_leaves - 1, n_nodes = 2 * n_leaves - 1;
    // dependency levels; children must precede parents (tree_structure order)
    std::vector<uint32_t> depth(n_nodes, 0);
    std::vector<std::vector<uint32_t>> levels;
    std::vector<uint8_t> used(n_nodes, 0);
    for (uint32_t k = 0; k < n_merges; ++k) {
        const int32_t a = tree[2 * k], b = tree[2 * k + 1];
        if (a < 0 || b < 0 || (uint32_t)a >= n_leaves + k || (uint32_t)b >= n_leaves + k || a == b || used[a] || used[b]) {
            set_error("famsa_prof_align_tree: node " + std::to_string(n_leaves + k) + " has invalid children");
            return FAMSA_E_INVALID;
        }
        used[a] = used[b] = 1;
        const uint32_t d = std::max(depth[a], depth[b]) + 1;
        depth[n_leaves + k] = d;
        if (levels.size() < d) levels.resize(d);
        levels[d - 1].push_back(k);
    }
    FB_TRY(ensure_widths(ctx, P.entries.size() + n_merges + 16));
    FB_TRY(pinned_reserve(reinterpret_cast<void**>(&P.h_tree_results), &P.h_tree_results_cap, sizeof(famsa_dp_result) * n_merges));

    std::vector<uint32_t> handle(n_nodes), width(n_nodes);           // width: layout width (bound until collected)
    for (uint32_t i = 0; i < n_leaves; ++i) { handle[i] = FAMSA_PROF_LEAF | i; width[i] = L.h_len_sorted[L.h_invperm[i]]; }
    struct InFlight { ProfTicket t; std::vector<uint32_t> merge_ids; uint64_t path_base; size_t res_base; };
    std::deque<InFlight> q;
    uint64_t path_cursor = 0, cells = 0;
    size_t res_cursor = 0;
    uint32_t n_batches = 0, max_in_flight = 0, n_drains = 0;
    uint64_t peak_bytes = 0;
    constexpr size_t kMaxInFlight = 8;
    FB_CUDA(cudaEventRecord(P.ev_tree[0], ctx->stream));
    double t_collect = 0, t_launch = 0;
    uint32_t max_exact = 0;                                         // widest profile whose real width is known
    for (uint32_t i = 0; i < n_leaves; ++i) max_exact = std::max(max_exact, width[i]);
    auto now = []() { return std::chrono::steady_clock::now(); };
    auto collect_front = [&]() -> int {
        InFlight& f = q.front();
        const auto t0 = now();
        const int rc = prof_collect(ctx, &f.t);
        t_collect += std::chrono::duration<double, std::micro>(now() - t0).count();
        for (size_t a = 0; a < f.merge_ids.size(); ++a) {
            const uint32_t k = f.merge_ids[a];
            famsa_dp_result& r = P.h_tree_results[f.res_base + a];
            r.path_offset += f.path_base;
            results[k] = r;
            width[n_leaves + k] = r.path_len;
            max_exact = std::max(max_exact, r.path_len);
            cells += (uint64_t)r.rows_width * r.cols_width;
        }
        q.pop_front();
        return rc;
    };
    int rc = FAMSA_OK;
    // paths of all merges: one pinned arena, grown only while nothing is in flight
    uint64_t arena_need = 0;
    for (uint32_t i = 0; i < n_leaves; ++i) arena_need += width[i];
    arena_need = arena_need * 8 + (64u << 20);
    FB_TRY(pinned_reserve(reinterpret_cast<void**>(&P.h_tree_paths), &P.h_tree_paths_cap, arena_need));
    // Consecutive levels of small merges are accumulated into ONE launch of the fused kernel (a grid barrier between the
    // levels instead of a kernel boundary): the chain-like stretches of a guide tree are a single merge per level.
    FB_TRY(ensure_rings(ctx));
    FusedAccum acc;
    std::vector<uint32_t> acc_merges;
    uint64_t acc_path_base = 0;
    size_t acc_res_base = 0;
    uint32_t acc_levels = 0;
    constexpr uint32_t kMaxFusedLevels = 32;
    auto flush_acc = [&]() -> int {
        if (acc.empty()) return FAMSA_OK;
        // at most two fused launches uncollected: the widths of everything older become exact, which keeps the upper bounds
        // of the levels being accumulated (sums over the uncollected part of a chain) from running away
        while (q.size() >= 2) { const int r = collect_front(); if (r) return r; }
        q.emplace_back();
        InFlight& f = q.back();
        f.merge_ids = acc_merges;
        f.path_base = acc_path_base;
        f.res_base = acc_res_base;
        if (dp_debug()) fprintf(stderr, "[tree] fused launch: %u levels, %zu merges\n", acc_levels, acc.jobs.size());
        const auto t0 = now();
        const int r = fused_flush(ctx, acc, gaps, P.h_tree_results + acc_res_base, P.h_tree_paths + acc_path_base, true, &f.t);
        t_launch += std::chrono::duration<double, std::micro>(now() - t0).count();
        if (r) { q.pop_back(); return r; }
        acc_merges.clear();
        acc_levels = 0;
        ++n_batches;
        max_in_flight = std::max<uint32_t>(max_in_flight, (uint32_t)q.size());
        return FAMSA_OK;
    };
    auto finished = [&](const ProfTicket& t) { return t.done_seq ? *P.h_done >= t.done_seq : (!t.done || cudaEventQuery(t.done) == cudaSuccess); };
    for (size_t lv = 0; lv < levels.size() && rc == FAMSA_OK; ++lv) {
        const std::vector<uint32_t>& level = levels[lv];
        std::vector<famsa_prof_merge> mg(level.size());
        for (size_t a = 0; a < level.size(); ++a) {
            const uint32_t k = level[a];
            mg[a].child1 = handle[(uint32_t)tree[2 * k]];
            mg[a].child2 = handle[(uint32_t)tree[2 * k + 1]];
        }
        {
            // small merges: join the accumulation when the level fits
            while (!q.empty() && finished(q.front().t) && rc == FAMSA_OK) rc = collect_front();
            if (rc) break;
            // A queued child is known by an upper bound only (the sum of its children's bounds), and along a chain the bounds
            // add up level after level however many older levels have been collected since.  Once a bound has drifted far
            // from anything real, wait for the device: every width becomes exact again.
            bool drifted = false;
            for (uint32_t k : level)
                for (int side = 0; side < 2; ++side) {
                    const uint32_t c = (uint32_t)tree[2 * k + side];
                    if (c >= n_leaves && P.entries[handle[c]].pending && width[c] > 1024 + 2 * max_exact) drifted = true;
                }
            if (drifted) {
                rc = flush_acc();
                while (!q.empty() && rc == FAMSA_OK) rc = collect_front();
                if (rc) break;
                ++n_drains;
            }
            std::vector<famsa_dp_job> jobs;
            std::vector<DpJobExt> ext;
            std::vector<LeafDesc> leaves;
            std::vector<std::pair<uint32_t, int>> leaf_slot;
            size_t leaf_bytes = 0;
            uint64_t pn = 0, cl = 0;
            rc = prof_resolve(ctx, mg.data(), (uint32_t)mg.size(), jobs, ext, leaves, leaf_slot, leaf_bytes, pn, cl);
            if (rc) break;
            uint64_t path_need = 0;
            for (const famsa_dp_job& j : jobs) path_need += align_up((uint64_t)j.p1.width + j.p2.width, 16);
            if (fused_eligible(jobs) && path_cursor + path_need <= P.h_tree_paths_cap) {
                if (!(acc_levels < kMaxFusedLevels && acc.jobs.size() + jobs.size() <= 8192 && fused_fits(ctx, acc, jobs))) {
                    rc = flush_acc();
                    if (rc) break;
                    while (q.size() >= kMaxInFlight && rc == FAMSA_OK) rc = collect_front();
                    while (!fused_fits(ctx, acc, jobs) && !q.empty() && rc == FAMSA_OK) rc = collect_front();   // ring space comes back in order
                    if (rc) break;
                }
                if (fused_fits(ctx, acc, jobs)) {
                    if (acc.empty()) { acc_path_base = path_cursor; acc_res_base = res_cursor; }
                    const size_t first = acc.merged_ids.size();
                    rc = fused_add(ctx, acc, mg.data(), (uint32_t)mg.size(), jobs, ext, leaves, leaf_slot, leaf_bytes, true);
                    if (rc) break;
                    for (size_t a = 0; a < level.size(); ++a) {
                        const uint32_t k = level[a];
                        handle[n_leaves + k] = acc.merged_ids[first + a];
                        width[n_leaves + k] = P.entries[acc.merged_ids[first + a]].width;   // the bound w1 + w2
                    }
                    acc_merges.insert(acc_merges.end(), level.begin(), level.end());
                    path_cursor += path_need;
                    res_cursor += level.size();
                    ++acc_levels;
                    peak_bytes = std::max(peak_bytes, P.resident_bytes);
                    continue;
                }
            }
            if (dp_debug()) fprintf(stderr, "[tree] level %zu (%zu merges) not fused: eligible %d, path room %d\n", lv, level.size(), (int)fused_eligible(jobs), (int)(path_cursor + path_need <= P.h_tree_paths_cap)), fprintf(stderr, "        first job: %u (card %u) x %u (card %u)\n", jobs[0].p1.width, jobs[0].p1.card, jobs[0].p2.width, jobs[0].p2.card);
            rc = flush_acc();                                         // this level goes launch by launch: everything before it first
            if (rc) break;
        }
        // collect whatever has finished already (tightens the bounds for free)
        while (!q.empty() && finished(q.front().t) && rc == FAMSA_OK) rc = collect_front();
        if (rc) break;
        auto level_cost = [&](uint64_t* bound_cells, uint64_t* path_need) {
            *bound_cells = *path_need = 0;
            for (uint32_t k : level) {
                const uint32_t a = (uint32_t)tree[2 * k], b = (uint32_t)tree[2 * k + 1];
                *bound_cells += (uint64_t)width[a] * width[b];
                *path_need += align_up((uint64_t)width[a] + width[b], 16);
            }
        };
        uint64_t bound_cells, path_need;
        level_cost(&bound_cells, &path_need);
        // Run ahead of the device only while that is cheap: a few batches deep, and not when the bounds of this level
        // (sums of bounds of uncollected children) would make its direction matrices much larger than they need to be.
        bool pending_child = false;
        for (uint32_t k : level)
            for (int s = 0; s < 2; ++s) {
                const uint32_t c = (uint32_t)tree[2 * k + s];
                if (c >= n_leaves && P.entries[handle[c]].pending) pending_child = true;
            }
        const bool heavy = bound_cells > (64ull << 20);
        if ((pending_child && heavy) || q.size() >= kMaxInFlight || path_cursor + path_need > P.h_tree_paths_cap) {
            const bool all = (pending_child && heavy) || path_cursor + path_need > P.h_tree_paths_cap;
            while (!q.empty() && rc == FAMSA_OK && (all || q.size() >= kMaxInFlight)) rc = collect_front();
            if (rc) break;
            ++n_drains;
            level_cost(&bound_cells, &path_need);
            if (path_cursor + path_need > P.h_tree_paths_cap) {      // nothing in flight now: the arena may move
                uint8_t* old = P.h_tree_paths;
                P.h_tree_paths = nullptr; P.h_tree_paths_cap = 0;
                FB_TRY(pinned_reserve(reinterpret_cast<void**>(&P.h_tree_paths), &P.h_tree_paths_cap, (path_cursor + path_need) * 2));
                memcpy(P.h_tree_paths, old, path_cursor);
                cudaFreeHost(old);
            }
        }
        q.emplace_back();
        InFlight& f = q.back();
        f.merge_ids = level;
        f.path_base = path_cursor;
        f.res_base = res_cursor;
        const auto t0 = now();
        rc = prof_launch(ctx, mg.data(), (uint32_t)mg.size(), gaps, P.h_tree_results + res_cursor, P.h_tree_paths + path_cursor,
                         P.h_tree_paths_cap - path_cursor, true, &f.t);
        t_launch += std::chrono::duration<double, std::micro>(now() - t0).count();
        if (rc) { q.pop_back(); break; }
        for (size_t a = 0; a < level.size(); ++a) {
            const uint32_t k = level[a];
            handle[n_leaves + k] = f.t.merged_ids[a];
            width[n_leaves + k] = P.entries[f.t.merged_ids[a]].width;       // the bound w1 + w2
        }
        path_cursor += path_need;
        res_cursor += level.size();
        ++n_batches;
        max_in_flight = std::max<uint32_t>(max_in_flight, (uint32_t)q.size());
        peak_bytes = std::max(peak_bytes, P.resident_bytes);
    }
    if (rc == FAMSA_OK) rc = flush_acc();
    while (!q.empty()) { const int r2 = collect_front(); if (rc == FAMSA_OK) rc = r2; }
    if (rc) return rc;
    if (dp_debug())
        fprintf(stderr, "[tree] host time: %.0f us in prof_launch, %.0f us waiting in prof_collect, %.0f us total so far, %u batches\n", t_launch, t_collect,
                std::chrono::duration<double, std::micro>(now() - t_begin).count(), n_batches);
    FB_CUDA(cudaEventRecord(P.ev_tree[1], ctx->stream));
    FB_CUDA(cudaEventSynchronize(P.ev_tree[1]));
    float dev_ms = 0.f;
    FB_CUDA(cudaEventElapsedTime(&dev_ms, P.ev_tree[0], P.ev_tree[1]));
    P.tree_path_bytes = path_cursor;
    P.tree_merges = n_merges;
    if (root_id) *root_id = handle[n_nodes - 1];
    if (path_bytes) *path_bytes = path_cursor;
    if (stats) {
        stats->wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        stats->device_ms = dev_ms;
        stats->cells = cells;
        stats->n_batches = n_batches;
        stats->n_drains = n_drains;
        stats->max_in_flight = max_in_flight;
        stats->peak_resident_bytes = peak_bytes;
    }
    return FAMSA_OK;
}

int prof_tree_paths(famsa_ctx* ctx, uint8_t* path_buf, uint64_t cap)
{
    ProfState& P = ctx->prof;
    if (!P.tree_merges) { set_error("famsa_prof_tree_paths: no famsa_prof_align_tree has run"); return FAMSA_E_STATE; }
    if (cap < P.tree_path_bytes) { set_error("famsa_prof_tree_paths: buffer holds " + std::to_string(cap) + " bytes, " + std::to_string(P.tree_path_bytes) + " needed"); return FAMSA_E_INVALID; }
    memcpy(path_buf, P.h_tree_paths, P.tree_path_bytes);
    return FAMSA_OK;
}

int prof_get(famsa_ctx* ctx, uint32_t id, uint32_t* width, uint32_t* card, int64_t* scores, int32_t* counters)
{
    ProfState& P = ctx->prof;
    FB_TRY(check_id(P, id, "famsa_prof_get"));
    const ProfEntry& e = P.entries[id];
    if (width) *width = e.width;
    if (card) *card = e.card;
    const size_t cells = ((size_t)e.width + 1) * kRows;
    if (scores) FB_CUDA(cudaMemcpyAsync(scores, e.scores, cells * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    if (counters) FB_CUDA(cudaMemcpyAsync(counters, e.counters, cells * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (scores || counters) FB_CUDA(cudaStreamSynchronize(ctx->stream));
    return FAMSA_OK;
}

int prof_drop(famsa_ctx* ctx, const uint32_t* ids, uint32_t n)
{
    ProfState& P = ctx->prof;
    for (uint32_t k = 0; k < n; ++k) FB_TRY(check_id(P, ids[k], "famsa_prof_drop"));
    for (uint32_t k = 0; k < n; ++k) {
        if (!P.entries[ids[k]].live) { set_error("famsa_prof_drop: profile listed twice"); return FAMSA_E_INVALID; }
        FB_TRY(release_entry(ctx, ids[k]));
    }
    return FAMSA_OK;
}

int prof_last_timing(famsa_ctx* ctx, float* total_ms, float* construct_ms)
{
    ProfState& P = ctx->prof;
    if (!P.timing_valid) { set_error("no famsa_prof_merge_batch has run"); return FAMSA_E_INVALID; }
    FB_CUDA(cudaEventSynchronize(P.ev[2]));
    float a = 0.f, b = 0.f;
    FB_CUDA(cudaEventElapsedTime(&a, P.ev[0], P.ev[2]));
    FB_CUDA(cudaEventElapsedTime(&b, P.ev[1], P.ev[2]));
    if (total_ms) *total_ms = a;
    if (construct_ms) *construct_ms = b;
    return FAMSA_OK;
}

void prof_release_all(famsa_ctx* ctx)
{
    ProfState& P = ctx->prof;
    cudaStreamSynchronize(ctx->stream);
    P.arena.release_all();
    for (DevBuf* b : {&P.d_sm, &P.d_widths}) b->release();
    for (cudaEvent_t e : P.free_events) cudaEventDestroy(e);
    if (P.h_ring_mem) cudaFreeHost(P.h_ring_mem);
    if (P.h_done) cudaFreeHost(const_cast<unsigned long long*>(P.h_done));
    P.d_block_counter.release();
    P.d_ring_mem.release();
    if (P.h_tree_results) cudaFreeHost(P.h_tree_results);
    if (P.h_tree_paths) cudaFreeHost(P.h_tree_paths);
    for (auto& e : P.ev)
        if (e) cudaEventDestroy(e);
    for (auto& e : P.ev_tree)
        if (e) cudaEventDestroy(e);
    P = ProfState();
}

} // namespace fb
