// Internal context of libfamsa_b200.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/famsa_b200.h"
#include "dp_dev.h"

namespace fb {

void set_error(const std::string& msg);
const char* get_error();

#define FB_CUDA(expr)                                                                        \
    do {                                                                                     \
        cudaError_t err__ = (expr);                                                          \
        if (err__ != cudaSuccess) {                                                          \
            fb::set_error(std::string(#expr) + " failed: " + cudaGetErrorString(err__) +     \
                          " (" __FILE__ ":" + std::to_string(__LINE__) + ")");               \
            return FAMSA_E_CUDA;                                                             \
        }                                                                                    \
    } while (0)

#define FB_TRY(expr)                       \
    do {                                   \
        int rc__ = (expr);                 \
        if (rc__ != FAMSA_OK) return rc__; \
    } while (0)

struct FusedParams;   // prof_dev.cuh

// Simple owning device buffer that only grows.
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);   // returns FAMSA_* code
    void release();
    template <class T> T* as() const { return static_cast<T*>(p); }
};

// One 32-sequence mask group (sequences are grouped in length-descending order).
struct LcsGroupInfo {
    uint32_t nl;          // instantiated limb count of the tile kernel (0 = longer than the tile kernel handles)
    uint64_t blob_word;   // offset (32-bit words) of the group's mask blob
};

struct LcsState {
    uint32_t n = 0;            // sequences
    uint32_t n_groups = 0;     // ceil(n/32)
    bool identity_perm = true; // caller order already length-descending
    uint32_t max_len = 0;
    std::vector<uint32_t> h_perm;      // sorted position -> caller id
    std::vector<uint32_t> h_invperm;   // caller id -> sorted position
    std::vector<uint32_t> h_len_sorted;
    std::vector<LcsGroupInfo> groups;
    std::vector<uint32_t> h_quirky;    // caller ids whose masks contain an all-ones 64-bit word
    std::vector<uint32_t> h_long;      // caller ids longer than the tile kernel handles as mask side
    DevBuf d_perm, d_invperm, d_len_sorted, d_code_off, d_codes, d_blob, d_group_blob;
    DevBuf d_raw_codes, d_raw_off, d_raw_len, d_flags, d_pow075, d_assign_lcs, d_assign, d_mind,
        d_pow075_f64, d_prim_tri, d_prim_side, d_prim_state, d_prim_out, d_prim_sideidx, d_prim_cand,
        d_prim_dtri, d_prim_comp, d_prim_best, d_prim_part;
    // per-call scratch
    DevBuf d_tiles, d_res, d_refpos, d_ids_a, d_ids_b, d_out_stage, d_masks64, d_x64;
    // last-call timing
    float last_total_ms = 0.f, last_main_ms = 0.f;
    uint64_t last_pairs = 0;
    uint64_t last_tiles = 0;                 // tiles launched by the most recent triangle call
    uint64_t tile_configured = 0;            // bit NL-1: k_lcs_tile<NL> has its shared-memory attribute on this device
    std::vector<uint32_t> h_order;           // famsa_lcs_upload_sorted: position in the library's order -> caller index
};

struct DpState {
    DevBuf d_dirs_out, d_tables, d_results, d_path;     // host entry point only; per-call scratch is stream-ordered
    void* h_pinned = nullptr;          // pinned staging buffer of the host entry point
    size_t h_pinned_cap = 0;
    uint64_t last_cells = 0;
    float last_total_ms = 0.f, last_kernel_ms = 0.f;
    // kernel attributes of the fill and fused kernels are set, and the cluster caps probed, on the first DP call
    bool configured = false;
    uint32_t cluster4_cap = 1, duo_cap = 1;   // largest cluster of k_dp_fill<4, true> / k_dp_fill_duo blocks
};

// Profiles kept resident in HBM between the levels of the guide tree (prof.cu).
struct ProfEntry {
    long long* scores = nullptr;   // (width+1) x 32 int64
    int* counters = nullptr;       // (width+1) x 32 int32
    uint32_t width = 0, card = 0;  // pending: width is the upper bound the tables were sized for
    int slab = -1;
    bool live = false;
    bool pending = false;          // produced by a batch the host has not collected yet: the real width lives in d_widths[id]
    uint32_t gen = 0;              // bumped whenever the id is handed out again
};
// One queued batch of merges (prof_launch ... prof_collect)
// In-order ring allocator (offsets only): batches take space when they are queued and give it back when they are
// collected, oldest first -- the stream is a FIFO, so that is the order they finish in.
struct Ring {
    size_t cap = 0, head = 0, tail = 0;
    bool empty = true;
    // returns the offset or (size_t)-1; `need` is rounded up to 256 bytes
    size_t alloc(size_t need)
    {
        need = (need + 255) & ~(size_t)255;
        if (need > cap) return (size_t)-1;
        if (empty) { head = tail = 0; }
        size_t off;
        if (empty || head > tail) {                 // free space: [head, cap) and [0, tail)
            if (head + need <= cap) off = head;
            else if (need <= tail && !empty) off = 0;
            else if (empty) off = 0;
            else return (size_t)-1;
        } else {                                    // head <= tail (wrapped, or full): free space is [head, tail)
            if (head == tail || head + need > tail) return (size_t)-1;
            off = head;
        }
        head = off + need;
        empty = false;
        return off;
    }
    void release_to(size_t pos) { tail = pos; if (tail == head) empty = true; }
    bool fits(size_t need) const { Ring r = *this; return r.alloc(need) != (size_t)-1; }
};

// Host-side sub-allocator over a few large device chunks for the resident profile tables.  Everything that touches a
// profile is ordered on the context's stream, so a block given back when the batch that consumes it is QUEUED may be handed
// to any batch queued later; no allocator call reaches the driver in steady state (a stream-ordered cudaMallocAsync per
// batch turned out to leave the device idle between the batches of a chain-like guide tree).
struct DevArena {
    struct Chunk { char* base; size_t bytes; };
    std::vector<Chunk> chunks;
    std::map<char*, std::pair<size_t, int>> free_by_addr;          // start -> (bytes, chunk)
    std::multimap<size_t, char*> free_by_size;
    size_t chunk_bytes = 256u << 20;
    bool defer = false;                                             // free() only queues (see FusedAccum)
    std::vector<std::pair<void*, size_t>> deferred;
    void flush_deferred() { defer = false; for (auto& d : deferred) free(d.first, d.second); deferred.clear(); }
    void* alloc(size_t n);                                          // nullptr when the device is out of memory
    void free(void* p, size_t n);
    void release_all();
    void erase_size(size_t n, char* p)
    {
        auto r = free_by_size.equal_range(n);
        for (auto it = r.first; it != r.second; ++it)
            if (it->second == p) { free_by_size.erase(it); return; }
    }
};

struct ProfTicket {
    size_t ring_host_end = (size_t)-1, ring_dev_end = (size_t)-1;    // ring positions to release when the batch is collected
    cudaEvent_t done = nullptr;
    unsigned long long done_seq = 0;   // != 0: completion is published in ProfState::h_done instead of an event
    uint32_t n = 0;
    std::vector<uint32_t> merged_ids, merged_gen;
    famsa_dp_result* h_results = nullptr;   // filled by the batch's D2H copy
    uint8_t* h_paths = nullptr;
    uint64_t path_bytes = 0;
    uint64_t cells_bound = 0;
};
struct ProfSlab {
    void* p = nullptr;
    size_t bytes = 0;
    uint32_t live = 0;             // resident profiles still inside
};
struct ProfState {
    std::vector<ProfEntry> entries;
    std::vector<uint32_t> free_ids;
    std::vector<ProfSlab> slabs;
    std::vector<int> free_slabs;
    bool has_scoring = false, pool_ready = false;
    DevBuf d_sm, d_widths;         // d_widths[id]: width of a pending profile, written by the fill kernel
    // small batches (the fused one-block-per-merge path): job descriptors live in mapped pinned host memory that the kernel
    // reads directly, scratch comes from a device ring -- no copy-engine operation and no allocator call per batch
    DevArena arena;                 // storage of the resident profiles
    volatile unsigned long long* h_done = nullptr;   // mapped host word: sequence number of the last finished flag-tracked batch
    unsigned long long done_seq = 0;
    DevBuf d_block_counter;
    unsigned char* h_ring_mem = nullptr; Ring h_ring;
    DevBuf d_ring_mem; Ring d_ring;
    std::vector<cudaEvent_t> free_events;
    // result of the most recent famsa_prof_align_tree (pinned): per-merge records and all paths
    famsa_dp_result* h_tree_results = nullptr; size_t h_tree_results_cap = 0;
    uint8_t* h_tree_paths = nullptr; size_t h_tree_paths_cap = 0; uint64_t tree_path_bytes = 0; uint32_t tree_merges = 0;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_tree[2] = {nullptr, nullptr};
    uint64_t resident_bytes = 0, n_live = 0;
    bool timing_valid = false;
};

} // namespace fb

struct famsa_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;                 // D2H of finished row blocks (famsa_lcs_triangle)
    cudaEvent_t ev_block[8] = {};
    cudaEvent_t ev_copy[4] = {};                        // end of the peer copies of famsa_lcs_triangle_exchange, per copy stream
    cudaStream_t peer_stream[3] = {};                   // further copy streams: the peers of a piece are served side by side
    cudaEvent_t ev_host[2] = {};
    // The context-owned scratch (tile lists, DP scratch, ...) is shared by every call.  A *_device call on a caller
    // stream returns while its kernels are still queued, so it leaves `ev_busy` recorded behind them and the next call
    // (on whatever stream) waits for it before it touches the scratch again.
    cudaEvent_t ev_busy = nullptr;
    bool busy = false;
    // fill launches of different shapes (cluster sizes) of one batch run side by side on these
    cudaStream_t aux_stream[4] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[4] = {};
    std::mutex mu;
    uint64_t launches = 0;
    int sm_count = 0;
    fb::LcsState lcs;
    fb::DpState dp;
    fb::ProfState prof;
};

namespace fb {
// capi.cu: ordering of calls that share the context's scratch
int scratch_acquire(famsa_ctx* ctx, cudaStream_t st);   // call before queueing work that uses the scratch on `st`
int scratch_release(famsa_ctx* ctx, cudaStream_t st, bool synced);   // call after queueing (synced: the stream was synchronised)
// lcs.cu
int lcs_upload(famsa_ctx* ctx, const int8_t* codes, const uint64_t* offsets, const uint32_t* lens,
               uint32_t n);
int lcs_triangle(famsa_ctx* ctx, uint32_t row_begin, uint32_t row_end, void* d_out, int elem_bytes,
                 cudaStream_t stream, const uint32_t* bounds = nullptr, int n_blocks = 1,
                 cudaEvent_t* block_events = nullptr, bool quirk_fixups = true, bool piece_streams = false);
int lcs_rows(famsa_ctx* ctx, const uint32_t* d_ref_ids, const uint32_t* h_ref_ids, uint32_t n_ref,
             const uint32_t* d_col_ids, uint32_t n_col, void* d_out, int elem_bytes,
             cudaStream_t stream, uint32_t g_begin = 0, uint32_t g_end = 0xffffffffu);
int lcs_upgma(famsa_ctx* ctx, int kind, int modified, int32_t* h_tree, const void* d_tri_in = nullptr, int tri_eb = 2);
int lcs_assign_shard(famsa_ctx* ctx, const uint32_t* h_seed_ids, uint32_t n_seeds, int kind, uint32_t shard, uint32_t n_shards,
                     long long* d_packed, cudaStream_t st);
int lcs_prim(famsa_ctx* ctx, int kind, int32_t* h_from, int32_t* h_to, double* h_dist, int32_t* h_order);
int lcs_assign(famsa_ctx* ctx, const uint32_t* h_seed_ids, uint32_t n_seeds, int kind, uint32_t* h_assign,
               float* h_mind);
// dp.cu
int dp_run_host(famsa_ctx* ctx, const famsa_dp_job* jobs, uint32_t n, const int64_t gaps[4], famsa_dp_result* results,
                uint8_t* path_buf, uint8_t* dirs_buf);
int dp_check_results(const famsa_dp_result* results, uint32_t n);
// d_meta_out / d_blob_out non-NULL: the per-job DpMeta records stay valid until the caller cudaFreeAsync()s *d_blob_out
int dp_run_device(famsa_ctx* ctx, const famsa_dp_job* jobs, const DpJobExt* ext, uint32_t n, const int64_t gaps[4],
                  famsa_dp_result* d_results, uint8_t* d_path, uint8_t* d_dirs, DpMeta** d_meta_out, void** d_blob_out,
                  cudaStream_t st);
int dp_fused_plan(const famsa_dp_job* jobs, const DpJobExt* ext, uint32_t n, bool align16, DpJobDev* out, DpFusedPlan* plan);
int dp_fused_launch(famsa_ctx* ctx, const DpJobDev* jobs, uint32_t n, const int64_t gaps[4], famsa_dp_result* d_results, uint8_t* d_path,
                    DpMeta* d_meta, uint8_t* d_scratch, uint8_t* d_skew, famsa_dp_result* h_results, uint8_t* h_path,
                    const FusedParams& fused, uint32_t grid, uint64_t cells, bool record_events, cudaStream_t st);
unsigned long long dp_scratch_bytes(uint32_t w1, uint32_t w2);
bool dp_debug();   // FAMSA_DP_DEBUG (development aid, read once per process): launch decisions go to stderr
// prof.cu
int prof_set_scoring(famsa_ctx* ctx, const int64_t* sm);
int prof_put(famsa_ctx* ctx, const famsa_dp_profile* profs, uint32_t n, uint32_t* ids);
int prof_merge_batch(famsa_ctx* ctx, const famsa_prof_merge* merges, uint32_t n, const int64_t gaps[4], uint32_t* merged_ids,
                     famsa_dp_result* results, uint8_t* path_buf, uint64_t path_cap);
int prof_get(famsa_ctx* ctx, uint32_t id, uint32_t* width, uint32_t* card, int64_t* scores, int32_t* counters);
int prof_drop(famsa_ctx* ctx, const uint32_t* ids, uint32_t n);
int prof_last_timing(famsa_ctx* ctx, float* total_ms, float* construct_ms);
int prof_align_tree(famsa_ctx* ctx, const int32_t* tree, uint32_t n_leaves, const int64_t gaps[4], famsa_dp_result* results,
                    uint32_t* root_id, uint64_t* path_bytes, famsa_tree_stats* stats);
int prof_tree_paths(famsa_ctx* ctx, uint8_t* path_buf, uint64_t cap);
void prof_release_all(famsa_ctx* ctx);
} // namespace fb
