// libyue_b200.so -- C ABI over the sm_100a kernels (include/yue_b200.h documents each entry
// point and the reference code it replaces).  No torch types here; the Python host side binds
// this with ctypes (yue_b200/_lib.py).
#include "../../include/yue_b200.h"

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <functional>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "bpr_sgd.cuh"
#include "bpr_sgd_blk.cuh"
#include "ingest.cuh"
#include "rank_exact.cuh"
#include "rank_metrics.cuh"
#include "rank_tc.cuh"
#include "wrmf_als.cuh"
#include "cune_sgd.cuh"
#include "lightgcn.cuh"
#include "bpr_adam.cuh"

using namespace yue;

namespace {

thread_local std::string g_create_error;

// ---- NCCL, resolved at run time so the library has no link-time dependency ----------------
struct NcclUniqueId { char internal[128]; };
typedef void* ncclComm_t;
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(NcclUniqueId*) = nullptr;
    int (*CommInitRank)(ncclComm_t*, int, NcclUniqueId, int) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool load(std::string& err) {
        if (lib) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) { lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
        if (!lib) { err = std::string("dlopen libnccl.so.2 failed: ") + dlerror(); return false; }
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy) {
            err = "libnccl is missing a required symbol";
            return false;
        }
        return true;
    }
};
NcclApi g_nccl;

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    cudaError_t resize(size_t count) {
        if (count <= n && p) return cudaSuccess;
        release();
        cudaError_t e = cudaMalloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) n = count; else p = nullptr;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

// pinned host staging that lives as long as the handle: no page faults and full-speed DMA on reuse
template <typename T>
struct PinBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t count) {
        if (count <= cap && p) return cudaSuccess;
        release();
        cudaError_t e = cudaHostAlloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T), cudaHostAllocDefault);
        if (e == cudaSuccess) cap = count; else p = nullptr;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

}  // namespace

struct yue_handle {
    int device = 0;
    int sm_count = 148;
    // Warps per SM that take work (one resident CTA per SM, a single wave).  Blocked kernel at config C2
    // (profiles/quality_study_r1.md section D): 8 warps 13.6 ms, 10 warps 13.6 ms, 12 warps 12.6 ms per epoch, Recall@10 /
    // NDCG@10 within 3e-4 / 3e-3 of the serial order in every run at all three (12 = the kernel's launch bound).
    int warps_per_sm = 12;
    // Small logs get fewer warps.  tools/quality_study.py: at >= 16 K events per warp (what config
    // C2 has on a full B200) the sliding-window schedule reproduces the serial model's Recall/NDCG to
    // 1e-4; at <= 4 K events per warp heavy-user items become stragglers, light users finish long
    // before the heavy ones (the opposite of the serial order) and Recall@10 drops by 2-8 points.
    int min_events_per_warp = 16384;
    int item_segs_env = 0;            // experiments: YUE_SGD_ITEM_SEGS overrides the heavy-user item size
    int seg_events = 32;              // experiments: YUE_SGD_SEG_EVENTS (<= 32) events between P[u] resyncs
    int max_items_per_user = 1 << 30; // YUE_SGD_MAX_ITEMS (experiments): cap on the items of one heavy user
    // Shared (multi-item) users publish and re-read P[u] every resync_events events.  At config C2 the
    // heaviest user is worked on by ~100 warps at once: with 32 events between publishes their summed
    // stale deltas inflate the epoch loss 1.7-2.5x; with <= 16 the loss is within 0.3 % of the serial
    // order and 8 reproduces its Recall@10 / NDCG@10 (profiles/quality_study_r1.md).
    int resync_events = 8;
    // Hot tracks (see SgdParams): a track is hot when it is the positive of >= hot_min_count events AND of
    // more than 1/hot_div of all events; it gets min(cap, pow2ceil(share * hot_div)) accumulator shards, so
    // the chain of dependent atomics on one address stays below ~T/hot_div updates (~11 ns each).
    int hot_max = 24;                 // one GPU: the table relieves L2 slices, a few rows do (YUE_SGD_HOT_MAX, up to kHotSlots)
    int hot_min_count = 16384;
    // Where the hot-row table starts inside its allocation, in 256-byte granules.  Which L2 slices the table's
    // sectors share with each other and with the rest of the working set depends on physical addresses the
    // library cannot see: the same epoch measured 12.6 to 15.5 ms at config C2 depending on nothing but where
    // the buffers happened to land (profiles/microbench/README.md).  So the placement is MEASURED: the first
    // Hogwild launch on a log times 1/32 of the epoch with lr = 0 (state untouched) for kHotCandidates offsets
    // and keeps the fastest; the choice is remembered while the table and the hot set stay the same.
    int hot_offset_granules = 0;
    int hot_offset_forced = -1;       // YUE_HOT_OFFSET_GRANULES (experiments): >= 0 disables the calibration
    uint64_t hot_calibrated_key = 0;
    std::vector<float> hot_calibration_ms;   // per candidate, of the last calibration (diagnostics)
    int hot_div = 128;
    int hot_shard_div = 40;           // blocked kernel: a track played by more than 1/hot_shard_div of the events gets two rows
    int n_hot = 0;
    std::vector<int32_t> h_hot_counts, h_hot_items;   // per hot slot
    int hot_meta_cap = 0, hot_meta_ld = 0;   // what the current hot_meta / hot_shards were built for
    int64_t hot_extra_rows = 0;
    int sgd_kernel = 2;               // YUE_SGD_KERNEL: 1 = per-triplet kernel, 2 = blocked kernel where it applies
    DevBuf<int32_t> hot_items, hot_slot, item_counts, hot_meta, hot_sorted, hot_sorted_slot, hot_dx;
    DevBuf<float> hot_shards, hotQ;
    size_t l2_bytes = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    int64_t launches = 0;

    // play log (local shard)
    int64_t m = 0, n = 0, T = 0, nnz = 0, user_begin = 0, event_base = 0;
    bool have_log = false;
    DevBuf<int64_t> ev_indptr, uq_indptr, ev_delta;
    bool have_ev_delta = false;
    DevBuf<int32_t> ev_items, uq_items, ev_user;
    bool have_ev_user = false;
    std::vector<int64_t> h_ev_indptr;
    // segments of the epoch kernels
    int64_t nseg = 0;
    int n_warps = 0;
    DevBuf<int64_t> item_ptr;
    int64_t n_items = 0;
    DevBuf<unsigned long long> cursor;
    DevBuf<SegRec> seg_rec, tmp_rec;
    PinBuf<SegRec> pin_rec;          // host staging of the segment records and item ranges
    PinBuf<int64_t> pin_items;
    std::vector<int64_t> h_uq_indptr;
    // Light users per work item: consecutive users until this many segments (YUE_SGD_GROUP_SEGS).  Measured at C2
    // (profiles/quality_raw/quality_study_r1t.txt): 8 is 2 % faster but Recall@10 scatters 0.094-0.099 between runs;
    // one user per item reproduces the serial order (0.0978-0.0981 in every run).
    int item_group_segs = 1;

    // factors
    int k = 0, ld = 0;
    bool have_factors = false;
    DevBuf<float> P, Q, Qsnap, Qdelta, delta_w;
    bool have_delta_w = false;
    // interleaved working copy of Q for the SGD kernels (d = 64); exactly one of the two is current
    DevBuf<float> Qilv;
    bool use_ilv = false, ilv_current = false, rowmajor_current = true;   // measured: no gain (the limit is per address, not per slice)
    bool have_snap = false;
    DevBuf<double> scal;          // [0] loss, [1] |P|^2, [2] |Q|^2

    // scratch
    DevBuf<int32_t> tmp_i, tmp_j, rk_users, rk_ids, rk_part_ids;
    DevBuf<int64_t> tmp_ws;
    DevBuf<float> rk_scores, pred, rk_part_scores;
    DevBuf<unsigned char> l2buf;
    RankTcState tc;
    // ranking metrics (K6)
    int64_t last_rank_B = 0; int last_rank_N = 0;
    bool have_test = false;
    int64_t n_test = 0;
    DevBuf<int64_t> test_indptr;
    DevBuf<int32_t> test_items;
    DevBuf<double> met_terms, met_sums;
    DevBuf<uint32_t> met_seen;
    DevBuf<unsigned long long> met_distinct;

    // WRMF (K7): plays per unique pair, the track-major form of the play sets, heavy-row chunk plans per side
    bool wrmf_ready = false;
    DevBuf<int32_t> uq_cnt, it_users, it_cnt;
    DevBuf<int64_t> it_indptr;
    struct WrmfPlan {
        DevBuf<int32_t> heavy_rows, heavy_first, chunk_row;
        DevBuf<int64_t> chunk_begin, chunk_end;
        int n_heavy = 0, n_chunks = 0;
        std::vector<int32_t> h_chunk_row;       // host copy: which chunks belong to a row range
    } wrmf_plan[2];
    DevBuf<double> wrmf_G, wrmf_part, wrmf_partA, wrmf_partb, wrmf_Binv;
    // Rows with 1..16 entries go through the d x d Woodbury kernel (wrmf_light_kernel, one warp per row): 2.9x faster per
    // row than the k x k factorisation at d = 64 (profiles/ncu_wrmf_r1.md).  YUE_WRMF_LIGHT=0 sends every row through the
    // factorisation (tests compare the two).
    int wrmf_light = 1;
    // 32 < k <= 64: 16 x 16 grid of 4 x 4 blocks on 160 threads (0, default) or 8 x 8 grid of 8 x 8 blocks on 64 threads
    // (YUE_WRMF_FAT=1; measured slower at config C2: 76 / 34 ms per user / track sweep against 64 / 27)
    int wrmf_fat = 0;

    // CUNE (K8): implicit positives per user (tracks of the user's top-K similar users it has not played, CUNE.py:95-113)
    bool have_ip = false;
    DevBuf<int64_t> ip_indptr;
    DevBuf<int32_t> ip_items;
    DevBuf<double> cune_scal;                 // [0] loss of the epoch
    DevBuf<int64_t> cune_items;               // work items of the epoch kernel (cune_plan_items)
    int64_t cune_n_work = 0, cune_chunk = -1; // -1: no plan for the current log
    DevBuf<unsigned long long> cune_ctr;      // [0] user cursor, [1] users with events


    // LightGCN (K9): the training events in FILE order (batches are slices of it), row lists of the product phases, the
    // layers, the backward buffers, Adam's moments and the batch scratch
    bool gcn_events = false, gcn_planned = false, gcn_final = false;
    DevBuf<int32_t> gcn_ev_user, gcn_ev_item, gcn_neg, gcn_slot_row, gcn_slot_of;
    DevBuf<int2> gcn_segs;
    DevBuf<GcnChunk> gcn_chunks;
    DevBuf<unsigned> gcn_arrived;
    DevBuf<unsigned long long> gcn_phase_ns;
    DevBuf<uint32_t> gcn_stamp;
    DevBuf<float> gcn_E[kGcnMaxLayers], gcn_rinv, gcn_D[2], gcn_am, gcn_av, gcn_slot_grad, gcn_NB, gcn_trip_loss, gcn_varP, gcn_varQ, gcn_partial;
    DevBuf<double> gcn_loss;
    std::vector<int64_t> h_it_indptr;
    int64_t gcn_n_chunk = 0, gcn_n_seg = 0, gcn_t = 0;
    uint32_t gcn_stamp_base = 0;

    // BPR's shipped Adam training (K10): Adam's moments (separate from K9's), the step counter, the per-step scratch
    DevBuf<float> ba_am, ba_av, ba_trip_c, ba_trip_loss, ba_ucopy, ba_ugrad, ba_row_c;
    DevBuf<int32_t> ba_fix, ba_row_u, ba_row_i, ba_row_e, ba_trip_j, ba_slot_row, ba_slot_pos, ba_list, ba_sorted, ba_cnt, ba_row_base, ba_row_size;
    DevBuf<uint32_t> ba_stamp;
    DevBuf<unsigned> ba_bump;
    DevBuf<double> ba_row_loss, ba_loss;
    int64_t ba_t = 0;
    uint32_t ba_tag = 0;

    ncclComm_t comm = nullptr;
    int nranks = 1, rank = 0;

    // multi-GPU, shared hot rows (yue_hot_share) and the overlapped exchange of the tail (yue_q_exchange_*)
    bool hot_shared = false;
    bool hot_stale = false;                   // a shared epoch trained the owners' rows: Q's copies wait for yue_hot_pull
    int hot_nranks = 1, hot_rank = 0;
    DevBuf<unsigned long long> hot_base;      // [n_hot] this process's address of the table that owns each slot
    std::vector<void*> ipc_opened;            // peer tables mapped by yue_hot_table_open ...
    std::vector<std::string> ipc_keys;        // ... and the 64-byte handle each came from (a handle is opened once per process)
    DevBuf<float> Qown;                       // this rank's packed delta while the sum is in flight
    DevBuf<float> Qsum;                       // yue_q_exchange_reduce_peers: the sum (the ranks' deltas must stay readable)
    bool sum_in_qsum = false;
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_pack = nullptr, ev_red = nullptr;
    bool exchange_pending = false;
    int sgd_warps_forced = 0, sgd_ctas_forced = 0;   // yue_set_sgd_concurrency
};

#define CK(...)                                                                           \
    do {                                                                                  \
        cudaError_t e_ = (__VA_ARGS__);                                                   \
        if (e_ != cudaSuccess) {                                                          \
            h->err = std::string(#__VA_ARGS__) + ": " + cudaGetErrorString(e_);           \
            return YUE_E_CUDA;                                                            \
        }                                                                                 \
    } while (0)

#define REQUIRE(cond, code, msg)            \
    do {                                    \
        if (!(cond)) { h->err = (msg); return (code); } \
    } while (0)

static int fail(yue_t* h, int code, const std::string& msg) { h->err = msg; return code; }

// YUE_TIMING=1: wall-clock of the phases of yue_set_interactions on stderr (diagnostics)
struct PhaseTimer {
    bool on; std::chrono::steady_clock::time_point t0;
    PhaseTimer() : on(getenv("YUE_TIMING") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void lap(const char* what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[yue timing] %-28s %7.2f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};
static int q_rowmajor(yue_t* h);
static int q_interleaved(yue_t* h);

// Cut every user's event range into <=32-event segments (one SegRec each) and group them into work
// items, returned as [begin, end) segment ranges in STREAM ORDER (the order the kernel's cursor hands
// them out and the order the reference visits users in, recommender/cf/BPR.py:42):
//   * consecutive light users share an item until it holds group_segs segments: the cursor atomic,
//     the item lookup and the cold start of the kernel's prefetch pipeline are paid once per item;
//   * a heavy user (more than item_segs segments) is cut into items of item_segs segments (a quarter
//     of a warp's fair share of the epoch), all at the user's stream position; its segments are flagged
//     kSegShared and the warps working on it publish and re-read P[u] every few events.
// What the measurements at config C2 say (tools/quality_study.py, profiles/quality_study_r1.md):
// a heavy user has to FINISH EARLY, like in the serial order -- big items make it a straggler, every
// light user's P[u] is then stale against the large Q changes it keeps making and Recall@10 drops
// from 0.098 to 0.005; spreading its items over the epoch does the same (0.17 -> 0.04 at 5 M events).
// So ~100 warps must share the heaviest user, and the staleness of P[u] is bounded by resync_events.
// A run r is the event range [begin(r), end(r)) of user(r); runs are independent, so the host cores
// split them (an item never spans two threads' shares).
struct ItemPlanArgs {
    bool allow_shared; int64_t item_segs, max_items, group_segs; int seg_events; const int64_t* uq_indptr;
};
// host threads a handle may use for planning: the cores divided by the processes that share the box
// (LOCAL_WORLD_SIZE is set by torchrun: one process per GPU), at most 4 -- the planner writes pinned staging while the
// DMA of the log reads pinned memory, and more writers slow that DMA down by more than they shorten the plan (config C2,
// 16 cores: 16 threads plan in 4.5 ms and yue_set_interactions takes 12.7 ms; 4 threads plan in 6.7 ms and it takes 10.5)
static size_t host_threads() {
    size_t hw = std::max(1u, std::thread::hardware_concurrency());
    if (const char* s = getenv("LOCAL_WORLD_SIZE")) hw = std::max<size_t>(1, hw / (size_t)std::max(1, atoi(s)));
    size_t cap = 4;
    if (const char* s = getenv("YUE_HOST_THREADS")) cap = (size_t)std::max(1, atoi(s));
    return std::min<size_t>(cap, hw);
}

// one pass over runs [r0, r1): WRITE = false only counts segments and items, WRITE = true fills
// rec[seg0...] and item_rng[2 * item0 ...]
template <bool WRITE, class RunFn>
static void plan_runs(size_t r0, size_t r1, RunFn run, const ItemPlanArgs& a, SegRec* rec, int64_t* item_rng,
                      int64_t seg0, int64_t item0, int64_t& nseg_out, int64_t& nitem_out) {
    int64_t s = seg0, it = item0, open_first = -1;
    auto emit = [&](int64_t b, int64_t e) { if (WRITE) { item_rng[2 * it] = b; item_rng[2 * it + 1] = e; } ++it; };
    auto close_open = [&]() { if (open_first >= 0) { emit(open_first, s); open_first = -1; } };
    for (size_t r = r0; r < r1; ++r) {
        int64_t b, e; int32_t u;
        run(r, b, e, u);
        const int64_t nsegs = (e - b + a.seg_events - 1) / a.seg_events;
        if (nsegs == 0) continue;
        const bool heavy = nsegs > a.item_segs && a.allow_shared;
        if (heavy) close_open();
        const int64_t first = s;
        if (WRITE) {
            const int64_t row0 = a.uq_indptr[u];
            const int32_t row_len = (int32_t)(a.uq_indptr[u + 1] - row0), flag = heavy ? kSegShared : 0;
            for (; b < e; b += a.seg_events, ++s) {
                SegRec& x = rec[s];
                x.user = u; x.len_flags = (int32_t)std::min<int64_t>(a.seg_events, e - b) | flag; x.begin = b;
                x.row_begin = row0; x.row_len = row_len; x.shared = flag;
            }
        } else {
            s += nsegs;
        }
        if (heavy) {
            const int64_t per = std::max(a.item_segs, (nsegs + a.max_items - 1) / a.max_items);
            for (int64_t i = first; i < s; i += per) emit(i, std::min(s, i + per));
        } else {
            if (open_first < 0) open_first = first;
            if (s - open_first >= a.group_segs) close_open();
        }
    }
    close_open();
    nseg_out = s - seg0; nitem_out = it - item0;
}
// plans all runs on the host cores (an item never spans two threads' shares); the buffers are (re)allocated
template <class RunFn>
static cudaError_t plan_items(size_t nruns, RunFn run, const ItemPlanArgs& a, PinBuf<SegRec>& rec_buf, PinBuf<int64_t>& item_buf,
                              int64_t& nseg, int64_t& nitems) {
    const size_t nthreads = nruns < 65536 ? 1 : host_threads();
    std::vector<int64_t> segs(nthreads), its(nthreads), seg_first(nthreads + 1, 0), item_first(nthreads + 1, 0);
    auto share = [&](size_t t) { return nruns * t / nthreads; };
    auto parallel = [&](auto fn) {
        std::vector<std::thread> th;
        for (size_t t = 1; t < nthreads; ++t) th.emplace_back(fn, t);
        fn(0);
        for (auto& x : th) x.join();
    };
    parallel([&](size_t t) { plan_runs<false>(share(t), share(t + 1), run, a, nullptr, nullptr, 0, 0, segs[t], its[t]); });
    for (size_t t = 0; t < nthreads; ++t) { seg_first[t + 1] = seg_first[t] + segs[t]; item_first[t + 1] = item_first[t] + its[t]; }
    nseg = seg_first[nthreads]; nitems = item_first[nthreads];
    cudaError_t e = rec_buf.ensure((size_t)nseg);
    if (e == cudaSuccess) e = item_buf.ensure((size_t)nitems * 2);
    if (e != cudaSuccess) return e;
    parallel([&](size_t t) {
        int64_t x, y;
        plan_runs<true>(share(t), share(t + 1), run, a, rec_buf.p, item_buf.p, seg_first[t], item_first[t], x, y);
    });
    return cudaSuccess;
}

// Every yue_* function below is declared extern "C" by include/yue_b200.h and inherits that linkage.

const char* yue_version(void) { return "yue_b200 0.1 (sm_100a)"; }

const char* yue_last_error(const yue_t* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int yue_create(int device, yue_t** out) {
    if (!out) { g_create_error = "out is NULL"; return YUE_E_ARG; }
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
        return YUE_E_CUDA;
    }
    if (device < 0 || device >= count) { g_create_error = "device index out of range"; return YUE_E_ARG; }
    yue_t* h = new yue_handle();
    h->device = device;
    cudaDeviceProp prop;
    auto release = [&]() {                       // error paths: nothing created so far may outlive the handle
        if (h->ev0) cudaEventDestroy(h->ev0);
        if (h->ev1) cudaEventDestroy(h->ev1);
        h->scal.release();
        if (h->stream) cudaStreamDestroy(h->stream);
        delete h;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreate(&h->ev0)) != cudaSuccess || (e = cudaEventCreate(&h->ev1)) != cudaSuccess ||
        (e = h->scal.resize(4)) != cudaSuccess) {
        g_create_error = std::string("device setup failed: ") + cudaGetErrorString(e);
        release();
        return YUE_E_CUDA;
    }
    if (prop.major < 10) {
        g_create_error = "yue_b200 needs an sm_100a device (B200); found sm_" + std::to_string(prop.major * 10 + prop.minor);
        release();
        return YUE_E_UNSUPPORTED;
    }
    h->sm_count = prop.multiProcessorCount;
    h->l2_bytes = (size_t)prop.l2CacheSize;
    if (const char* s = getenv("YUE_HOT_OFFSET_GRANULES")) h->hot_offset_forced = std::max(0, std::min(kHotCandidates * kHotCandidateStep, atoi(s)));
    if (const char* s = getenv("YUE_SGD_HOT_MAX")) h->hot_max = std::max(0, std::min(kHotSlots, atoi(s)));
    if (const char* s = getenv("YUE_SGD_HOT_MIN_COUNT")) h->hot_min_count = std::max(1, atoi(s));
    if (const char* s = getenv("YUE_SGD_HOT_DIV")) h->hot_div = std::max(1, atoi(s));
    if (const char* s = getenv("YUE_SGD_HOT_SHARD_DIV")) h->hot_shard_div = std::max(1, atoi(s));
    if (const char* s = getenv("YUE_SGD_GROUP_SEGS")) h->item_group_segs = std::max(1, atoi(s));
    if (const char* s = getenv("YUE_WRMF_LIGHT")) h->wrmf_light = atoi(s) != 0;
    if (const char* s = getenv("YUE_WRMF_FAT")) h->wrmf_fat = atoi(s) != 0;
    if (const char* s = getenv("YUE_SGD_KERNEL")) h->sgd_kernel = atoi(s) == 1 ? 1 : 2;
    if (const char* s = getenv("YUE_SGD_ITEM_SEGS")) h->item_segs_env = std::max(0, atoi(s));   // 0 = automatic
    if (const char* s = getenv("YUE_SGD_MAX_ITEMS")) h->max_items_per_user = std::max(1, atoi(s));
    if (const char* s = getenv("YUE_SGD_Q_INTERLEAVE")) h->use_ilv = atoi(s) != 0;
    if (const char* s = getenv("YUE_SGD_RESYNC_EVENTS")) h->resync_events = std::max(1, std::min(32, atoi(s)));
    if (const char* s = getenv("YUE_SGD_SEG_EVENTS")) h->seg_events = std::max(1, std::min(32, atoi(s)));
    if (const char* s = getenv("YUE_SGD_WARPS_PER_SM")) h->warps_per_sm = std::max(1, std::min(kSgdThreads / 32, atoi(s)));
    if (const char* s = getenv("YUE_SGD_MIN_EVENTS_PER_WARP")) h->min_events_per_warp = std::max(32, atoi(s));
    *out = h;
    return YUE_OK;
}

int yue_destroy(yue_t* h) {
    if (!h) return YUE_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    rank_tc_release(h->tc);
    for (auto* b : {&h->ev_indptr, &h->uq_indptr, &h->ev_delta, &h->item_ptr, &h->tmp_ws}) b->release();
    h->seg_rec.release(); h->tmp_rec.release(); h->pin_rec.release(); h->pin_items.release();
    h->cursor.release();
    for (auto* b : {&h->ev_items, &h->uq_items, &h->ev_user, &h->tmp_i, &h->tmp_j, &h->rk_part_ids, &h->rk_users, &h->rk_ids, &h->hot_items, &h->hot_slot, &h->item_counts, &h->hot_meta, &h->hot_sorted, &h->hot_sorted_slot, &h->hot_dx}) b->release();
    for (auto* b : {&h->P, &h->Q, &h->Qsnap, &h->Qdelta, &h->delta_w, &h->Qilv, &h->rk_scores, &h->pred, &h->rk_part_scores, &h->hot_shards, &h->hotQ}) b->release();
    h->scal.release();
    h->ip_indptr.release(); h->ip_items.release(); h->cune_scal.release(); h->cune_ctr.release(); h->cune_items.release();
    h->l2buf.release();
    for (auto* b : {&h->gcn_ev_user, &h->gcn_ev_item, &h->gcn_neg, &h->gcn_slot_row, &h->gcn_slot_of}) b->release();
    h->gcn_segs.release(); h->gcn_chunks.release(); h->gcn_arrived.release(); h->gcn_phase_ns.release();
    for (auto* b : {&h->gcn_E[0], &h->gcn_E[1], &h->gcn_E[2], &h->gcn_E[3], &h->gcn_rinv, &h->gcn_D[0], &h->gcn_D[1], &h->gcn_am, &h->gcn_av, &h->gcn_slot_grad, &h->gcn_NB, &h->gcn_trip_loss, &h->gcn_varP, &h->gcn_varQ, &h->gcn_partial}) b->release();
    h->gcn_stamp.release(); h->gcn_loss.release();
    for (auto* b : {&h->ba_am, &h->ba_av, &h->ba_trip_c, &h->ba_trip_loss, &h->ba_ucopy, &h->ba_ugrad, &h->ba_row_c}) b->release();
    for (auto* b : {&h->ba_fix, &h->ba_row_u, &h->ba_row_i, &h->ba_row_e, &h->ba_trip_j, &h->ba_slot_row, &h->ba_slot_pos, &h->ba_list, &h->ba_sorted, &h->ba_cnt, &h->ba_row_base, &h->ba_row_size}) b->release();
    h->ba_stamp.release(); h->ba_bump.release(); h->ba_row_loss.release(); h->ba_loss.release();
    h->hot_base.release(); h->Qown.release(); h->Qsum.release();
    for (void* p : h->ipc_opened) cudaIpcCloseMemHandle(p);
    if (h->ev_pack) cudaEventDestroy(h->ev_pack);
    if (h->ev_red) cudaEventDestroy(h->ev_red);
    if (h->stream2) { cudaStreamSynchronize(h->stream2); cudaStreamDestroy(h->stream2); }
    h->uq_cnt.release(); h->it_users.release(); h->it_cnt.release(); h->it_indptr.release();
    for (auto* b : {&h->wrmf_G, &h->wrmf_part, &h->wrmf_partA, &h->wrmf_partb, &h->wrmf_Binv}) b->release();
    for (auto& pl : h->wrmf_plan) { pl.heavy_rows.release(); pl.heavy_first.release(); pl.chunk_row.release(); pl.chunk_begin.release(); pl.chunk_end.release(); }
    h->test_indptr.release(); h->test_items.release(); h->met_terms.release(); h->met_sums.release(); h->met_seen.release(); h->met_distinct.release();
    cudaEventDestroy(h->ev0);
    cudaEventDestroy(h->ev1);
    cudaStreamDestroy(h->stream);
    delete h;
    return YUE_OK;
}

int yue_device_count(int* count) {
    if (!count) return YUE_E_ARG;
    *count = 0;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return YUE_OK; }   // no driver / no device: 0
    *count = n;
    return YUE_OK;
}

int yue_sync(yue_t* h) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

int yue_host_alloc(size_t bytes, void** out) {
    if (!out) return YUE_E_ARG;
    return cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocDefault) == cudaSuccess ? YUE_OK : YUE_E_CUDA;
}
int yue_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? YUE_OK : YUE_E_CUDA; }

// Make `cand` (slot order) the hot set: lookup tables for the kernels, second rows for tracks above 1/hot_shard_div of
// `total` events, and the hot positives of the device copy of ev_items re-labelled -slot-1 (ev_items must be unmarked).
static int install_hot_set(yue_t* h, const std::vector<int32_t>& cand, const std::vector<int64_t>& cand_counts, int64_t total) {
    const int64_t n = h->n, T = h->T;
    h->n_hot = (int)cand.size();
    h->h_hot_counts.clear();
    for (int64_t c : cand_counts) h->h_hot_counts.push_back((int32_t)std::min<int64_t>(c, INT32_MAX));
    h->h_hot_items = cand;
    h->hot_meta_cap = 0;
    if (!h->n_hot) return YUE_OK;
    std::vector<int32_t> slot((size_t)n, -1);
    for (int s2 = 0; s2 < h->n_hot; ++s2) slot[cand[s2]] = s2;
    std::vector<int32_t> order((size_t)h->n_hot), sorted_ids, sorted_slots;      // ascending track id, for the kernel's lookup of negatives
    for (int s2 = 0; s2 < h->n_hot; ++s2) order[s2] = s2;
    std::sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return cand[a] < cand[b]; });
    for (int32_t s2 : order) { sorted_ids.push_back(cand[s2]); sorted_slots.push_back(s2); }
    std::vector<int32_t> dx((size_t)h->n_hot, 0);       // second rows for the most played tracks (blocked kernel)
    for (int s2 = 0, extra = 0; s2 < h->n_hot && extra < kHotExtra; ++s2)
        if (cand_counts[s2] * h->hot_shard_div > total) {
            dx[s2] = (int32_t)((hot_slot_offset(h->n_hot + extra) - hot_slot_offset(s2)) * sizeof(float));
            ++extra;
        }
    CK(h->hot_dx.resize(h->n_hot));
    CK(cudaMemcpyAsync(h->hot_dx.p, dx.data(), dx.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(h->hot_sorted.resize(h->n_hot)); CK(h->hot_sorted_slot.resize(h->n_hot)); CK(h->hotQ.resize(kHotTableFloats + (size_t)(kHotCandidates + 1) * kHotCandidateStep * 64));
    CK(cudaMemcpyAsync(h->hot_sorted.p, sorted_ids.data(), sorted_ids.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->hot_sorted_slot.p, sorted_slots.data(), sorted_slots.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(h->hot_items.resize(h->n_hot)); CK(h->hot_slot.resize(n));
    CK(cudaMemcpyAsync(h->hot_items.p, cand.data(), cand.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->hot_slot.p, slot.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    if (T > 0) {
        const int grid = (int)std::min<int64_t>((T + 255) / 256, (int64_t)h->sm_count * 16);
        mark_hot_kernel<<<grid, 256, 0, h->stream>>>(h->ev_items.p, T, h->hot_slot.p);
        ++h->launches;
        CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(h->stream));      // host vectors die here
    return YUE_OK;
}

// second half of yue_set_interactions / yue_ingest_events: the four arrays are on the device (h->m, n, T, nnz set),
// ev_indptr / uq_indptr are their host copies.  Validates, plans segments and work items, selects the hot tracks.
static int finish_interactions(yue_t* h, const int64_t* ev_indptr, const int64_t* uq_indptr, bool check_items) {
    const int64_t m_local = h->m, n = h->n, T = h->T;
    PhaseTimer pt;
    {   // validation on the host cores: monotone indptr; a user who played the whole catalog has no negative
        // (the reference would spin forever, BPR.py:47-48)
        const size_t nth = m_local < 65536 ? 1 : host_threads();
        std::vector<int64_t> bad_mono(nth, -1), bad_full(nth, -1);
        auto check = [&](size_t t) {
            for (int64_t u = m_local * (int64_t)t / (int64_t)nth, e = m_local * (int64_t)(t + 1) / (int64_t)nth; u < e; ++u) {
                if (!(ev_indptr[u + 1] >= ev_indptr[u] && uq_indptr[u + 1] >= uq_indptr[u])) { bad_mono[t] = u; return; }
                if (!(uq_indptr[u + 1] - uq_indptr[u] < n || ev_indptr[u + 1] == ev_indptr[u])) { bad_full[t] = u; return; }
            }
        };
        std::vector<std::thread> th;
        for (size_t t = 1; t < nth; ++t) th.emplace_back(check, t);
        check(0);
        for (auto& x : th) x.join();
        for (size_t t = 0; t < nth; ++t) {
            REQUIRE(bad_mono[t] < 0, YUE_E_ARG, "indptr not monotone");
            REQUIRE(bad_full[t] < 0, YUE_E_ARG, "user " + std::to_string(bad_full[t] + h->user_begin) + " played every track: no negative exists");
        }
    }
    h->h_ev_indptr.clear(); h->h_uq_indptr.clear();       // host copies are fetched back on demand (host_indptrs)
    h->have_ev_user = false;
    h->have_log = false;
    h->have_ev_delta = false;
    h->have_ip = false;                                    // implicit positives belong to the log they were set for
    h->cune_chunk = -1;
    h->gcn_events = false; h->gcn_planned = false; h->gcn_final = false;
    h->last_rank_B = 0;
    pt.lap("validate + host copies");

    // concurrency: at most one resident wave, fewer warps on small logs (bounds Hogwild staleness
    // and keeps the in-flight window a small fraction of the users)
    h->n_warps = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)h->sm_count * h->warps_per_sm, T / h->min_events_per_warp));
    // a heavy user's item is at most a quarter of a warp's fair share, so no item is a straggler
    int64_t item_segs = std::max<int64_t>(32, std::min<int64_t>(256, T / ((int64_t)h->n_warps * 4 * 32)));
    if (h->item_segs_env > 0) item_segs = h->item_segs_env;
    const ItemPlanArgs plan{true, item_segs, h->max_items_per_user, h->item_group_segs, h->seg_events, uq_indptr};
    CK(plan_items((size_t)m_local, [=](size_t r, int64_t& b, int64_t& e, int32_t& u) { b = ev_indptr[r]; e = ev_indptr[r + 1]; u = (int32_t)r; },
                  plan, h->pin_rec, h->pin_items, h->nseg, h->n_items));
    pt.lap("plan segments/items");
    CK(h->seg_rec.resize(h->nseg)); CK(h->item_ptr.resize(2 * h->n_items)); CK(h->cursor.resize(1));
    if (h->nseg) CK(cudaMemcpyAsync(h->seg_rec.p, h->pin_rec.p, h->nseg * sizeof(SegRec), cudaMemcpyHostToDevice, h->stream));
    if (h->n_items) CK(cudaMemcpyAsync(h->item_ptr.p, h->pin_items.p, 2 * h->n_items * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    if (check_items && (T > 0 || h->nnz > 0)) {
        // the caller's arrays (the ingest path has checked and sorted its own): ids inside the catalog, play rows sorted-unique
        int* bad = (int*)(h->scal.p + 3);
        CK(cudaMemsetAsync(bad, 0, sizeof(int), h->stream));
        const int64_t work = std::max(T, h->nnz);
        interaction_check_kernel<<<(int)std::min<int64_t>((work + 255) / 256, (int64_t)h->sm_count * 16), 256, 0, h->stream>>>(
            h->ev_items.p, T, h->uq_indptr.p, h->uq_items.p, h->nnz, m_local, n, bad);
        ++h->launches;
        CK(cudaGetLastError());
        int hbad = 0;
        CK(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        REQUIRE(!(hbad & 1), YUE_E_ARG, "ev_items names a track outside [0, n)");
        REQUIRE(!(hbad & 2), YUE_E_ARG, "uq_items names a track outside [0, n)");
        REQUIRE(!(hbad & 4), YUE_E_ARG, "uq_items rows must be strictly increasing (sorted, unique)");
        pt.lap("wait: uploads + id check");
    }
    // hot tracks: device histogram of the positives, top hot_max by count on the host, then the hot
    // positives of the device copy of ev_items are re-labelled -slot-1 (see SgdParams::hot_items)
    h->n_hot = 0;
    h->h_hot_items.clear();
    h->hot_shared = false;                     // a new log: its hot set is private until yue_hot_share is called again
    h->hot_stale = false;
    if (T > 0 && h->hot_max > 0) {
        CK(h->item_counts.resize(n));
        CK(cudaMemsetAsync(h->item_counts.p, 0, n * sizeof(int32_t), h->stream));
        const int grid = (int)std::min<int64_t>((T + 255) / 256, (int64_t)h->sm_count * 16);
        // every stride-th event is enough to find tracks with > 1/hot_div of the plays, and keeps the atomics on the
        // counters of those very tracks short (all 50 M events of C2: 5 ms, 3.9 M of them on one address)
        const int64_t stride = std::max<int64_t>(1, std::min<int64_t>(64, T >> 20));
        item_count_kernel<<<grid, 256, 0, h->stream>>>(h->ev_items.p, T, stride, h->item_counts.p);
        ++h->launches;
        CK(cudaGetLastError());
        std::vector<int32_t> counts((size_t)n);
        CK(cudaMemcpyAsync(counts.data(), h->item_counts.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        pt.lap("wait: uploads + histogram");
        std::vector<int32_t> cand;
        for (int64_t t = 0; t < n; ++t)
            if ((int64_t)counts[t] * stride >= h->hot_min_count && (int64_t)counts[t] * stride * h->hot_div > T) cand.push_back((int32_t)t);
        std::sort(cand.begin(), cand.end(), [&](int32_t a, int32_t b) { return counts[a] != counts[b] ? counts[a] > counts[b] : a < b; });
        if ((int)cand.size() > h->hot_max) cand.resize(h->hot_max);
        std::vector<int64_t> cand_counts;
        for (int32_t t : cand) cand_counts.push_back((int64_t)counts[t] * stride);
        if (int rc = install_hot_set(h, cand, cand_counts, T)) return rc;
    }
    CK(cudaStreamSynchronize(h->stream));      // host vectors die here
    pt.lap("hot tracks");
    h->have_log = true;
    h->wrmf_ready = false;
    return YUE_OK;
}

int yue_set_interactions_shard(yue_t* h, int64_t m_local, int64_t n, int64_t user_begin, int64_t event_base,
                               const int64_t* ev_indptr, const int32_t* ev_items,
                               const int64_t* uq_indptr, const int32_t* uq_items) {
    REQUIRE(h && ev_indptr && uq_indptr, YUE_E_ARG, "null argument");
    REQUIRE(m_local >= 0 && n > 0 && n < (int64_t)1 << 31 && m_local < (int64_t)1 << 31, YUE_E_ARG, "m/n out of range");
    REQUIRE(ev_indptr[0] == 0 && uq_indptr[0] == 0, YUE_E_ARG, "indptr must start at 0 (rebase shards)");
    const int64_t T = ev_indptr[m_local], nnz = uq_indptr[m_local];
    REQUIRE((T == 0 || ev_items) && (nnz == 0 || uq_items), YUE_E_ARG, "null item array");
    REQUIRE(T >= 0 && nnz >= 0, YUE_E_ARG, "indptr not monotone");
    CK(cudaSetDevice(h->device));
    // from here on the old log is gone: a failure below must not leave its plan behind for the new arrays, and tables
    // sized for another m or n must not be indexed by the new log
    h->have_log = false;
    if (m_local != h->m || n != h->n) h->have_factors = false;
    if (n != h->n) h->have_delta_w = false;   // per-track weights belong to a catalog
    h->m = m_local; h->n = n; h->T = T; h->nnz = nnz; h->user_begin = user_begin; h->event_base = event_base;
    h->have_test = false;              // a new log: the held-out set of the old one no longer applies
    CK(h->ev_indptr.resize(m_local + 1)); CK(h->uq_indptr.resize(m_local + 1));
    CK(h->ev_items.resize(T)); CK(h->uq_items.resize(nnz));
    CK(cudaMemcpyAsync(h->ev_indptr.p, ev_indptr, (m_local + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->uq_indptr.p, uq_indptr, (m_local + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    if (T) CK(cudaMemcpyAsync(h->ev_items.p, ev_items, T * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    if (nnz) CK(cudaMemcpyAsync(h->uq_items.p, uq_items, nnz * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    return finish_interactions(h, ev_indptr, uq_indptr, true);
}

int yue_set_interactions(yue_t* h, int64_t m, int64_t n, const int64_t* ev_indptr, const int32_t* ev_items,
                         const int64_t* uq_indptr, const int32_t* uq_items) {
    return yue_set_interactions_shard(h, m, n, 0, 0, ev_indptr, ev_items, uq_indptr, uq_items);
}


// ---- K0: array form of the play log built on the device (ingest.cuh) --------------------------------
namespace {
struct CubTemp {
    DevBuf<unsigned char> buf;
    cudaError_t ensure(size_t bytes) { return buf.resize(bytes + 256); }
};
}  // namespace

int yue_ingest_events(yue_t* h, int64_t m, int64_t n, int64_t E, const int32_t* ev_user, const int32_t* ev_item,
                      const uint8_t* is_test) {
    REQUIRE(h && (E == 0 || (ev_user && ev_item)), YUE_E_ARG, "null argument");
    REQUIRE(m >= 0 && n > 0 && n < (int64_t)1 << 31 && m < (int64_t)1 << 31 && E >= 0 && E < (int64_t)1 << 31, YUE_E_ARG, "m/n/E out of range");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const size_t Ez = (size_t)std::max<int64_t>(E, 1);
    DevBuf<int32_t> du, di, tu, ti, su, xu, xi;
    DevBuf<uint8_t> dt, f_train, f_test, f_keep;
    DevBuf<uint64_t> k0, k1, k2;
    DevBuf<int> counts;        // [0] train events, [1] unique train pairs, [2] test events, [3] unique test pairs, [4] kept test pairs, [5] bad
    CubTemp tmp;
    struct Free { std::vector<std::function<void()>> fs; ~Free() { for (auto& f : fs) f(); } } guard;
    guard.fs = {[&] { du.release(); di.release(); tu.release(); ti.release(); su.release(); xu.release(); xi.release(); },
                [&] { dt.release(); f_train.release(); f_test.release(); f_keep.release(); },
                [&] { k0.release(); k1.release(); k2.release(); counts.release(); tmp.buf.release(); }};
    CK(du.resize(Ez)); CK(di.resize(Ez)); CK(tu.resize(Ez)); CK(ti.resize(Ez)); CK(su.resize(Ez)); CK(xu.resize(Ez)); CK(xi.resize(Ez));
    CK(dt.resize(Ez)); CK(f_train.resize(Ez)); CK(f_test.resize(Ez)); CK(f_keep.resize(Ez));
    CK(k0.resize(Ez)); CK(k1.resize(Ez)); CK(k2.resize(Ez)); CK(counts.resize(8));
    CK(cudaMemsetAsync(counts.p, 0, 8 * sizeof(int), st));
    const int grid = (int)std::min<int64_t>((E + 255) / 256 + 1, (int64_t)h->sm_count * 16);
    int hc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (E) {
        CK(cudaMemcpyAsync(du.p, ev_user, E * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(di.p, ev_item, E * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        if (is_test) CK(cudaMemcpyAsync(dt.p, is_test, E * sizeof(uint8_t), cudaMemcpyHostToDevice, st));
        ingest_range_check_kernel<<<grid, 256, 0, st>>>(du.p, di.p, E, m, n, counts.p + 5);
        ingest_flags_kernel<<<grid, 256, 0, st>>>(is_test ? dt.p : nullptr, E, f_train.p, f_test.p);
        h->launches += 2;
        // temp storage: the largest request of the primitives used below
        size_t need = 0, b = 0;
        cub::DeviceSelect::Flagged(nullptr, b, du.p, f_train.p, tu.p, counts.p, (int)E, st); need = std::max(need, b);
        cub::DeviceRadixSort::SortPairs(nullptr, b, tu.p, su.p, ti.p, xi.p, (int)E, 0, 32, st); need = std::max(need, b);
        cub::DeviceRadixSort::SortKeys(nullptr, b, k0.p, k1.p, (int)E, 0, 64, st); need = std::max(need, b);
        cub::DeviceSelect::Unique(nullptr, b, k1.p, k2.p, counts.p, (int)E, st); need = std::max(need, b);
        cub::DeviceSelect::Flagged(nullptr, b, k1.p, f_keep.p, k2.p, counts.p, (int)E, st); need = std::max(need, b);
        CK(tmp.ensure(need));
        size_t tb = tmp.buf.n;
        // training events in file order
        CK(cub::DeviceSelect::Flagged(tmp.buf.p, tb, du.p, f_train.p, tu.p, counts.p + 0, (int)E, st));
        CK(cub::DeviceSelect::Flagged(tmp.buf.p, tb, di.p, f_train.p, ti.p, counts.p + 0, (int)E, st));
        CK(cub::DeviceSelect::Flagged(tmp.buf.p, tb, du.p, f_test.p, xu.p, counts.p + 2, (int)E, st));
        CK(cub::DeviceSelect::Flagged(tmp.buf.p, tb, di.p, f_test.p, xi.p, counts.p + 2, (int)E, st));
        h->launches += 8;
        CK(cudaMemcpyAsync(hc, counts.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        REQUIRE(hc[5] == 0, YUE_E_ARG, "an event names a user or track outside [0, m) x [0, n)");
    }
    const int64_t T = hc[0], Et = hc[2];
    h->have_log = false;                       // see yue_set_interactions_shard
    if (m != h->m || n != h->n) h->have_factors = false;
    if (n != h->n) h->have_delta_w = false;
    h->m = m; h->n = n; h->T = T; h->user_begin = 0; h->event_base = 0;
    CK(h->ev_indptr.resize(m + 1)); CK(h->uq_indptr.resize(m + 1)); CK(h->test_indptr.resize(m + 1));
    CK(h->ev_items.resize(T));
    size_t tb = tmp.buf.n;
    if (T) {
        // ev: stable sort by user keeps the file order inside a user (BPR.py:42-45)
        CK(cub::DeviceRadixSort::SortPairs(tmp.buf.p, tb, tu.p, su.p, ti.p, h->ev_items.p, (int)T, 0, 32, st));
        // uq: sorted unique (user, track) pairs
        ingest_keys_kernel<<<grid, 256, 0, st>>>(tu.p, ti.p, T, k0.p);
        CK(cub::DeviceRadixSort::SortKeys(tmp.buf.p, tb, k0.p, k1.p, (int)T, 0, 64, st));
        CK(cub::DeviceSelect::Unique(tmp.buf.p, tb, k1.p, k2.p, counts.p + 1, (int)T, st));
        h->launches += 6;
    }
    ingest_indptr_from_users_kernel<<<(unsigned)((m + 256) / 256), 256, 0, st>>>(su.p, T, m, h->ev_indptr.p);
    ++h->launches;
    CK(cudaMemcpyAsync(hc + 1, counts.p + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const int64_t nnz = hc[1];
    h->nnz = nnz;
    CK(h->uq_items.resize(nnz));
    if (nnz) { ingest_low_words_kernel<<<grid, 256, 0, st>>>(k2.p, nnz, h->uq_items.p); ++h->launches; }
    ingest_indptr_from_keys_kernel<<<(unsigned)((m + 256) / 256), 256, 0, st>>>(k2.p, nnz, m, h->uq_indptr.p);
    ++h->launches;
    // test set: unique held-out pairs that are not training pairs (record.py:182-202); k2 = training pairs stays live
    int64_t n_test = 0;
    if (Et) {
        ingest_keys_kernel<<<grid, 256, 0, st>>>(xu.p, xi.p, Et, k0.p);
        CK(cub::DeviceRadixSort::SortKeys(tmp.buf.p, tb, k0.p, k1.p, (int)Et, 0, 64, st));
        CK(cub::DeviceSelect::Unique(tmp.buf.p, tb, k1.p, k0.p, counts.p + 3, (int)Et, st));
        CK(cudaMemcpyAsync(hc + 3, counts.p + 3, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const int64_t nt = hc[3];
        ingest_antijoin_kernel<<<grid, 256, 0, st>>>(k0.p, nt, k2.p, nnz, f_keep.p);
        CK(cub::DeviceSelect::Flagged(tmp.buf.p, tb, k0.p, f_keep.p, k1.p, counts.p + 4, (int)nt, st));
        CK(cudaMemcpyAsync(hc + 4, counts.p + 4, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        n_test = hc[4];
        h->launches += 7;
    }
    CK(h->test_items.resize(n_test));
    if (n_test) { ingest_low_words_kernel<<<grid, 256, 0, st>>>(k1.p, n_test, h->test_items.p); ++h->launches; }
    ingest_indptr_from_keys_kernel<<<(unsigned)((m + 256) / 256), 256, 0, st>>>(k1.p, n_test, m, h->test_indptr.p);
    ++h->launches;
    CK(cudaGetLastError());
    h->have_test = true;
    h->n_test = n_test;
    std::vector<int64_t> hev((size_t)m + 1), huq((size_t)m + 1);
    CK(cudaMemcpyAsync(hev.data(), h->ev_indptr.p, (m + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(huq.data(), h->uq_indptr.p, (m + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return finish_interactions(h, hev.data(), huq.data(), false);
}

int yue_interaction_sizes(yue_t* h, int64_t* m, int64_t* n, int64_t* T, int64_t* nnz, int64_t* n_test) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "interactions not set");
    if (m) *m = h->m;
    if (n) *n = h->n;
    if (T) *T = h->T;
    if (nnz) *nnz = h->nnz;
    if (n_test) *n_test = h->have_test ? h->n_test : 0;
    return YUE_OK;
}

int yue_get_interactions(yue_t* h, int64_t* ev_indptr, int32_t* ev_items, int64_t* uq_indptr, int32_t* uq_items) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "interactions not set");
    CK(cudaSetDevice(h->device));
    if (ev_indptr) CK(cudaMemcpyAsync(ev_indptr, h->ev_indptr.p, (h->m + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    if (uq_indptr) CK(cudaMemcpyAsync(uq_indptr, h->uq_indptr.p, (h->m + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    if (ev_items && h->T) CK(cudaMemcpyAsync(ev_items, h->ev_items.p, h->T * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (uq_items && h->nnz) CK(cudaMemcpyAsync(uq_items, h->uq_items.p, h->nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (ev_items)                       // hot positives are stored re-labelled -slot-1 on the device
        for (int64_t e = 0; e < h->T; ++e) if (ev_items[e] < 0) ev_items[e] = h->h_hot_items[(size_t)(-ev_items[e] - 1)];
    return YUE_OK;
}

int yue_get_test_set(yue_t* h, int64_t* test_indptr, int32_t* test_items) {
    REQUIRE(h && h->have_log && h->have_test, YUE_E_STATE, "no test set on the device");
    CK(cudaSetDevice(h->device));
    if (test_indptr) CK(cudaMemcpyAsync(test_indptr, h->test_indptr.p, (h->m + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    if (test_items && h->n_test) CK(cudaMemcpyAsync(test_items, h->test_items.p, h->n_test * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

int yue_set_event_offsets(yue_t* h, const int64_t* delta) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "call yue_set_interactions first");
    CK(cudaSetDevice(h->device));
    if (!delta) { h->have_ev_delta = false; return YUE_OK; }
    CK(h->ev_delta.resize(std::max<int64_t>(h->m, 1)));
    if (h->m) CK(cudaMemcpyAsync(h->ev_delta.p, delta, h->m * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->have_ev_delta = true;
    return YUE_OK;
}

int yue_set_factors(yue_t* h, int k, const float* P, const float* Q) {
    REQUIRE(h && P && Q, YUE_E_ARG, "null argument");
    REQUIRE(h->have_log, YUE_E_STATE, "call yue_set_interactions first (it fixes m and n)");
    REQUIRE(k >= 1 && k <= 256, YUE_E_UNSUPPORTED, "num.factors must be in 1..256");
    CK(cudaSetDevice(h->device));
    // Row stride: k rounded up to 4 floats (128-bit accesses).  Between 65 and 127 factors the blocked SGD kernel would run
    // its 4-floats-per-lane form with masked lanes, which does not fit the register file (1.3 KB of spills): those widths
    // are padded to 128 floats instead (the full-width instantiation; pad columns stay zero under every update).
    int ld = (k + 3) & ~3;
    if (ld > 64 && ld < 128 && !(getenv("YUE_LD_PAD128") && atoi(getenv("YUE_LD_PAD128")) == 0)) ld = 128;
    h->k = k; h->ld = ld;
    CK(h->P.resize((size_t)std::max<int64_t>(h->m, 1) * ld));
    CK(h->Q.resize((size_t)h->n * ld));
    if (ld != k) {   // zero the pad columns; they stay zero under every update
        CK(cudaMemsetAsync(h->P.p, 0, (size_t)std::max<int64_t>(h->m, 1) * ld * sizeof(float), h->stream));
        CK(cudaMemsetAsync(h->Q.p, 0, (size_t)h->n * ld * sizeof(float), h->stream));
    }
    if (h->m) CK(cudaMemcpy2DAsync(h->P.p, ld * sizeof(float), P, k * sizeof(float), k * sizeof(float), h->m, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpy2DAsync(h->Q.p, ld * sizeof(float), Q, k * sizeof(float), k * sizeof(float), h->n, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->have_factors = true;
    h->gcn_t = 0; h->gcn_final = false;         // new variables: Adam starts over
    h->ba_t = 0;                                // (K9's and K10's Adam alike)
    h->have_snap = false;
    h->exchange_pending = false;
    h->hot_shared = false;                     // new tables: the owners' rows no longer describe them
    h->hot_stale = false;
    h->tc.q_dirty = true;
    h->rowmajor_current = true;
    h->ilv_current = false;
    return YUE_OK;
}

int yue_get_factors(yue_t* h, float* P, float* Q) {
    REQUIRE(h && h->have_factors, YUE_E_STATE, "factors not set");
    if (Q) REQUIRE(!h->hot_stale, YUE_E_STATE, "the shared hot rows were trained since the last yue_hot_pull: Q holds stale copies of them");
    CK(cudaSetDevice(h->device));
    if (Q) { if (int rc = q_rowmajor(h)) return rc; }
    const int k = h->k, ld = h->ld;
    if (P && h->m) CK(cudaMemcpy2DAsync(P, k * sizeof(float), h->P.p, ld * sizeof(float), k * sizeof(float), h->m, cudaMemcpyDeviceToHost, h->stream));
    if (Q) CK(cudaMemcpy2DAsync(Q, k * sizeof(float), h->Q.p, ld * sizeof(float), k * sizeof(float), h->n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

// Q lives in two layouts (see q_ilv_float_offset); these make one of them current.
static int q_rowmajor(yue_t* h) {
    if (h->rowmajor_current) return YUE_OK;
    q_from_ilv_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>((float4*)h->Q.p, h->Qilv.p, h->n);
    ++h->launches;
    CK(cudaGetLastError());
    h->rowmajor_current = true;
    return YUE_OK;
}
static int q_interleaved(yue_t* h) {
    if (h->ilv_current) return YUE_OK;
    const size_t floats = (size_t)((h->n + 15) / 16) * 1024;
    CK(h->Qilv.resize(floats));
    q_to_ilv_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>((const float4*)h->Q.p, h->Qilv.p, h->n);
    ++h->launches;
    CK(cudaGetLastError());
    h->ilv_current = true;
    return YUE_OK;
}

// host copies of the two indptr arrays, for the rarely used paths that need them (check hooks)
static int host_indptrs(yue_t* h) {
    if ((int64_t)h->h_ev_indptr.size() == h->m + 1) return YUE_OK;
    h->h_ev_indptr.resize((size_t)h->m + 1); h->h_uq_indptr.resize((size_t)h->m + 1);
    CK(cudaMemcpyAsync(h->h_ev_indptr.data(), h->ev_indptr.p, (h->m + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->h_uq_indptr.data(), h->uq_indptr.p, (h->m + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

static int ensure_ev_user(yue_t* h) {
    if (h->have_ev_user) return YUE_OK;
    if (int rc = host_indptrs(h)) return rc;
    std::vector<int32_t> eu((size_t)h->T);
    for (int64_t u = 0; u < h->m; ++u)
        std::fill(eu.begin() + h->h_ev_indptr[u], eu.begin() + h->h_ev_indptr[u + 1], (int32_t)u);
    CK(h->ev_user.resize(h->T));
    if (h->T) CK(cudaMemcpy(h->ev_user.p, eu.data(), eu.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    h->have_ev_user = true;
    return YUE_OK;
}

int yue_sample_negatives(yue_t* h, uint64_t seed, uint32_t epoch, uint32_t slot, int32_t* j_out) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "interactions not set");
    REQUIRE(j_out || h->T == 0, YUE_E_ARG, "null output");
    REQUIRE(slot < 4096, YUE_E_ARG, "slot must be < 4096");
    CK(cudaSetDevice(h->device));
    if (h->T == 0) return YUE_OK;
    if (int rc = ensure_ev_user(h)) return rc;
    CK(h->tmp_j.resize(h->T));
    const int grid = (int)std::min<int64_t>((h->T + 255) / 256, (int64_t)h->sm_count * 16);
    sample_negatives_kernel<<<grid, 256, 0, h->stream>>>(h->T, h->ev_user.p, h->uq_indptr.p, h->uq_items.p, seed, epoch,
                                                         slot, h->event_base, h->have_ev_delta ? h->ev_delta.p : nullptr, (uint32_t)h->n, h->tmp_j.p);
    ++h->launches;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(j_out, h->tmp_j.p, h->T * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

template <int NCH, bool ILV, bool APR>
static cudaError_t launch_sgd(const SgdParams& sp, int mode, int warps_per_cta, cudaStream_t st) {
    if (mode == YUE_MODE_SERIAL) {
        bpr_sgd_kernel<NCH, kSerial, 1, ILV, APR><<<1, 32, 0, st>>>(sp);
        return cudaGetLastError();
    }
    constexpr int PF = NCH <= 2 ? 4 : 2;
    // one CTA per SM with warps_per_cta warps each (not n_warps packed into full CTAs: that would
    // leave SMs idle when fewer than 16 warps per SM are wanted)
    const int grid = (sp.n_warps + warps_per_cta - 1) / warps_per_cta;
    const size_t smem = (size_t)sp.n_hot * 8;
    auto kern = mode == YUE_MODE_HOGWILD ? bpr_sgd_kernel<NCH, kAtomic, PF, ILV, APR> : bpr_sgd_kernel<NCH, kStore, PF, ILV, APR>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024));
    if (e != cudaSuccess) return e;
    kern<<<grid, warps_per_cta * 32, smem, st>>>(sp);
    return cudaGetLastError();
}

// blocked kernel: hot rows move into the slice-friendly table for the launch and back after it
template <int V, bool APR>
static cudaError_t launch_sgd_blk(const SgdParams& sp, int warps_per_cta, cudaStream_t st, int64_t& launches) {
    const bool mask = sp.ld != 32 * V;          // rows narrower than the warp's 32 x V floats: tail lanes switched off
    warps_per_cta = std::min(warps_per_cta, kBlkThreads / 32);
    const int grid = (sp.n_warps + warps_per_cta - 1) / warps_per_cta;
    if (sp.hot_base) {                          // yue_hot_share: the rows stay in the owners' tables across launches
        const size_t smem = (size_t)((3 * sp.n_hot + 3) & ~3) * 4 + (size_t)sp.n_hot * 8;
        bpr_sgd_blk_kernel<V, APR, false, true><<<grid, warps_per_cta * 32, smem, st>>>(sp);
        return cudaGetLastError();
    }
    if (sp.n_hot > 0) { hot_gather_kernel<V><<<(sp.n_hot + 7) / 8, 256, 0, st>>>(sp.Q, sp.hotQ, sp.hot_items, sp.hot_dx, sp.n_hot, sp.ld, sp.hot_plane); ++launches; }
    if (mask) bpr_sgd_blk_kernel<V, APR, true><<<grid, warps_per_cta * 32, (size_t)sp.n_hot * 12, st>>>(sp);
    else bpr_sgd_blk_kernel<V, APR, false><<<grid, warps_per_cta * 32, (size_t)sp.n_hot * 12, st>>>(sp);
    if (sp.n_hot > 0) { hot_scatter_kernel<V><<<(sp.n_hot + 7) / 8, 256, 0, st>>>(sp.Q, sp.hotQ, sp.hot_items, sp.hot_dx, sp.n_hot, sp.ld, sp.hot_plane); ++launches; }
    return cudaGetLastError();
}

// floats per lane of the blocked kernel for rows of ld floats (ld <= 128)
static int blk_width(int ld) { return ld <= 32 ? 1 : ld <= 64 ? 2 : 4; }

// does the blocked kernel (bpr_sgd_blk.cuh) take this launch?
static bool use_blk_kernel(const yue_t* h, int mode, bool apr) {
    (void)apr;
    return h->sgd_kernel == 2 && mode == YUE_MODE_HOGWILD && h->ld <= 128 &&
           (uint64_t)h->n * h->ld * 4 < ((uint64_t)1 << 32);      // 32-bit byte offsets inside Q
}

// (re)build the shard table of the hot tracks for the kernel about to run
static int ensure_hot_meta(yue_t* h, int cap) {
    if (h->n_hot == 0 || (h->hot_meta_cap == cap && h->hot_meta_ld == h->ld)) return YUE_OK;
    std::vector<int32_t> meta((size_t)h->n_hot);
    int64_t rows = 0;
    for (int s = 0; s < h->n_hot; ++s) {
        const int64_t want = ((int64_t)h->h_hot_counts[s] * h->hot_div + h->T - 1) / std::max<int64_t>(h->T, 1);
        int R = 1;
        while (R < want && R < cap) R *= 2;
        meta[s] = (int32_t)((rows << 4) | R);
        rows += R - 1;
    }
    CK(h->hot_meta.resize(h->n_hot));
    CK(cudaMemcpyAsync(h->hot_meta.p, meta.data(), meta.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(h->hot_shards.resize((size_t)std::max<int64_t>(rows, 1) * h->ld));
    CK(cudaMemsetAsync(h->hot_shards.p, 0, (size_t)std::max<int64_t>(rows, 1) * h->ld * sizeof(float), h->stream));
    CK(cudaStreamSynchronize(h->stream));       // meta dies here
    h->hot_extra_rows = rows; h->hot_meta_cap = cap; h->hot_meta_ld = h->ld;
    return YUE_OK;
}

// see yue_handle::hot_offset_granules
static int calibrate_hot_offset(yue_t* h, SgdParams sp, int wpc) {
    uint64_t key = (uint64_t)(uintptr_t)h->hotQ.p * 1000003ull + (uint64_t)h->n_hot * 7919ull + (uint64_t)h->ld * 31ull + (uint64_t)h->T;
    for (int32_t t : h->h_hot_items) key = key * 6364136223846793005ull + (uint64_t)t + 1442695040888963407ull;
    if (key == 0) key = 1;
    if (h->hot_calibrated_key == key) return YUE_OK;
    h->hot_calibrated_key = key;
    if (h->hot_offset_forced >= 0) { h->hot_offset_granules = h->hot_offset_forced; return YUE_OK; }
    h->hot_offset_granules = 0;
    const int64_t n_items = sp.n_work;
    if (h->T < ((int64_t)1 << 22) || n_items < 4096) return YUE_OK;      // small logs: not worth 8 probes
    sp.lr = 0.f; sp.c_u = 0.f; sp.c_i = 0.f; sp.lr_d = 0.0; sp.loss = h->scal.p + 3; sp.ev_neg = nullptr;
    sp.item_first = n_items / 3; sp.n_work = sp.item_first + std::max<int64_t>(1024, n_items / 32);
    sp.n_work = std::min(sp.n_work, n_items);
    h->hot_calibration_ms.assign(kHotCandidates, 0.f);
    float best = 1e30f;
    for (int c = 0; c < kHotCandidates; ++c) {
        sp.hotQ = h->hotQ.p + (size_t)c * kHotCandidateStep * 64;
        const unsigned long long c0 = (unsigned long long)sp.item_first;
        CK(cudaMemcpyAsync(h->cursor.p, &c0, sizeof(c0), cudaMemcpyHostToDevice, h->stream));
        CK(cudaEventRecord(h->ev0, h->stream));
        switch (blk_width(h->ld)) {
            case 1: CK(launch_sgd_blk<1, false>(sp, wpc, h->stream, h->launches)); break;
            case 2: CK(launch_sgd_blk<2, false>(sp, wpc, h->stream, h->launches)); break;
            default: CK(launch_sgd_blk<4, false>(sp, wpc, h->stream, h->launches)); break;
        }
        ++h->launches;
        CK(cudaEventRecord(h->ev1, h->stream));
        CK(cudaEventSynchronize(h->ev1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        h->hot_calibration_ms[c] = ms;
        if (ms < best) { best = ms; h->hot_offset_granules = c * kHotCandidateStep; }
    }
    return YUE_OK;
}

static int run_sgd(yue_t* h, SgdParams sp, int mode, double* loss_out, bool apr = false) {
    REQUIRE(mode >= YUE_MODE_SERIAL && mode <= YUE_MODE_HOGWILD_STORE, YUE_E_ARG, "unknown mode");
    sp.cursor = h->cursor.p;
    sp.hot_plane = hot_plane_floats(sp.n_hot + kHotExtra);       // every rank of a shared table has the same n_hot
    const bool blk = use_blk_kernel(h, mode, apr);
    { int rb = 1; while (rb * 2 * kBlkK <= sp.resync_events) rb *= 2; sp.resync_mask = rb - 1; }
    // YUE_SGD_L2_PREFETCH = stride in bytes (experiments): prefetch a segment's rows into L2 when its negatives are drawn.  Off:
    // measured at config C3's shard (Q = 1 GB, d = 128), ms per epoch: off 41.7, one prefetch per 128 B 42.7, per 64 B 46.1, per
    // 32 B 62.6 -- the register loads issued one block ahead already cover the DRAM latency; the extra requests only load the L2
    sp.pf_stride = 0;
    if (const char* s = getenv("YUE_SGD_L2_PREFETCH")) sp.pf_stride = std::max(0, atoi(s));
    const bool ilv = h->use_ilv && h->ld == 64 && mode != YUE_MODE_SERIAL && !apr && !blk;
    if (ilv) { if (int rc = q_interleaved(h)) return rc; } else { if (int rc = q_rowmajor(h)) return rc; }
    sp.P = h->P.p; sp.Q = ilv ? h->Qilv.p : h->Q.p; sp.ld = h->ld; sp.nchunks = h->ld / 4; sp.n_items = (uint32_t)h->n;
    sp.uq_indptr = h->uq_indptr.p; sp.uq_items = h->uq_items.p; sp.loss = h->scal.p;
    if (h->hot_shared && sp.n_hot > 0)
        REQUIRE(blk && h->ld == 32 * blk_width(h->ld) && mode == YUE_MODE_HOGWILD, YUE_E_STATE,
                "the hot rows are shared between ranks (yue_hot_share): only the Hogwild epochs at num.factors 32/64/128 may run; call yue_hot_unshare first");
    if (sp.n_hot > 0) {
        if (blk && h->hot_shared) {
            sp.hot_sorted = h->hot_sorted.p; sp.hot_sorted_slot = h->hot_sorted_slot.p; sp.hot_dx = h->hot_dx.p;
            sp.hot_base = h->hot_base.p; sp.hotQ = h->hotQ.p;
        } else if (blk) {
            sp.hot_sorted = h->hot_sorted.p; sp.hot_sorted_slot = h->hot_sorted_slot.p; sp.hot_dx = h->hot_dx.p;
            if (int rc = calibrate_hot_offset(h, sp, std::max(1, std::min(kSgdThreads / 32, h->warps_per_sm)))) return rc;
            sp.hotQ = h->hotQ.p + (size_t)h->hot_offset_granules * 64;
        }
        else {
            if (int rc = ensure_hot_meta(h, kHotShards)) return rc;
            sp.hot_meta = h->hot_meta.p; sp.hot_shards = h->hot_shards.p;
        }
    }
    CK(cudaMemsetAsync(h->scal.p, 0, sizeof(double), h->stream));
    if (sp.item_first == 0) CK(cudaMemsetAsync(h->cursor.p, 0, sizeof(unsigned long long), h->stream));
    else { const unsigned long long c0 = (unsigned long long)sp.item_first; CK(cudaMemcpyAsync(h->cursor.p, &c0, sizeof(c0), cudaMemcpyHostToDevice, h->stream)); CK(cudaStreamSynchronize(h->stream)); }
    const int nch = (sp.nchunks + 15) / 16;
    int wpc = std::max(1, std::min(kSgdThreads / 32, h->warps_per_sm));
    if (mode != YUE_MODE_SERIAL && h->sgd_warps_forced > 0) {        // yue_set_sgd_concurrency
        sp.n_warps = h->sgd_warps_forced;
        const int ctas = h->sgd_ctas_forced > 0 ? h->sgd_ctas_forced : h->sm_count;
        wpc = std::max(1, std::min(blk ? kBlkThreads / 32 : kSgdThreads / 32, (sp.n_warps + ctas - 1) / ctas));
        sp.n_warps = std::min(sp.n_warps, wpc * ctas);
    }
    if (blk) {
        switch (blk_width(h->ld)) {
            case 1: CK(apr ? launch_sgd_blk<1, true>(sp, wpc, h->stream, h->launches) : launch_sgd_blk<1, false>(sp, wpc, h->stream, h->launches)); break;
            case 2: CK(apr ? launch_sgd_blk<2, true>(sp, wpc, h->stream, h->launches) : launch_sgd_blk<2, false>(sp, wpc, h->stream, h->launches)); break;
            default: CK(apr ? launch_sgd_blk<4, true>(sp, wpc, h->stream, h->launches) : launch_sgd_blk<4, false>(sp, wpc, h->stream, h->launches)); break;
        }
    } else
    switch (nch) {
        case 1: if (apr) CK(launch_sgd<1, false, true>(sp, mode, wpc, h->stream));
                else if (ilv) CK(launch_sgd<1, true, false>(sp, mode, wpc, h->stream));
                else CK(launch_sgd<1, false, false>(sp, mode, wpc, h->stream));
                break;
        case 2: if (apr) CK(launch_sgd<2, false, true>(sp, mode, wpc, h->stream)); else CK(launch_sgd<2, false, false>(sp, mode, wpc, h->stream)); break;
        case 3: if (apr) CK(launch_sgd<3, false, true>(sp, mode, wpc, h->stream)); else CK(launch_sgd<3, false, false>(sp, mode, wpc, h->stream)); break;
        case 4: if (apr) CK(launch_sgd<4, false, true>(sp, mode, wpc, h->stream)); else CK(launch_sgd<4, false, false>(sp, mode, wpc, h->stream)); break;
        default: return fail(h, YUE_E_UNSUPPORTED, "num.factors > 256");
    }
    ++h->launches;
    if (mode != YUE_MODE_SERIAL && !blk && sp.n_hot > 0 && h->hot_extra_rows > 0) {     // fold the hot-row shards back into Q
        const int fgrid = (sp.n_hot * (h->ld / 4) + 255) / 256;
        if (ilv) hot_fold_kernel<true><<<fgrid, 256, 0, h->stream>>>(sp.Q, sp.hot_shards, sp.hot_items, sp.hot_meta, sp.n_hot, h->ld);
        else hot_fold_kernel<false><<<fgrid, 256, 0, h->stream>>>(sp.Q, sp.hot_shards, sp.hot_items, sp.hot_meta, sp.n_hot, h->ld);
        ++h->launches;
        CK(cudaGetLastError());
    }
    if (ilv) h->rowmajor_current = false; else h->ilv_current = false;   // the other copy is stale now
    h->tc.q_dirty = true;
    if (blk && h->hot_shared && sp.n_hot > 0) h->hot_stale = true;      // the hot rows were trained in the owners' tables
    if (loss_out) {
        CK(cudaMemcpyAsync(loss_out, h->scal.p, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (!std::isfinite(*loss_out))
            return fail(h, YUE_E_NUMERIC, "Loss = NaN or Infinity: current settings does not fit the recommender!");
    }
    return YUE_OK;
}

static void fill_rates(SgdParams& sp, double lr, double regU, double regI) {
    sp.lr_d = lr; sp.lr = (float)lr; sp.c_u = (float)(lr * regU); sp.c_i = (float)(lr * regI);
}

static int sgd_epoch(yue_t* h, double lr, double regU, double regI, uint64_t seed, uint32_t epoch, uint32_t slot,
                     int mode, double* loss_out, bool apr, double eps, double regA, int part = 0, int n_parts = 1) {
    REQUIRE(n_parts >= 1 && part >= 0 && part < n_parts, YUE_E_ARG, "part must be in [0, n_parts)");
    REQUIRE(h && h->have_log && h->have_factors, YUE_E_STATE, "set interactions and factors first");
    REQUIRE(slot < 4096, YUE_E_ARG, "slot must be < 4096");
    CK(cudaSetDevice(h->device));
    if (h->T == 0) { if (loss_out) *loss_out = 0.0; return YUE_OK; }
    SgdParams sp{};
    fill_rates(sp, lr, regU, regI);
    sp.seg_rec = h->seg_rec.p;
    sp.item_ptr = h->item_ptr.p;
    // sub-epoch: the part-th of n_parts consecutive ranges of the work items (stream order)
    sp.item_first = h->n_items * part / n_parts; sp.n_work = h->n_items * (part + 1) / n_parts;
    if (sp.item_first == sp.n_work) { if (loss_out) *loss_out = 0.0; return YUE_OK; }
    sp.n_warps = mode == YUE_MODE_SERIAL ? 1 : h->n_warps;
    sp.ev_items = h->ev_items.p; sp.ev_neg = nullptr;
    sp.hot_items = h->hot_items.p; sp.n_hot = h->n_hot;
    sp.resync_events = h->resync_events;
    sp.seed = seed; sp.epoch = epoch; sp.event_base = h->event_base; sp.ev_delta = h->have_ev_delta ? h->ev_delta.p : nullptr; sp.slot = slot;
    sp.eps = (float)eps; sp.regA = (float)regA;
    return run_sgd(h, sp, mode, loss_out, apr);
}
int yue_bpr_epoch(yue_t* h, double lr, double regU, double regI, uint64_t seed, uint32_t epoch, int mode,
                  double* loss_out) {
    return sgd_epoch(h, lr, regU, regI, seed, epoch, 0u, mode, loss_out, false, 0.0, 0.0);
}
int yue_bpr_epoch_part(yue_t* h, double lr, double regU, double regI, uint64_t seed, uint32_t epoch, int mode,
                       int part, int n_parts, double* loss_out) {
    return sgd_epoch(h, lr, regU, regI, seed, epoch, 0u, mode, loss_out, false, 0.0, 0.0, part, n_parts);
}
int yue_apr_epoch(yue_t* h, double lr, double regU, double regI, double eps, double regA, uint64_t seed,
                  uint32_t epoch, uint32_t slot, int mode, double* loss_out) {
    return sgd_epoch(h, lr, regU, regI, seed, epoch, slot, mode, loss_out, true, eps, regA);
}

int yue_apr_epoch_part(yue_t* h, double lr, double regU, double regI, double eps, double regA, uint64_t seed,
                       uint32_t epoch, uint32_t slot, int mode, int part, int n_parts, double* loss_out) {
    return sgd_epoch(h, lr, regU, regI, seed, epoch, slot, mode, loss_out, true, eps, regA, part, n_parts);
}

static int sgd_apply(yue_t* h, const int32_t* u, const int32_t* i, const int32_t* j, int64_t T, double lr,
                     double regU, double regI, int mode, double* loss_out, bool apr, double eps, double regA) {
    REQUIRE(h && h->have_log && h->have_factors, YUE_E_STATE, "set interactions and factors first");
    REQUIRE(T >= 0 && (T == 0 || (u && i && j)), YUE_E_ARG, "null triplet array");
    CK(cudaSetDevice(h->device));
    if (T == 0) { if (loss_out) *loss_out = 0.0; return YUE_OK; }
    std::vector<int64_t> rb, re;
    std::vector<int32_t> ru;
    for (int64_t t = 0; t < T;) {               // runs of one user
        REQUIRE(u[t] >= 0 && u[t] < h->m, YUE_E_ARG, "triplet user out of range");
        int64_t e = t;
        while (e < T && u[e] == u[t]) {
            REQUIRE(i[e] >= 0 && i[e] < h->n && j[e] >= 0 && j[e] < h->n, YUE_E_ARG, "triplet item out of range");
            ++e;
        }
        rb.push_back(t); re.push_back(e); ru.push_back(u[t]);
        t = e;
    }
    const int n_warps = mode == YUE_MODE_SERIAL ? 1
        : (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)h->sm_count * h->warps_per_sm, T / h->min_events_per_warp));
    if (int rc = host_indptrs(h)) return rc;
    const ItemPlanArgs plan{mode != YUE_MODE_SERIAL, std::max<int64_t>(32, std::min<int64_t>(256, T / ((int64_t)n_warps * 4 * 32))),
                            h->max_items_per_user, mode == YUE_MODE_SERIAL ? 1 : h->item_group_segs, 32, h->h_uq_indptr.data()};
    int64_t nseg = 0, nitems = 0;
    PinBuf<SegRec> recs;
    PinBuf<int64_t> ip;
    cudaError_t pe = plan_items(rb.size(), [&](size_t r, int64_t& b, int64_t& e, int32_t& uu) { b = rb[r]; e = re[r]; uu = ru[r]; },
                                plan, recs, ip, nseg, nitems);
    struct Guard { PinBuf<SegRec>& a; PinBuf<int64_t>& b; cudaStream_t st; ~Guard() { cudaStreamSynchronize(st); a.release(); b.release(); } } guard{recs, ip, h->stream};
    if (pe != cudaSuccess) return fail(h, YUE_E_CUDA, std::string("plan_items: ") + cudaGetErrorString(pe));
    CK(h->tmp_rec.resize((size_t)nseg));
    CK(cudaMemcpyAsync(h->tmp_rec.p, recs.p, (size_t)nseg * sizeof(SegRec), cudaMemcpyHostToDevice, h->stream));
    CK(h->tmp_i.resize(T)); CK(h->tmp_j.resize(T));
    CK(h->tmp_ws.resize((size_t)nitems * 2)); CK(h->cursor.resize(1));
    CK(cudaMemcpyAsync(h->tmp_i.p, i, T * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->tmp_j.p, j, T * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->tmp_ws.p, ip.p, (size_t)nitems * 2 * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    SgdParams sp{};
    fill_rates(sp, lr, regU, regI);
    sp.seg_rec = h->tmp_rec.p;
    sp.item_ptr = h->tmp_ws.p; sp.n_work = nitems; sp.n_warps = n_warps;
    sp.ev_items = h->tmp_i.p; sp.ev_neg = h->tmp_j.p;
    sp.n_hot = 0;                                // explicit triplets take the direct path
    sp.resync_events = h->resync_events;
    sp.eps = (float)eps; sp.regA = (float)regA;
    int rc = run_sgd(h, sp, mode, loss_out, apr);
    cudaStreamSynchronize(h->stream);           // host staging vectors die here
    return rc;
}
int yue_bpr_apply(yue_t* h, const int32_t* u, const int32_t* i, const int32_t* j, int64_t T, double lr,
                  double regU, double regI, int mode, double* loss_out) {
    return sgd_apply(h, u, i, j, T, lr, regU, regI, mode, loss_out, false, 0.0, 0.0);
}
int yue_apr_apply(yue_t* h, const int32_t* u, const int32_t* i, const int32_t* j, int64_t T, double lr,
                  double regU, double regI, double eps, double regA, int mode, double* loss_out) {
    return sgd_apply(h, u, i, j, T, lr, regU, regI, mode, loss_out, true, eps, regA);
}

// ---- K8: CUNE's two-level BPR epoch (cune_sgd.cuh) --------------------------------------------------------------------
int yue_cune_set_implicit(yue_t* h, const int64_t* ip_indptr, const int32_t* ip_items) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "call yue_set_interactions first");
    REQUIRE(ip_indptr, YUE_E_ARG, "null ip_indptr");
    CK(cudaSetDevice(h->device));
    REQUIRE(ip_indptr[0] == 0, YUE_E_ARG, "ip_indptr[0] must be 0");
    for (int64_t u = 0; u < h->m; ++u) REQUIRE(ip_indptr[u + 1] >= ip_indptr[u], YUE_E_ARG, "ip_indptr not monotone");
    const int64_t nip = ip_indptr[h->m];
    REQUIRE(nip == 0 || ip_items, YUE_E_ARG, "null ip_items");
    // an implicit positive is a track the user has NOT played (CUNE.py:111-113); the kernel relies on it (k != i)
    if (int rc = host_indptrs(h)) return rc;
    std::vector<int32_t> uq((size_t)std::max<int64_t>(h->nnz, 1));
    if (h->nnz) CK(cudaMemcpyAsync(uq.data(), h->uq_items.p, h->nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int64_t u = 0; u < h->m; ++u) {
        const int32_t* rb = uq.data() + h->h_uq_indptr[u];
        const int32_t* re = uq.data() + h->h_uq_indptr[u + 1];
        for (int64_t x = ip_indptr[u]; x < ip_indptr[u + 1]; ++x) {
            REQUIRE(ip_items[x] >= 0 && ip_items[x] < h->n, YUE_E_ARG, "implicit positive out of range");
            REQUIRE(!std::binary_search(rb, re, ip_items[x]), YUE_E_ARG,
                    "implicit positive " + std::to_string(ip_items[x]) + " was played by user " + std::to_string(u + h->user_begin));
        }
    }
    CK(h->ip_indptr.resize((size_t)h->m + 1)); CK(h->ip_items.resize((size_t)std::max<int64_t>(nip, 1)));
    CK(cudaMemcpyAsync(h->ip_indptr.p, ip_indptr, (h->m + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    if (nip) CK(cudaMemcpyAsync(h->ip_items.p, ip_items, nip * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));                   // the caller owns the host arrays
    h->have_ip = true;
    return YUE_OK;
}

template <int NC>
static cudaError_t launch_cune(const CuneParams& cp, int mode, int grid, int wpc, cudaStream_t st) {
    if (mode == YUE_MODE_SERIAL) cune_sgd_kernel<NC, kSerial><<<1, 32, 0, st>>>(cp);
    else cune_sgd_kernel<NC, kAtomic><<<grid, wpc * 32, 0, st>>>(cp);
    return cudaGetLastError();
}

int yue_cune_epoch(yue_t* h, double lr, double regU, double regI, double s, uint64_t seed, uint32_t epoch, int mode,
                   double* loss_out) {
    REQUIRE(h && h->have_log && h->have_factors, YUE_E_STATE, "set interactions and factors first");
    REQUIRE(h->have_ip, YUE_E_STATE, "call yue_cune_set_implicit first");
    REQUIRE(mode == YUE_MODE_SERIAL || mode == YUE_MODE_HOGWILD, YUE_E_ARG, "mode must be YUE_MODE_SERIAL or YUE_MODE_HOGWILD");
    REQUIRE(s > 0.0 && std::isfinite(s), YUE_E_ARG, "s must be positive");
    REQUIRE(h->ld <= 128 * kCuneMaxC && h->ld % 4 == 0, YUE_E_UNSUPPORTED, "num.factors > 256");
    CK(cudaSetDevice(h->device));
    if (h->T == 0) { if (loss_out) *loss_out = 0.0; return YUE_OK; }
    if (int rc = q_rowmajor(h)) return rc;
    CK(h->cune_scal.resize(1)); CK(h->cune_ctr.resize(2));
    // One warp per work item.  Like K2 (yue_handle::min_events_per_warp) a small log gets few warps: with every user of a
    // tiny log in flight at once the schedule is no longer a window sliding over the reference's user stream (first
    // hardware run, profiles/cune_r2.md: 60 users on 64 warps moved P[u] of the heaviest user by 2x its norm; one warp
    // reproduces the serial tables to 1e-6; 400 K events: 73 warps +1.1 points of Recall@10 against the serial order,
    // 293 warps +2.4).
    int n_warps = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)h->sm_count * 16, h->T / h->min_events_per_warp));
    if (const char* e = getenv("YUE_CUNE_WARPS")) n_warps = std::max(1, std::min(h->sm_count * 16, atoi(e)));   // tests, experiments
    if (mode == YUE_MODE_SERIAL) n_warps = 1;
    const int wpc = std::min(8, n_warps);
    const int grid = (n_warps + wpc - 1) / wpc;
    {   // work items: whole users in serial order; Hogwild cuts a user above a quarter of a warp's fair share of the epoch
        int64_t chunk = 0;
        if (mode != YUE_MODE_SERIAL) {
            chunk = std::max<int64_t>(256, std::min<int64_t>(8192, h->T / ((int64_t)n_warps * 4)));
            if (const char* e = getenv("YUE_CUNE_CHUNK")) chunk = std::max<int64_t>(32, atoll(e));
            chunk = (chunk + 31) / 32 * 32;
        }
        if (h->cune_chunk != chunk) {
            if (int rc = host_indptrs(h)) return rc;
            std::vector<int64_t> items;
            cune_plan_items(h->m, h->h_ev_indptr.data(), chunk, items);
            h->cune_n_work = (int64_t)items.size() / kCuneItemWords;
            CK(h->cune_items.resize(std::max<size_t>(items.size(), 1)));
            if (!items.empty()) CK(cudaMemcpyAsync(h->cune_items.p, items.data(), items.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
            CK(cudaStreamSynchronize(h->stream));           // the staging vector dies here
            h->cune_chunk = chunk;
        }
    }
    CK(cudaMemsetAsync(h->cune_scal.p, 0, sizeof(double), h->stream));
    CK(cudaMemsetAsync(h->cune_ctr.p, 0, 2 * sizeof(unsigned long long), h->stream));
    CuneParams cp{};
    cp.P = h->P.p; cp.Q = h->Q.p; cp.ld = h->ld; cp.k = h->k; cp.m = h->m; cp.n = h->n;
    cp.ev_indptr = h->ev_indptr.p; cp.ev_items = h->ev_items.p; cp.hot_items = h->hot_items.p;
    cp.items = h->cune_items.p; cp.n_work = h->cune_n_work;
    cp.uq_indptr = h->uq_indptr.p; cp.uq_items = h->uq_items.p;
    cp.ip_indptr = h->ip_indptr.p; cp.ip_items = h->ip_items.p;
    cp.seed = seed; cp.epoch = epoch; cp.event_base = h->event_base; cp.ev_delta = h->have_ev_delta ? h->ev_delta.p : nullptr;
    cp.lr = lr; cp.inv_s = 1.0 / s; cp.regU = regU; cp.regI = regI;
    cp.c_u = (float)(lr * regU); cp.c_i = (float)(lr * regI);
    cp.cursor = h->cune_ctr.p; cp.users_done = h->cune_ctr.p + 1; cp.loss = h->cune_scal.p;
    const bool event_loss = getenv("YUE_CUNE_EVENT_LOSS") != nullptr;      // the -log terms alone, in both modes (schedule comparisons)
    cp.skip_user_norms = (regU == 0.0 && regI == 0.0) || event_loss;
    if (h->ld <= 128) CK(launch_cune<1>(cp, mode, grid, wpc, h->stream));       // one 16-byte chunk per lane
    else CK(launch_cune<kCuneMaxC>(cp, mode, grid, wpc, h->stream));
    ++h->launches;
    h->ilv_current = false;
    h->tc.q_dirty = true;
    double loss = 0.0;
    unsigned long long users = 0;
    CK(cudaMemcpyAsync(&loss, h->cune_scal.p, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&users, h->cune_ctr.p + 1, sizeof(users), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (mode != YUE_MODE_SERIAL && (regU != 0.0 || regI != 0.0) && !event_loss) {
        // CUNE.py:174 adds the norms after every user; a parallel schedule has no per-user table state, so the
        // end-of-epoch norms stand in for all of them
        double p2 = 0.0, q2 = 0.0;
        if (int rc = yue_frob2(h, &p2, &q2)) return rc;
        loss += (double)users * (regU * p2 + regI * q2);
    }
    if (loss_out) *loss_out = loss;
    if (!std::isfinite(loss))
        return fail(h, YUE_E_NUMERIC, "Loss = NaN or Infinity: current settings does not fit the recommender!");
    return YUE_OK;
}

// ---- K9: LightGCN (lightgcn.cuh) --------------------------------------------------------------------------------------
static int wrmf_prepare(yue_t* h);

// the row lists of the product phases: a row with more than kGcnHeavy neighbours is worked on by a whole CTA
static int gcn_plan(yue_t* h) {
    if (h->gcn_planned) return YUE_OK;
    if (int rc = wrmf_prepare(h)) return rc;           // play counts per pair and the track-major copy of the pairs
    const int64_t m = h->m, n = h->n;
    REQUIRE(m + n < ((int64_t)1 << 31), YUE_E_UNSUPPORTED, "more than 2^31 graph rows");
    std::vector<int32_t> heavy;
    std::vector<int2> segs;
    auto deg = [&](int64_t r) { return r < m ? h->h_uq_indptr[r + 1] - h->h_uq_indptr[r] : h->h_it_indptr[r - m + 1] - h->h_it_indptr[r - m]; };
    int64_t open_row = -1, open_edges = 0;                // the segment being filled: rows [open_row, r)
    auto close = [&](int64_t r) { if (open_row >= 0) segs.push_back(make_int2((int)open_row, (int)(r - open_row))); open_row = -1; open_edges = 0; };
    for (int64_t r = 0; r < m + n; ++r) {
        const int64_t d = deg(r);
        if (r == m) close(r);                              // a segment stays on one side of the graph
        if (d > kGcnHeavy) { close(r); heavy.push_back((int32_t)r); continue; }
        if (open_row >= 0 && (r - open_row >= kGcnSegRows || open_edges + d > kGcnSegEdges)) close(r);
        if (open_row < 0) open_row = r;
        open_edges += d;
    }
    close(m + n);
    // largest first: the groups take items in turn, so every group's share ends with the small ones
    auto seg_edges = [&](const int2& sg) {
        const int64_t r0 = sg.x, r1 = sg.x + sg.y;
        return r0 < m ? h->h_uq_indptr[r1] - h->h_uq_indptr[r0] : h->h_it_indptr[r1 - m] - h->h_it_indptr[r0 - m];
    };
    std::stable_sort(segs.begin(), segs.end(), [&](const int2& a, const int2& b) { return seg_edges(a) > seg_edges(b); });
    // heavy rows, heaviest first, cut into chunks of ~sqrt(degree) (>= kGcnHeavy) neighbours: the gather of a chunk and the
    // sum of the row's partials by the last group to arrive then take about the same number of load rounds
    std::stable_sort(heavy.begin(), heavy.end(), [&](int32_t a, int32_t b) { return deg(a) > deg(b); });
    std::vector<GcnChunk> chunks;
    for (size_t hi = 0; hi < heavy.size(); ++hi) {
        const int64_t d = deg(heavy[hi]);
        int64_t c = (int64_t)std::ceil(std::sqrt((double)d) / 8.0) * 8;
        c = std::max<int64_t>(c, kGcnHeavy);
        const int nck = (int)((d + c - 1) / c), first = (int)chunks.size();
        for (int q = 0; q < nck; ++q)
            chunks.push_back(GcnChunk{heavy[hi], (int32_t)(q * c), (int32_t)std::min<int64_t>(c, d - q * c), first + q, first, nck, (int32_t)hi, 0});
    }
    // the groups of a warp (up to 4 of 8 lanes) take consecutive items and walk them in lockstep: they must be of one kind, so
    // the chunk list is padded to a multiple of 4 with empty chunks that never complete a row (their own counter, slot, row 0)
    while (chunks.size() % 4) chunks.push_back(GcnChunk{0, 0, 0, (int32_t)chunks.size(), (int32_t)chunks.size(), 0x7fffffff, (int32_t)heavy.size(), 0});
    CK(h->gcn_chunks.resize(std::max<size_t>(chunks.size(), 1))); CK(h->gcn_segs.resize(std::max<size_t>(segs.size(), 1)));
    CK(h->gcn_arrived.resize(heavy.size() + 1));
    CK(cudaMemsetAsync(h->gcn_arrived.p, 0, (heavy.size() + 1) * sizeof(unsigned), h->stream));
    if (!chunks.empty()) CK(cudaMemcpyAsync(h->gcn_chunks.p, chunks.data(), chunks.size() * sizeof(GcnChunk), cudaMemcpyHostToDevice, h->stream));
    if (!segs.empty()) CK(cudaMemcpyAsync(h->gcn_segs.p, segs.data(), segs.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->gcn_n_chunk = (int64_t)chunks.size(); h->gcn_n_seg = (int64_t)segs.size();
    h->gcn_planned = true;
    return YUE_OK;
}

int yue_gcn_set_events(yue_t* h, int64_t T, const int32_t* ev_user, const int32_t* ev_item) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "call yue_set_interactions first");
    REQUIRE(T == h->T && (T == 0 || (ev_user && ev_item)), YUE_E_ARG, "the events must be the resident log's training events (same number), in file order");
    REQUIRE(h->user_begin == 0 && h->event_base == 0 && !h->have_ev_delta, YUE_E_UNSUPPORTED, "LightGCN needs the whole log on one handle");
    CK(cudaSetDevice(h->device));
    if (int rc = host_indptrs(h)) return rc;
    std::vector<int64_t> per_user((size_t)h->m, 0);
    for (int64_t e = 0; e < T; ++e) {
        REQUIRE(ev_user[e] >= 0 && ev_user[e] < h->m && ev_item[e] >= 0 && ev_item[e] < h->n, YUE_E_ARG, "event " + std::to_string(e) + ": id out of range");
        ++per_user[ev_user[e]];
    }
    for (int64_t u = 0; u < h->m; ++u)
        REQUIRE(per_user[u] == h->h_ev_indptr[u + 1] - h->h_ev_indptr[u], YUE_E_ARG, "user " + std::to_string(u) + ": not the resident log's events");
    CK(h->gcn_ev_user.resize((size_t)std::max<int64_t>(T, 1))); CK(h->gcn_ev_item.resize((size_t)std::max<int64_t>(T, 1)));
    if (T) {
        CK(cudaMemcpyAsync(h->gcn_ev_user.p, ev_user, T * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->gcn_ev_item.p, ev_item, T * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    h->gcn_events = true;
    return YUE_OK;
}

// buffers for L layers and batches of up to `batch` triplets; the variables come back if yue_gcn_finalize replaced them
static int gcn_buffers(yue_t* h, int L, int batch) {
    const size_t M = (size_t)(h->m + h->n), ld = (size_t)h->ld, rows = std::max<size_t>(M * ld, 1);
    cudaStream_t st = h->stream;
    for (int k = 0; k < L; ++k) CK(h->gcn_E[k].resize(rows));
    CK(h->gcn_rinv.resize(std::max<size_t>((size_t)L * M, 1)));
    CK(h->gcn_D[0].resize(rows)); CK(h->gcn_D[1].resize(rows));
    CK(h->gcn_partial.resize(std::max<size_t>((size_t)h->gcn_n_chunk * ld, 1)));
    const bool fresh_adam = h->gcn_am.n < rows || h->gcn_av.n < rows || h->gcn_t == 0;
    CK(h->gcn_am.resize(rows)); CK(h->gcn_av.resize(rows));
    if (fresh_adam) {
        CK(cudaMemsetAsync(h->gcn_am.p, 0, rows * sizeof(float), st)); CK(cudaMemsetAsync(h->gcn_av.p, 0, rows * sizeof(float), st));
        h->gcn_t = 0;
    }
    if (h->gcn_stamp.n < M || h->gcn_stamp_base > 0xF0000000u) {
        CK(h->gcn_stamp.resize(std::max<size_t>(M, 1))); CK(h->gcn_slot_of.resize(std::max<size_t>(M, 1)));
        CK(cudaMemsetAsync(h->gcn_stamp.p, 0, std::max<size_t>(M, 1) * sizeof(uint32_t), st));
        h->gcn_stamp_base = 0;
    }
    CK(h->gcn_slot_of.resize(std::max<size_t>(M, 1)));
    const size_t slots = 3 * (size_t)batch;
    CK(h->gcn_slot_row.resize(slots)); CK(h->gcn_slot_grad.resize(slots * ld)); CK(h->gcn_NB.resize((size_t)(L + 1) * slots * ld));
    CK(h->gcn_trip_loss.resize((size_t)batch));
    if (h->gcn_final) {                       // P, Q hold the propagated tables: the variables come back
        CK(cudaMemcpyAsync(h->P.p, h->gcn_varP.p, (size_t)h->m * ld * sizeof(float), cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(h->Q.p, h->gcn_varQ.p, (size_t)h->n * ld * sizeof(float), cudaMemcpyDeviceToDevice, st));
        h->gcn_final = false;
    }
    return YUE_OK;
}

template <int G, int NC>
static cudaError_t gcn_launch_as(yue_t* h, GcnParams& gp) {
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gcn_steps_kernel<G, NC>, kGcnThreads, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    int ctas = std::min(per_sm, 2) * h->sm_count;
    if (const char* s = getenv("YUE_GCN_CTAS")) ctas = std::max(1, std::min(per_sm * h->sm_count, atoi(s)));
    void* args[] = {&gp};
    return cudaLaunchCooperativeKernel((void*)gcn_steps_kernel<G, NC>, dim3((unsigned)ctas), dim3(kGcnThreads), args, 0, h->stream);
}

static int gcn_launch(yue_t* h, GcnParams& gp) {
    gp.m = h->m; gp.n = h->n; gp.ld = h->ld;
    gp.u_indptr = h->uq_indptr.p; gp.u_items = h->uq_items.p; gp.u_cnt = h->uq_cnt.p;
    gp.t_indptr = h->it_indptr.p; gp.t_users = h->it_users.p; gp.t_cnt = h->it_cnt.p;
    gp.P = h->P.p; gp.Q = h->Q.p;
    for (int k = 0; k < gp.L; ++k) gp.E[k] = h->gcn_E[k].p;
    gp.rinv = h->gcn_rinv.p; gp.D[0] = h->gcn_D[0].p; gp.D[1] = h->gcn_D[1].p; gp.am = h->gcn_am.p; gp.av = h->gcn_av.p;
    gp.stamp = h->gcn_stamp.p; gp.slot_of = h->gcn_slot_of.p; gp.slot_row = h->gcn_slot_row.p; gp.slot_grad = h->gcn_slot_grad.p;
    gp.NB = h->gcn_NB.p; gp.trip_loss = h->gcn_trip_loss.p; gp.loss_out = h->gcn_loss.p;
    gp.chunks = h->gcn_chunks.p; gp.n_chunk = h->gcn_n_chunk; gp.partial = h->gcn_partial.p; gp.arrived = h->gcn_arrived.p;
    gp.segs = h->gcn_segs.p; gp.n_seg = h->gcn_n_seg;
    gp.stamp_base = h->gcn_stamp_base; gp.adam_t = h->gcn_t;
    const bool timing = getenv("YUE_GCN_TIMING") != nullptr;
    if (timing) { CK(h->gcn_phase_ns.resize(32 + 1024)); CK(cudaMemsetAsync(h->gcn_phase_ns.p, 0, (32 + 1024) * sizeof(unsigned long long), h->stream)); gp.phase_ns = h->gcn_phase_ns.p; }
    if (h->ld <= 32) CK(gcn_launch_as<8, 1>(h, gp));
    else if (h->ld <= 64) CK(gcn_launch_as<16, 1>(h, gp));
    else if (h->ld <= 128) CK(gcn_launch_as<32, 1>(h, gp));
    else CK(gcn_launch_as<32, 2>(h, gp));
    ++h->launches;
    if (timing) {
        unsigned long long ns[32];
        CK(cudaMemcpyAsync(ns, h->gcn_phase_ns.p, sizeof(ns), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        const double steps = (double)std::max<int64_t>(1, gp.step_end - gp.step_begin);
        fprintf(stderr, "[yue gcn timing] us per step, work / barrier after it (CTA 0):");
        const char* names[10] = {"fwd1", "fwd2", "fwd3", "fwd4", "batch", "combine", "bwd0+adam", "bwd1", "bwd2", "bwd3"};
        for (int i = 0; i < 10; ++i) if (ns[i] || ns[16 + i]) fprintf(stderr, "  %s %.1f/%.1f", names[i], ns[i] / steps * 1e-3, ns[16 + i] / steps * 1e-3);
        fprintf(stderr, "\n");
        std::vector<unsigned long long> per((size_t)1024);
        CK(cudaMemcpy(per.data(), h->gcn_phase_ns.p + 32, 1024 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        fprintf(stderr, "[yue gcn timing] Adam phase, us per step by CTA:");
        for (int c = 0; c < h->sm_count; ++c) fprintf(stderr, " %.0f", per[c] / steps * 1e-3);
        fprintf(stderr, "\n");
    }
    return YUE_OK;
}

static int gcn_run_steps(yue_t* h, GcnParams& gp, double* loss_out) {
    const int64_t steps = gp.step_end - gp.step_begin;
    CK(h->gcn_loss.resize((size_t)std::max<int64_t>(steps, 1)));
    if (int rc = gcn_launch(h, gp)) return rc;
    h->gcn_stamp_base += (uint32_t)steps; h->gcn_t += steps;
    h->ilv_current = false; h->tc.q_dirty = true;
    std::vector<double> loss((size_t)steps);
    CK(cudaMemcpyAsync(loss.data(), h->gcn_loss.p, steps * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    bool finite = true;
    for (int64_t s = 0; s < steps; ++s) { if (loss_out) loss_out[s] = loss[s]; finite = finite && std::isfinite(loss[s]); }
    if (!finite) return fail(h, YUE_E_NUMERIC, "Loss = NaN or Infinity: current settings does not fit the recommender!");
    return YUE_OK;
}

static int gcn_check(yue_t* h, int n_layers, int64_t batch) {
    REQUIRE(h && h->have_log && h->have_factors, YUE_E_STATE, "log and factors must be set");
    REQUIRE(n_layers >= 1 && n_layers <= kGcnMaxLayers, YUE_E_UNSUPPORTED, "1..4 propagation layers");
    REQUIRE(batch >= 1 && batch <= kGcnMaxBatch, YUE_E_UNSUPPORTED, "batch_size must be in 1..4096");
    CK(cudaSetDevice(h->device));
    if (int rc = q_rowmajor(h)) return rc;
    if (int rc = gcn_plan(h)) return rc;
    return YUE_OK;
}

int yue_gcn_epoch(yue_t* h, int n_layers, int batch_size, double lr, double reg, uint64_t seed, uint32_t epoch,
                  int64_t step_begin, int64_t step_end, double* loss_out) {
    if (int rc = gcn_check(h, n_layers, batch_size)) return rc;
    REQUIRE(h->gcn_events, YUE_E_STATE, "call yue_gcn_set_events first (batches are slices of the log in file order)");
    const int64_t n_steps = (h->T + batch_size - 1) / batch_size;
    if (step_end < 0) step_end = n_steps;
    REQUIRE(step_begin >= 0 && step_begin <= step_end && step_end <= n_steps, YUE_E_ARG, "step range outside the epoch");
    if (step_begin == step_end) return YUE_OK;
    if (int rc = gcn_buffers(h, n_layers, batch_size)) return rc;
    GcnParams gp{};
    gp.L = n_layers; gp.ev_user = h->gcn_ev_user.p; gp.ev_item = h->gcn_ev_item.p; gp.ev_neg = nullptr; gp.T = h->T; gp.batch = batch_size;
    gp.step_begin = step_begin; gp.step_end = step_end; gp.seed = seed; gp.epoch = epoch; gp.lr = (float)lr; gp.reg = (float)reg;
    return gcn_run_steps(h, gp, loss_out);
}

int yue_gcn_apply(yue_t* h, int n_layers, int64_t B, const int32_t* u, const int32_t* i, const int32_t* j,
                  double lr, double reg, double* loss_out) {
    if (int rc = gcn_check(h, n_layers, B)) return rc;
    REQUIRE(u && i && j, YUE_E_ARG, "null argument");
    for (int64_t b = 0; b < B; ++b)
        REQUIRE(u[b] >= 0 && u[b] < h->m && i[b] >= 0 && i[b] < h->n && j[b] >= 0 && j[b] < h->n, YUE_E_ARG, "triplet " + std::to_string(b) + ": id out of range");
    if (int rc = gcn_buffers(h, n_layers, (int)B)) return rc;
    CK(h->tmp_i.resize((size_t)B)); CK(h->tmp_j.resize((size_t)B)); CK(h->gcn_neg.resize((size_t)B));
    CK(cudaMemcpyAsync(h->tmp_i.p, u, B * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->tmp_j.p, i, B * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->gcn_neg.p, j, B * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    GcnParams gp{};
    gp.L = n_layers; gp.ev_user = h->tmp_i.p; gp.ev_item = h->tmp_j.p; gp.ev_neg = h->gcn_neg.p; gp.T = B; gp.batch = (int)B;
    gp.step_begin = 0; gp.step_end = 1; gp.lr = (float)lr; gp.reg = (float)reg;
    return gcn_run_steps(h, gp, loss_out);
}

int yue_gcn_finalize(yue_t* h, int n_layers) {
    if (int rc = gcn_check(h, n_layers, 1)) return rc;
    if (h->gcn_final) return YUE_OK;
    if (int rc = gcn_buffers(h, n_layers, 1)) return rc;
    const size_t ld = (size_t)h->ld;
    CK(h->gcn_varP.resize(std::max<size_t>((size_t)h->m * ld, 1))); CK(h->gcn_varQ.resize(std::max<size_t>((size_t)h->n * ld, 1)));
    GcnParams gp{};
    gp.L = n_layers; gp.forward_only = 1; gp.batch = 1;
    gp.FP = h->gcn_varP.p; gp.FQ = h->gcn_varQ.p;
    if (int rc = gcn_launch(h, gp)) return rc;
    std::swap(h->P, h->gcn_varP); std::swap(h->Q, h->gcn_varQ);      // P, Q <- F; the variables wait in gcn_var*
    h->gcn_final = true;
    h->ilv_current = false; h->tc.q_dirty = true;
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

int yue_gcn_moments(yue_t* h, float* m_users, float* m_tracks, float* v_users, float* v_tracks, int64_t* steps) {
    REQUIRE(h && h->have_factors, YUE_E_STATE, "factors not set");
    CK(cudaSetDevice(h->device));
    const size_t k = (size_t)h->k, ld = (size_t)h->ld, M = (size_t)(h->m + h->n);
    if (steps) *steps = h->gcn_t;
    const bool have = h->gcn_t > 0 && h->gcn_am.n >= M * ld;
    struct { float* dst; const float* src; int64_t rows; } parts[4] = {
        {m_users, h->gcn_am.p, h->m}, {m_tracks, have ? h->gcn_am.p + (size_t)h->m * ld : nullptr, h->n},
        {v_users, h->gcn_av.p, h->m}, {v_tracks, have ? h->gcn_av.p + (size_t)h->m * ld : nullptr, h->n}};
    for (auto& x : parts) {
        if (!x.dst || x.rows == 0) continue;
        if (!have) { std::memset(x.dst, 0, (size_t)x.rows * k * sizeof(float)); continue; }
        CK(cudaMemcpy2DAsync(x.dst, k * sizeof(float), x.src, ld * sizeof(float), k * sizeof(float), (size_t)x.rows, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

// ---- K10: BPR's shipped Adam training (bpr_adam.cuh) ------------------------------------------------------------------
static int bpr_adam_check(yue_t* h, int64_t batch, int64_t negatives, bool need_factors = true) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "interactions not set");
    REQUIRE(h->have_factors || !need_factors, YUE_E_STATE, "factors not set");
    REQUIRE(batch >= 1 && batch <= (1 << 16), YUE_E_ARG, "batch must be in 1..65536");
    REQUIRE(negatives >= 1 && negatives <= (int64_t)kBprAdamPosSlot, YUE_E_ARG, "negatives must be in 1..4095 (slot 4095 draws the positive)");
    REQUIRE(batch * negatives <= (1 << 24), YUE_E_ARG, "batch x negatives must be at most 2^24 triplets");
    REQUIRE(h->user_begin == 0 && h->event_base == 0 && !h->have_ev_delta, YUE_E_UNSUPPORTED, "Adam training needs the whole log on one handle");
    REQUIRE(!h->hot_shared, YUE_E_UNSUPPORTED, "the hot rows are shared (yue_hot_unshare first)");
    REQUIRE(h->m + h->n < ((int64_t)1 << 31), YUE_E_UNSUPPORTED, "more than 2^31 table rows");
    CK(cudaSetDevice(h->device));
    return need_factors ? q_rowmajor(h) : YUE_OK;
}

// scratch for `rows` x `negatives`; Adam's moments (zero when the step counter is)
static int bpr_adam_buffers(yue_t* h, int64_t rows, int64_t negatives) {
    const size_t M = (size_t)(h->m + h->n), ld = (size_t)h->ld, N = (size_t)(rows * negatives), S = 2 * (size_t)rows + N;
    cudaStream_t st = h->stream;
    const bool fresh = h->ba_am.n < M * ld || h->ba_av.n < M * ld || h->ba_t == 0;
    CK(h->ba_am.resize(M * ld)); CK(h->ba_av.resize(M * ld));
    if (fresh) {
        CK(cudaMemsetAsync(h->ba_am.p, 0, M * ld * sizeof(float), st)); CK(cudaMemsetAsync(h->ba_av.p, 0, M * ld * sizeof(float), st));
        h->ba_t = 0;
    }
    if (h->ba_stamp.n < M || h->ba_tag > 0xF0000000u) {
        CK(h->ba_stamp.resize(M)); CK(h->ba_cnt.resize(M));
        CK(cudaMemsetAsync(h->ba_stamp.p, 0, M * sizeof(uint32_t), st)); CK(cudaMemsetAsync(h->ba_cnt.p, 0, M * sizeof(int32_t), st));
        h->ba_tag = 0;
    }
    CK(h->ba_row_base.resize(M)); CK(h->ba_row_size.resize(M));
    CK(h->ba_row_u.resize((size_t)rows)); CK(h->ba_row_i.resize((size_t)rows)); CK(h->ba_row_e.resize((size_t)rows));
    CK(h->ba_row_c.resize((size_t)rows)); CK(h->ba_row_loss.resize((size_t)rows));
    CK(h->ba_ucopy.resize((size_t)rows * ld)); CK(h->ba_ugrad.resize((size_t)rows * ld));
    CK(h->ba_trip_j.resize(N)); CK(h->ba_trip_c.resize(N)); CK(h->ba_trip_loss.resize(N));
    CK(h->ba_slot_row.resize(S)); CK(h->ba_slot_pos.resize(S)); CK(h->ba_list.resize(S)); CK(h->ba_sorted.resize(S));
    CK(h->ba_bump.resize(1));
    return YUE_OK;
}

static BprAdamParams bpr_adam_params(yue_t* h, int64_t rows, int64_t negatives, double reg) {
    BprAdamParams p{};
    p.m = h->m; p.n = h->n; p.T = h->T; p.ld = h->ld; p.B = (int)rows; p.K = (int)negatives;
    p.ev_user = h->ev_user.p; p.ev_items = h->ev_items.p; p.hot_items = h->hot_items.p;
    p.uq_indptr = h->uq_indptr.p; p.uq_items = h->uq_items.p;
    p.P = h->P.p; p.Q = h->Q.p; p.am = h->ba_am.p; p.av = h->ba_av.p;
    p.reg = (float)reg;
    p.row_u = h->ba_row_u.p; p.row_i = h->ba_row_i.p; p.row_e = h->ba_row_e.p;
    p.trip_j = h->ba_trip_j.p; p.trip_c = h->ba_trip_c.p; p.trip_loss = h->ba_trip_loss.p;
    p.ucopy = h->ba_ucopy.p; p.ugrad = h->ba_ugrad.p; p.row_c = h->ba_row_c.p; p.row_loss = h->ba_row_loss.p;
    p.slot_row = h->ba_slot_row.p; p.slot_pos = h->ba_slot_pos.p; p.list = h->ba_list.p; p.sorted = h->ba_sorted.p;
    p.cnt = h->ba_cnt.p; p.row_base = h->ba_row_base.p; p.row_size = h->ba_row_size.p; p.stamp = h->ba_stamp.p; p.bump = h->ba_bump.p;
    return p;
}

template <int G, int NC>
static void bpr_adam_launch_groups(yue_t* h, const BprAdamParams& p) {
    constexpr int GPB = kBprAdamThreads / G;
    const int64_t N = (int64_t)p.B * p.K;
    const int cap = h->sm_count * 8;
    bpr_adam_triplet_kernel<G, NC><<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((N + GPB - 1) / GPB, cap)), kBprAdamThreads, 0, h->stream>>>(p);
    bpr_adam_row_kernel<G, NC><<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((p.B + GPB - 1) / GPB, cap)), kBprAdamThreads, 0, h->stream>>>(p);
}

// one step: six launches on the handle's stream; the loss stays on the device (p.loss_out)
static int bpr_adam_step(yue_t* h, BprAdamParams& p, double lr) {
    const int64_t t = h->ba_t + 1;
    p.lr_t = (float)(lr * std::sqrt(1.0 - std::pow(0.999, (double)t)) / (1.0 - std::pow(0.9, (double)t)));
    p.tag = ++h->ba_tag;
    if (h->ld <= 16) bpr_adam_launch_groups<4, 1>(h, p);
    else if (h->ld <= 32) bpr_adam_launch_groups<8, 1>(h, p);
    else if (h->ld <= 64) bpr_adam_launch_groups<16, 1>(h, p);
    else if (h->ld <= 128) bpr_adam_launch_groups<32, 1>(h, p);
    else bpr_adam_launch_groups<32, 2>(h, p);
    const int64_t S = 2 * (int64_t)p.B + (int64_t)p.B * p.K;
    const unsigned sg = (unsigned)std::max<int64_t>(1, std::min<int64_t>((S + 255) / 256, (int64_t)h->sm_count * 8));
    bpr_adam_alloc_kernel<<<sg, 256, 0, h->stream>>>(p);
    bpr_adam_scatter_kernel<<<sg, 256, 0, h->stream>>>(p);
    bpr_adam_rank_kernel<<<sg, 256, 0, h->stream>>>(p);
    // the dense pass: one float4 per thread, as many CTAs as keep the SMs' load queues full
    const int64_t f4 = (h->m + h->n) * (h->ld / 4);
    const unsigned ug = (unsigned)std::max<int64_t>(1, std::min<int64_t>((f4 + kBprAdamThreads - 1) / kBprAdamThreads, (int64_t)h->sm_count * 32));
    bpr_adam_update_kernel<<<ug, kBprAdamThreads, 0, h->stream>>>(p);
    h->launches += 6;
    CK(cudaGetLastError());
    h->ba_t = t;
    return YUE_OK;
}

// copies `steps` losses back, marks the derived copies of Q stale, refuses a non-finite loss
static int bpr_adam_finish(yue_t* h, int64_t steps, double* loss_out) {
    h->ilv_current = false; h->tc.q_dirty = true;
    std::vector<double> loss((size_t)steps);
    CK(cudaMemcpyAsync(loss.data(), h->ba_loss.p, steps * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    bool finite = true;
    for (int64_t s = 0; s < steps; ++s) { if (loss_out) loss_out[s] = loss[s]; finite = finite && std::isfinite(loss[s]); }
    if (!finite) return fail(h, YUE_E_NUMERIC, "Loss = NaN or Infinity: current settings does not fit the recommender!");
    return YUE_OK;
}

int yue_bpr_adam_sample(yue_t* h, uint64_t seed, int64_t step, int batch, int negatives, int32_t* events_out, int32_t* neg_out) {
    if (int rc = bpr_adam_check(h, batch, negatives, false)) return rc;
    REQUIRE(events_out && neg_out, YUE_E_ARG, "null output");
    REQUIRE(step >= 0 && step <= (int64_t)UINT32_MAX, YUE_E_ARG, "step must be in 0..2^32-1");
    REQUIRE(h->T > 0 && h->T < ((int64_t)1 << 32), YUE_E_UNSUPPORTED, "the log must hold 1..2^32-1 training events");
    if (int rc = ensure_ev_user(h)) return rc;
    const int64_t N = (int64_t)batch * negatives;
    CK(h->tmp_i.resize((size_t)batch)); CK(h->tmp_j.resize((size_t)N));
    BprAdamParams p = bpr_adam_params(h, batch, negatives, 0.0);
    p.seed = seed; p.epoch = (uint32_t)step;
    bpr_adam_sample_kernel<<<(unsigned)std::min<int64_t>((N + 255) / 256, (int64_t)h->sm_count * 16), 256, 0, h->stream>>>(p, h->tmp_i.p, h->tmp_j.p);
    ++h->launches;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(events_out, h->tmp_i.p, batch * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(neg_out, h->tmp_j.p, N * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

int yue_bpr_adam_steps(yue_t* h, int batch, int negatives, double lr, double reg, uint64_t seed, int64_t step_begin,
                       int64_t step_end, double* loss_out) {
    if (int rc = bpr_adam_check(h, batch, negatives)) return rc;
    REQUIRE(step_begin >= 0 && step_begin <= step_end && step_end <= (int64_t)UINT32_MAX + 1, YUE_E_ARG, "step range must lie in 0..2^32");
    REQUIRE(h->T > 0 && h->T < ((int64_t)1 << 32), YUE_E_UNSUPPORTED, "the log must hold 1..2^32-1 training events");
    if (step_begin == step_end) return YUE_OK;
    if (int rc = ensure_ev_user(h)) return rc;
    if (int rc = bpr_adam_buffers(h, batch, negatives)) return rc;
    const int64_t steps = step_end - step_begin;
    CK(h->ba_loss.resize((size_t)steps));
    BprAdamParams p = bpr_adam_params(h, batch, negatives, reg);
    p.seed = seed;
    for (int64_t s = 0; s < steps; ++s) {
        p.epoch = (uint32_t)(step_begin + s);
        p.loss_out = h->ba_loss.p + s;
        if (int rc = bpr_adam_step(h, p, lr)) return rc;
    }
    return bpr_adam_finish(h, steps, loss_out);
}

int yue_bpr_adam_apply(yue_t* h, int64_t B, const int32_t* u, const int32_t* i, const int32_t* j, double lr, double reg,
                       double* loss_out) {
    if (int rc = bpr_adam_check(h, B, 1)) return rc;
    REQUIRE(u && i && j, YUE_E_ARG, "null argument");
    for (int64_t b = 0; b < B; ++b)
        REQUIRE(u[b] >= 0 && u[b] < h->m && i[b] >= 0 && i[b] < h->n && j[b] >= 0 && j[b] < h->n, YUE_E_ARG, "triplet " + std::to_string(b) + ": id out of range");
    if (int rc = bpr_adam_buffers(h, B, 1)) return rc;
    CK(h->ba_fix.resize(3 * (size_t)B));
    int32_t* du = h->ba_fix.p;
    CK(cudaMemcpyAsync(du, u, B * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(du + B, i, B * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(du + 2 * B, j, B * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(h->ba_loss.resize(1));
    BprAdamParams p = bpr_adam_params(h, B, 1, reg);
    p.fix_u = du; p.fix_i = du + B; p.fix_j = du + 2 * B;
    p.loss_out = h->ba_loss.p;
    if (int rc = bpr_adam_step(h, p, lr)) return rc;
    double loss = 0.0;
    if (int rc = bpr_adam_finish(h, 1, &loss)) return rc;
    if (loss_out) *loss_out = loss;
    return YUE_OK;
}

int yue_bpr_adam_moments(yue_t* h, float* m_users, float* m_tracks, float* v_users, float* v_tracks, int64_t* steps) {
    REQUIRE(h && h->have_factors, YUE_E_STATE, "factors not set");
    CK(cudaSetDevice(h->device));
    const size_t k = (size_t)h->k, ld = (size_t)h->ld, M = (size_t)(h->m + h->n);
    if (steps) *steps = h->ba_t;
    const bool have = h->ba_t > 0 && h->ba_am.n >= M * ld;
    struct { float* dst; const float* src; int64_t rows; } parts[4] = {
        {m_users, h->ba_am.p, h->m}, {m_tracks, have ? h->ba_am.p + (size_t)h->m * ld : nullptr, h->n},
        {v_users, h->ba_av.p, h->m}, {v_tracks, have ? h->ba_av.p + (size_t)h->m * ld : nullptr, h->n}};
    for (auto& x : parts) {
        if (!x.dst || x.rows == 0) continue;
        if (!have) { std::memset(x.dst, 0, (size_t)x.rows * k * sizeof(float)); continue; }
        CK(cudaMemcpy2DAsync(x.dst, k * sizeof(float), x.src, ld * sizeof(float), k * sizeof(float), (size_t)x.rows, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

int yue_frob2(yue_t* h, double* p2, double* q2) {
    REQUIRE(h && h->have_factors, YUE_E_STATE, "factors not set");
    CK(cudaSetDevice(h->device));
    if (int rc = q_rowmajor(h)) return rc;
    CK(cudaMemsetAsync(h->scal.p + 1, 0, 2 * sizeof(double), h->stream));
    const int grid = h->sm_count * 8;
    if (h->m) { frob2_kernel<<<grid, 256, 0, h->stream>>>(h->P.p, (size_t)h->m * h->ld, h->scal.p + 1); ++h->launches; }
    frob2_kernel<<<grid, 256, 0, h->stream>>>(h->Q.p, (size_t)h->n * h->ld, h->scal.p + 2); ++h->launches;
    CK(cudaGetLastError());
    double r[2];
    CK(cudaMemcpyAsync(r, h->scal.p + 1, sizeof(r), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (p2) *p2 = r[0];
    if (q2) *q2 = r[1];
    return YUE_OK;
}

int yue_predict(yue_t* h, int64_t user, float* scores_out) {
    REQUIRE(h && h->have_factors, YUE_E_STATE, "factors not set");
    REQUIRE(user >= 0 && user < h->m && scores_out, YUE_E_ARG, "bad user or null output");
    REQUIRE(!h->hot_stale, YUE_E_STATE, "the shared hot rows were trained since the last yue_hot_pull: Q holds stale copies of them");
    CK(cudaSetDevice(h->device));
    if (int rc = q_rowmajor(h)) return rc;
    CK(h->pred.resize(h->n));
    predict_kernel<<<(int)std::min<int64_t>((h->n + 255) / 256, 4096), 256, 0, h->stream>>>(h->P.p, h->Q.p, h->ld, h->k, user, (int)h->n, h->pred.p);
    ++h->launches;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(scores_out, h->pred.p, h->n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

template <int BU, int CAP>
static cudaError_t launch_rank_exact(const RankParams& rp, int splits, cudaStream_t st) {
    const size_t smem = sizeof(RankSmem<BU, CAP>);
    cudaError_t e = cudaFuncSetAttribute(rank_exact_kernel<BU, CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const dim3 grid((unsigned)((rp.B + BU - 1) / BU), (unsigned)splits);
    rank_exact_kernel<BU, CAP><<<grid, 256, smem, st>>>(rp);
    return cudaGetLastError();
}

// A CTA of the exact kernel scans the whole catalog for its 64/128 users, so a handful of users would
// leave the GPU idle (0.17 s for ONE row block at 2 M tracks).  Few rows: split the catalog over
// gridDim.y CTAs per row block, each writes a partial top-N, rank_merge_kernel folds them.
static int yue_rank_exact_device(yue_t* h, const int32_t* d_users, int64_t B, int N, int32_t* d_ids, float* d_scores) {
    RankParams rp{};
    rp.P = h->P.p; rp.Q = h->Q.p; rp.ld = h->ld; rp.n_items = (int)h->n; rp.users = d_users; rp.B = B; rp.N = N;
    rp.uq_indptr = h->uq_indptr.p; rp.uq_items = h->uq_items.p; rp.ids_out = d_ids; rp.scores_out = d_scores;
    const int BU = N <= 32 ? 128 : 64, BI = 16384 / BU;
    const int64_t row_blocks = (B + BU - 1) / BU, ntiles = (h->n + BI - 1) / BI;
    int splits = 1;
    if (row_blocks < h->sm_count) splits = (int)std::max<int64_t>(1, std::min<int64_t>(ntiles / 8, 2 * h->sm_count / row_blocks));
    if (splits > 1) {
        CK(h->rk_part_ids.resize((size_t)B * splits * N)); CK(h->rk_part_scores.resize((size_t)B * splits * N));
        rp.ids_out = h->rk_part_ids.p; rp.scores_out = h->rk_part_scores.p;
    }
    if (N <= 32) CK(launch_rank_exact<128, 64>(rp, splits, h->stream));
    else CK(launch_rank_exact<64, 256>(rp, splits, h->stream));
    ++h->launches;
    if (splits > 1) {
        rank_merge_kernel<<<(unsigned)((B + 7) / 8), 256, 0, h->stream>>>(h->rk_part_ids.p, h->rk_part_scores.p, B, splits, N, d_ids, d_scores);
        ++h->launches;
        CK(cudaGetLastError());
    }
    return YUE_OK;
}

int yue_rank_topn(yue_t* h, const int32_t* users, int64_t B, int N, int algo, int32_t* ids_out, float* scores_out) {
    REQUIRE(h && h->have_log && h->have_factors, YUE_E_STATE, "set interactions and factors first");
    REQUIRE(B >= 0 && (B == 0 || (users && ids_out && scores_out)), YUE_E_ARG, "null argument");
    REQUIRE(N >= 1 && N <= 128, YUE_E_ARG, "N must be in 1..128 (the reference caps it at 100)");
    REQUIRE(algo >= YUE_RANK_EXACT && algo <= YUE_RANK_AUTO, YUE_E_ARG, "unknown algo");
    REQUIRE(!h->hot_stale, YUE_E_STATE, "the shared hot rows were trained since the last yue_hot_pull: Q holds stale copies of them");
    for (int64_t b = 0; b < B; ++b) REQUIRE(users[b] >= 0 && users[b] < h->m, YUE_E_ARG, "user index out of range");
    CK(cudaSetDevice(h->device));
    if (B == 0) return YUE_OK;
    if (int rc = q_rowmajor(h)) return rc;
    CK(h->rk_users.resize(B)); CK(h->rk_ids.resize((size_t)B * N)); CK(h->rk_scores.resize((size_t)B * N));
    CK(cudaMemcpyAsync(h->rk_users.p, users, B * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    int rc;
    const bool tc_ok = rank_tc_supported(h->k, N);
    if (algo == YUE_RANK_TC && !tc_ok) return fail(h, YUE_E_UNSUPPORTED, "tcgen05 ranking needs num.factors <= 128 and N <= 32");
    if (algo == YUE_RANK_TC || (algo == YUE_RANK_AUTO && tc_ok && B >= 256)) {
        rc = rank_tc_run(h->tc, h->stream, h->sm_count, h->P.p, h->Q.p, h->ld, h->k, (int)h->n, h->rk_users.p, B, N,
                         h->uq_indptr.p, h->uq_items.p, h->rk_ids.p, h->rk_scores.p, h->err, h->launches,
                         [&](const int32_t* du, int64_t b, int32_t* di, float* ds) {
                             return yue_rank_exact_device(h, du, b, N, di, ds);
                         });
        if (rc) return rc;
    } else {
        rc = yue_rank_exact_device(h, h->rk_users.p, B, N, h->rk_ids.p, h->rk_scores.p);
        if (rc) return rc;
    }
    h->last_rank_B = B; h->last_rank_N = N;
    CK(cudaMemcpyAsync(ids_out, h->rk_ids.p, (size_t)B * N * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(scores_out, h->rk_scores.p, (size_t)B * N * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return YUE_OK;
}

// ---- ranking metrics on the device (K6) ------------------------------------------------------
int yue_set_test_set(yue_t* h, const int64_t* test_indptr, const int32_t* test_items) {
    REQUIRE(h && test_indptr, YUE_E_ARG, "null argument");
    REQUIRE(h->have_log, YUE_E_STATE, "call yue_set_interactions first (it fixes m and n)");
    REQUIRE(test_indptr[0] == 0, YUE_E_ARG, "indptr must start at 0");
    const int64_t nnz = test_indptr[h->m];
    REQUIRE(nnz == 0 || test_items, YUE_E_ARG, "null item array");
    for (int64_t u = 0; u < h->m; ++u) REQUIRE(test_indptr[u + 1] >= test_indptr[u], YUE_E_ARG, "indptr not monotone");
    CK(cudaSetDevice(h->device));
    CK(h->test_indptr.resize(h->m + 1)); CK(h->test_items.resize(nnz));
    CK(cudaMemcpyAsync(h->test_indptr.p, test_indptr, (h->m + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    if (nnz) CK(cudaMemcpyAsync(h->test_items.p, test_items, nnz * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->have_test = true;
    h->n_test = nnz;
    return YUE_OK;
}

int yue_rank_metrics(yue_t* h, int n_cuts, const int32_t* cuts, double* sums_out, int64_t* distinct_out) {
    REQUIRE(h && cuts && sums_out && distinct_out, YUE_E_ARG, "null argument");
    REQUIRE(h->have_test, YUE_E_STATE, "call yue_set_test_set first");
    REQUIRE(h->last_rank_B > 0, YUE_E_STATE, "no ranking lists on the device: call yue_rank_topn first");
    REQUIRE(n_cuts >= 1 && n_cuts <= kMaxCuts, YUE_E_ARG, "1..8 cut-offs");
    CK(cudaSetDevice(h->device));
    MetricsParams mp{};
    mp.ids = h->rk_ids.p; mp.users = h->rk_users.p; mp.B = h->last_rank_B; mp.N = h->last_rank_N;
    mp.test_indptr = h->test_indptr.p; mp.test_items = h->test_items.p; mp.n_cuts = n_cuts;
    for (int k = 0; k < n_cuts; ++k) {
        REQUIRE(cuts[k] >= 1 && cuts[k] <= mp.N, YUE_E_ARG, "a cut-off must be in 1..N of the last yue_rank_topn");
        mp.cuts[k] = cuts[k];
    }
    mp.seen_words = (h->n + 31) / 32;
    CK(h->met_terms.resize((size_t)n_cuts * 4 * mp.B)); CK(h->met_sums.resize((size_t)n_cuts * 4));
    CK(h->met_seen.resize((size_t)n_cuts * mp.seen_words)); CK(h->met_distinct.resize(n_cuts));
    CK(cudaMemsetAsync(h->met_seen.p, 0, (size_t)n_cuts * mp.seen_words * sizeof(uint32_t), h->stream));
    CK(cudaMemsetAsync(h->met_distinct.p, 0, n_cuts * sizeof(unsigned long long), h->stream));
    mp.terms = h->met_terms.p; mp.seen = h->met_seen.p;
    rank_metrics_kernel<<<(unsigned)((mp.B * 32 + 255) / 256), 256, 0, h->stream>>>(mp);
    metrics_reduce_kernel<<<n_cuts * 4, 1024, 0, h->stream>>>(h->met_terms.p, mp.B, h->met_sums.p);
    popcount_kernel<<<dim3((unsigned)std::min<int64_t>((mp.seen_words + 255) / 256, 1024), (unsigned)n_cuts), 256, 0, h->stream>>>(h->met_seen.p, mp.seen_words, h->met_distinct.p);
    h->launches += 3;
    CK(cudaGetLastError());
    unsigned long long dist[kMaxCuts];
    CK(cudaMemcpyAsync(sums_out, h->met_sums.p, (size_t)n_cuts * 4 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(dist, h->met_distinct.p, n_cuts * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int k = 0; k < n_cuts; ++k) distinct_out[k] = (int64_t)dist[k];
    return YUE_OK;
}

// ---- K7: WRMF half-sweeps (wrmf_als.cuh) -------------------------------------------------------------
static int wrmf_plan_side(yue_t* h, int side, const int64_t* indptr, int64_t rows) {
    std::vector<int32_t> heavy, first, crow;
    std::vector<int64_t> cb, ce;
    for (int64_t r = 0; r < rows; ++r) {
        const int64_t e0 = indptr[r], deg = indptr[r + 1] - e0;
        if (deg <= kWrmfChunk) continue;
        heavy.push_back((int32_t)r);
        first.push_back((int32_t)crow.size());
        const int64_t nch = (deg + kWrmfChunk - 1) / kWrmfChunk;
        for (int64_t c = 0; c < nch; ++c) {
            cb.push_back(e0 + deg * c / nch);
            ce.push_back(e0 + deg * (c + 1) / nch);
            crow.push_back((int32_t)r);
        }
    }
    first.push_back((int32_t)crow.size());
    auto& pl = h->wrmf_plan[side];
    pl.n_heavy = (int)heavy.size();
    pl.n_chunks = (int)crow.size();
    pl.h_chunk_row = crow;
    CK(pl.heavy_rows.resize(heavy.size())); CK(pl.heavy_first.resize(first.size())); CK(pl.chunk_row.resize(crow.size()));
    CK(pl.chunk_begin.resize(cb.size())); CK(pl.chunk_end.resize(ce.size()));
    cudaStream_t st = h->stream;
    if (!heavy.empty()) CK(cudaMemcpyAsync(pl.heavy_rows.p, heavy.data(), heavy.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(pl.heavy_first.p, first.data(), first.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (!crow.empty()) {
        CK(cudaMemcpyAsync(pl.chunk_row.p, crow.data(), crow.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(pl.chunk_begin.p, cb.data(), cb.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(pl.chunk_end.p, ce.data(), ce.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    }
    CK(cudaStreamSynchronize(st));            // host vectors die here
    return YUE_OK;
}

// plays per unique (user, track) pair (WRMF.py:28-33) and the track-major copy of the pairs (record.py:160-163)
static int wrmf_prepare(yue_t* h) {
    if (h->wrmf_ready) return YUE_OK;
    REQUIRE(h->user_begin == 0 && h->event_base == 0 && !h->have_ev_delta, YUE_E_UNSUPPORTED,
            "WRMF needs the whole log on one handle (the track sweep reads every user)");
    REQUIRE(h->nnz < ((int64_t)1 << 31), YUE_E_UNSUPPORTED, "more than 2^31 unique pairs");
    cudaStream_t st = h->stream;
    const int64_t m = h->m, n = h->n, T = h->T, nnz = h->nnz;
    const size_t nz = (size_t)std::max<int64_t>(nnz, 1);
    CK(h->uq_cnt.resize(nz)); CK(h->it_users.resize(nz)); CK(h->it_cnt.resize(nz)); CK(h->it_indptr.resize(n + 1));
    CK(cudaMemsetAsync(h->uq_cnt.p, 0, nz * sizeof(int32_t), st));
    const int grid = h->sm_count * 16;
    DevBuf<uint64_t> k0, k1;
    CubTemp tmp;
    struct Free { std::function<void()> f; ~Free() { f(); } } guard{[&] { k0.release(); k1.release(); tmp.buf.release(); }};
    CK(k0.resize(nz)); CK(k1.resize(nz));
    if (T && m) {
        wrmf_count_kernel<<<grid, 256, 0, st>>>(h->ev_indptr.p, h->ev_items.p, h->uq_indptr.p, h->uq_items.p, m, T, h->hot_items.p, h->uq_cnt.p);
        ++h->launches;
    }
    if (nnz) {
        wrmf_keys_kernel<<<grid, 256, 0, st>>>(h->uq_indptr.p, h->uq_items.p, m, nnz, k0.p);
        size_t need = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, need, k0.p, k1.p, h->uq_cnt.p, h->it_cnt.p, (int)nnz, 0, 64, st);
        CK(tmp.ensure(need));
        size_t tb = tmp.buf.n;
        CK(cub::DeviceRadixSort::SortPairs(tmp.buf.p, tb, k0.p, k1.p, h->uq_cnt.p, h->it_cnt.p, (int)nnz, 0, 64, st));
        ingest_low_words_kernel<<<grid, 256, 0, st>>>(k1.p, nnz, h->it_users.p);
        h->launches += 3;
    }
    ingest_indptr_from_keys_kernel<<<(unsigned)((n + 256) / 256), 256, 0, st>>>(k1.p, nnz, n, h->it_indptr.p);
    ++h->launches;
    CK(cudaGetLastError());
    std::vector<int64_t>& hit = h->h_it_indptr;
    hit.assign((size_t)n + 1, 0);
    CK(cudaMemcpyAsync(hit.data(), h->it_indptr.p, (n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (int rc = host_indptrs(h)) return rc;
    if (int rc = wrmf_plan_side(h, 0, h->h_uq_indptr.data(), m)) return rc;
    if (int rc = wrmf_plan_side(h, 1, hit.data(), n)) return rc;
    h->wrmf_ready = true;
    return YUE_OK;
}

template <int TD, int GB>
static int wrmf_sweep_impl(yue_t* h, int side, int64_t row_begin, int64_t row_end, double reg, double alpha, double* loss_out) {
    constexpr int KP = TD * GB, kWrmfThreads = WrmfShape<TD, GB>::NT;
    constexpr size_t elems = (size_t)TD * TD * kWrmfThreads;
    cudaStream_t st = h->stream;
    const int64_t other_rows = side == 0 ? h->n : h->m;
    if (row_end <= row_begin) { if (loss_out) *loss_out = 0.0; return YUE_OK; }
    const bool want_loss = loss_out != nullptr;
    auto& pl = h->wrmf_plan[side];
    const int n_part = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)h->sm_count * 4, other_rows / 64));
    CK(h->wrmf_part.resize((size_t)n_part * elems)); CK(h->wrmf_G.resize(elems));
    CK(h->wrmf_partA.resize((size_t)pl.n_chunks * elems)); CK(h->wrmf_partb.resize((size_t)pl.n_chunks * KP));
    const size_t sm_acc = wrmf_accum_smem<TD, GB>(), sm_solve = wrmf_solve_smem<TD, GB>();
    CK(cudaFuncSetAttribute(wrmf_gram_kernel<TD, GB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_acc));
    CK(cudaFuncSetAttribute(wrmf_chunk_kernel<TD, GB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_acc));
    CK(cudaFuncSetAttribute(wrmf_chunk_kernel<TD, GB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_acc));
    CK(cudaFuncSetAttribute(wrmf_solve_kernel<TD, GB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_solve));
    CK(cudaFuncSetAttribute(wrmf_solve_kernel<TD, GB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_solve));
    WrmfSide sd{};
    sd.out = side == 0 ? h->P.p : h->Q.p;
    sd.other = side == 0 ? h->Q.p : h->P.p;
    sd.indptr = side == 0 ? h->uq_indptr.p : h->it_indptr.p;
    sd.idx = side == 0 ? h->uq_items.p : h->it_users.p;
    sd.cnt = side == 0 ? h->uq_cnt.p : h->it_cnt.p;
    sd.row_begin = row_begin; sd.rows = row_end; sd.ld = h->ld; sd.k = h->k; sd.reg = reg; sd.alpha = alpha; sd.G = h->wrmf_G.p;
    sd.heavy_rows = pl.heavy_rows.p; sd.heavy_first = pl.heavy_first.p; sd.n_heavy = pl.n_heavy;
    sd.chunk_begin = pl.chunk_begin.p; sd.chunk_end = pl.chunk_end.p; sd.chunk_row = pl.chunk_row.p;
    sd.partA = h->wrmf_partA.p; sd.partb = h->wrmf_partb.p; sd.loss = h->scal.p;
    CK(cudaMemsetAsync(h->scal.p, 0, sizeof(double), st));
    if (other_rows) {
        wrmf_gram_kernel<TD, GB><<<n_part, kWrmfThreads, sm_acc, st>>>(sd.other, other_rows, h->ld, h->k, h->wrmf_part.p);
        wrmf_gram_reduce_kernel<<<(unsigned)((elems + 255) / 256), 256, 0, st>>>(h->wrmf_part.p, n_part, (int)elems, h->wrmf_G.p);
        h->launches += 2;
    } else {
        CK(cudaMemsetAsync(h->wrmf_G.p, 0, elems * sizeof(double), st));
    }
    // rows with 1..32 entries: one warp per row on the d x d Woodbury system (k <= 64, positive weights)
    const bool light = h->wrmf_light && KP <= 64 && alpha > 0.0 && other_rows > 0;
    sd.light_max = light ? kWrmfLightMax : 0;
    if (light) {
        constexpr int KPL = KP <= 64 ? KP : 64;             // (the kernel is not instantiated for k > 64)
        CK(h->wrmf_Binv.resize((size_t)KP * KP));
        const size_t sm_binv = sizeof(double) * (size_t)(KP * (KP + 1) + 2 * KP), sm_light = wrmf_light_smem<KPL>();
        CK(cudaFuncSetAttribute(wrmf_binv_kernel<TD, GB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_binv));
        CK(cudaFuncSetAttribute(wrmf_light_kernel<KPL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_light));
        CK(cudaFuncSetAttribute(wrmf_light_kernel<KPL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_light));
        wrmf_binv_kernel<TD, GB><<<1, 256, sm_binv, st>>>(h->wrmf_G.p, h->k, reg, h->wrmf_Binv.p);
        int lp = 1;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&lp, wrmf_light_kernel<KPL, false>, kWrmfLightWarps * 32, sm_light));
        const int64_t want = (row_end - row_begin + kWrmfLightWarps - 1) / kWrmfLightWarps;
        const int lgrid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)h->sm_count * std::max(lp, 1)));
        if (want_loss) wrmf_light_kernel<KPL, true><<<lgrid, kWrmfLightWarps * 32, sm_light, st>>>(sd, h->wrmf_Binv.p);
        else wrmf_light_kernel<KPL, false><<<lgrid, kWrmfLightWarps * 32, sm_light, st>>>(sd, h->wrmf_Binv.p);
        h->launches += 2;
    }
    const int c0 = (int)(std::lower_bound(pl.h_chunk_row.begin(), pl.h_chunk_row.end(), (int32_t)row_begin) - pl.h_chunk_row.begin());
    const int c1 = (int)(std::lower_bound(pl.h_chunk_row.begin(), pl.h_chunk_row.end(), (int32_t)std::min<int64_t>(row_end, INT32_MAX)) - pl.h_chunk_row.begin());
    sd.chunk_off = c0;
    if (c1 > c0) {
        if (want_loss) wrmf_chunk_kernel<TD, GB, true><<<c1 - c0, kWrmfThreads, sm_acc, st>>>(sd);
        else wrmf_chunk_kernel<TD, GB, false><<<c1 - c0, kWrmfThreads, sm_acc, st>>>(sd);
        ++h->launches;
    }
    int per_sm = 1;
    if (want_loss) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wrmf_solve_kernel<TD, GB, true>, kWrmfThreads, sm_solve));
    else CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wrmf_solve_kernel<TD, GB, false>, kWrmfThreads, sm_solve));
    const int grid = (int)std::min<int64_t>(row_end - row_begin, (int64_t)h->sm_count * std::max(per_sm, 1));
    if (want_loss) wrmf_solve_kernel<TD, GB, true><<<grid, kWrmfThreads, sm_solve, st>>>(sd);
    else wrmf_solve_kernel<TD, GB, false><<<grid, kWrmfThreads, sm_solve, st>>>(sd);
    ++h->launches;
    CK(cudaGetLastError());
    if (side == 1) { h->tc.q_dirty = true; h->ilv_current = false; }
    if (want_loss) {
        CK(cudaMemcpyAsync(loss_out, h->scal.p, sizeof(double), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (!std::isfinite(*loss_out)) return fail(h, YUE_E_NUMERIC, "WRMF loss is not finite");
    }
    return YUE_OK;
}

int yue_wrmf_sweep_rows(yue_t* h, int side, int64_t row_begin, int64_t row_end, double reg, double alpha, double* loss_out) {
    REQUIRE(h, YUE_E_ARG, "null handle");
    REQUIRE(h->have_log && h->have_factors, YUE_E_STATE, "interactions or factors not set");
    REQUIRE(side == 0 || side == 1, YUE_E_ARG, "side must be 0 (users) or 1 (tracks)");
    REQUIRE(reg >= 0.0 && alpha >= 0.0, YUE_E_ARG, "reg and alpha must be non-negative");
    REQUIRE(h->k <= 128, YUE_E_UNSUPPORTED, "WRMF: num.factors must be <= 128");
    const int64_t rows = side == 0 ? h->m : h->n;
    REQUIRE(0 <= row_begin && row_begin <= row_end && row_end <= rows, YUE_E_ARG, "row range outside the table");
    CK(cudaSetDevice(h->device));
    if (int rc = q_rowmajor(h)) return rc;
    if (int rc = wrmf_prepare(h)) return rc;
    if (h->k <= 16) return wrmf_sweep_impl<1, 16>(h, side, row_begin, row_end, reg, alpha, loss_out);
    if (h->k <= 32) return wrmf_sweep_impl<2, 16>(h, side, row_begin, row_end, reg, alpha, loss_out);
    if (h->k <= 64) return h->wrmf_fat ? wrmf_sweep_impl<8, 8>(h, side, row_begin, row_end, reg, alpha, loss_out)
                                       : wrmf_sweep_impl<4, 16>(h, side, row_begin, row_end, reg, alpha, loss_out);
    return wrmf_sweep_impl<8, 16>(h, side, row_begin, row_end, reg, alpha, loss_out);
}

int yue_wrmf_sweep(yue_t* h, int side, double reg, double alpha, double* loss_out) {
    REQUIRE(h && (side == 0 || side == 1), YUE_E_ARG, "null handle or bad side");
    return yue_wrmf_sweep_rows(h, side, 0, side == 0 ? h->m : h->n, reg, alpha, loss_out);
}

int yue_wrmf_pair_counts(yue_t* h, int32_t* uq_counts, int64_t* it_indptr, int32_t* it_users, int32_t* it_counts) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "interactions not set");
    CK(cudaSetDevice(h->device));
    if (int rc = wrmf_prepare(h)) return rc;
    cudaStream_t st = h->stream;
    if (uq_counts && h->nnz) CK(cudaMemcpyAsync(uq_counts, h->uq_cnt.p, h->nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (it_indptr) CK(cudaMemcpyAsync(it_indptr, h->it_indptr.p, (h->n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    if (it_users && h->nnz) CK(cudaMemcpyAsync(it_users, h->it_users.p, h->nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (it_counts && h->nnz) CK(cudaMemcpyAsync(it_counts, h->it_cnt.p, h->nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return YUE_OK;
}

// ---- multi-GPU Q reconciliation ------------------------------------------------------------
static int ensure_snap(yue_t* h) {
    CK(h->Qsnap.resize((size_t)h->n * h->ld));
    CK(h->Qdelta.resize((size_t)h->n * h->ld));
    return YUE_OK;
}
int yue_q_snapshot(yue_t* h) {
    REQUIRE(h && h->have_factors, YUE_E_STATE, "factors not set");
    CK(cudaSetDevice(h->device));
    if (int rc = ensure_snap(h)) return rc;
    if (int rc = q_rowmajor(h)) return rc;
    CK(cudaMemcpyAsync(h->Qsnap.p, h->Q.p, (size_t)h->n * h->ld * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
    h->have_snap = true;
    return YUE_OK;
}
int yue_q_delta_pack(yue_t* h) {
    REQUIRE(h && h->have_factors && h->have_snap, YUE_E_STATE, "call yue_q_snapshot first");
    CK(cudaSetDevice(h->device));
    if (int rc = q_rowmajor(h)) return rc;
    const size_t n4 = (size_t)h->n * h->ld / 4;
    q_delta_pack_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>((const float4*)h->Q.p, (const float4*)h->Qsnap.p, (float4*)h->Qdelta.p, n4);
    ++h->launches;
    CK(cudaGetLastError());
    return YUE_OK;
}
int yue_set_delta_weights(yue_t* h, const float* w) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "call yue_set_interactions first (it fixes n)");
    CK(cudaSetDevice(h->device));
    if (!w) { h->have_delta_w = false; return YUE_OK; }
    CK(h->delta_w.resize(h->n));
    CK(cudaMemcpyAsync(h->delta_w.p, w, h->n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->have_delta_w = true;
    return YUE_OK;
}
int yue_q_delta_apply(yue_t* h) {
    REQUIRE(h && h->have_factors && h->have_snap, YUE_E_STATE, "call yue_q_snapshot first");
    CK(cudaSetDevice(h->device));
    const size_t n4 = (size_t)h->n * h->ld / 4;
    q_delta_apply_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>((float4*)h->Q.p, (float4*)h->Qsnap.p, (const float4*)h->Qdelta.p,
                                                                 h->have_delta_w ? h->delta_w.p : nullptr, h->ld / 4, n4);
    ++h->launches;
    CK(cudaGetLastError());
    h->tc.q_dirty = true;
    h->rowmajor_current = true;
    h->ilv_current = false;
    return YUE_OK;
}
int yue_device_buffer(yue_t* h, int which, void** dev_ptr, size_t* bytes) {
    REQUIRE(h && dev_ptr && bytes, YUE_E_ARG, "null argument");
    REQUIRE(h->have_factors, YUE_E_STATE, "factors not set");
    switch (which) {
        case YUE_BUF_P: *dev_ptr = h->P.p; *bytes = (size_t)h->m * h->ld * sizeof(float); break;
        case YUE_BUF_Q: if (int rc = q_rowmajor(h)) return rc; *dev_ptr = h->Q.p; *bytes = (size_t)h->n * h->ld * sizeof(float); break;
        case YUE_BUF_Q_DELTA:
        case YUE_BUF_Q_SNAPSHOT:
            if (int rc = ensure_snap(h)) return rc;
            *dev_ptr = which == YUE_BUF_Q_DELTA ? h->Qdelta.p : h->Qsnap.p;
            *bytes = (size_t)h->n * h->ld * sizeof(float);
            break;
        default: return fail(h, YUE_E_ARG, "unknown buffer");
    }
    return YUE_OK;
}
int yue_stream(yue_t* h, void** cuda_stream) {
    REQUIRE(h && cuda_stream, YUE_E_ARG, "null argument");
    *cuda_stream = (void*)h->stream;
    return YUE_OK;
}

int yue_comm_unique_id(void* id128) {
    std::string err;
    if (!id128 || !g_nccl.load(err)) { g_create_error = err; return YUE_E_NCCL; }
    return g_nccl.GetUniqueId((NcclUniqueId*)id128) == 0 ? YUE_OK : YUE_E_NCCL;
}
int yue_comm_init(yue_t* h, int nranks, int rank, const void* id128) {
    REQUIRE(h && id128 && nranks >= 1 && rank >= 0 && rank < nranks, YUE_E_ARG, "bad communicator arguments");
    if (!g_nccl.load(h->err)) return YUE_E_NCCL;
    CK(cudaSetDevice(h->device));
    NcclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    const int rc = g_nccl.CommInitRank(&h->comm, nranks, id, rank);
    if (rc != 0) return fail(h, YUE_E_NCCL, std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "error"));
    h->nranks = nranks; h->rank = rank;
    return YUE_OK;
}
int yue_allreduce_q_delta(yue_t* h) {
    REQUIRE(h && h->comm, YUE_E_STATE, "call yue_comm_init first");
    if (int rc = yue_q_delta_pack(h)) return rc;
    const int rc = g_nccl.AllReduce(h->Qdelta.p, h->Qdelta.p, (size_t)h->n * h->ld, /*ncclFloat32*/ 7, /*ncclSum*/ 0, h->comm, h->stream);
    if (rc != 0) return fail(h, YUE_E_NCCL, std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "error"));
    return yue_q_delta_apply(h);
}

// ---- multi-GPU: shared hot rows (one copy per row, on its owner's GPU) + overlapped exchange of the tail --------------
int yue_hot_tracks(yue_t* h, int32_t* tracks_out, int* n_hot) {
    REQUIRE(h && h->have_log && n_hot, YUE_E_STATE, "interactions not set");
    *n_hot = h->n_hot;
    if (tracks_out) for (int s = 0; s < h->n_hot; ++s) tracks_out[s] = h->h_hot_items[(size_t)s];
    return YUE_OK;
}

int yue_set_hot_tracks(yue_t* h, const int32_t* tracks, const int64_t* counts, int n_hot, int64_t total_events) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "call yue_set_interactions first");
    REQUIRE(!h->hot_shared, YUE_E_STATE, "the hot rows are shared (yue_hot_unshare first)");
    REQUIRE(n_hot >= 0 && n_hot <= kHotSlots && (n_hot == 0 || (tracks && counts)) && total_events >= 0, YUE_E_ARG, "bad hot set");
    CK(cudaSetDevice(h->device));
    std::vector<int32_t> cand(tracks, tracks + n_hot), seen(cand);
    std::sort(seen.begin(), seen.end());
    REQUIRE(std::adjacent_find(seen.begin(), seen.end()) == seen.end(), YUE_E_ARG, "a track is listed twice");
    REQUIRE(n_hot == 0 || (seen.front() >= 0 && seen.back() < h->n), YUE_E_ARG, "hot track outside [0, n)");
    if (h->n_hot > 0 && h->T > 0) {             // back to plain ids before the new labels go on
        const int grid = (int)std::min<int64_t>((h->T + 255) / 256, (int64_t)h->sm_count * 16);
        unmark_hot_kernel<<<grid, 256, 0, h->stream>>>(h->ev_items.p, h->T, h->hot_items.p);
        ++h->launches;
        CK(cudaGetLastError());
    }
    h->hot_calibrated_key = 0;
    return install_hot_set(h, cand, std::vector<int64_t>(counts, counts + n_hot), total_events);
}

int yue_hot_table_export(yue_t* h, void* ipc_handle64, void** dev_ptr) {
    REQUIRE(h && h->have_log, YUE_E_STATE, "call yue_set_interactions first");
    CK(cudaSetDevice(h->device));
    CK(h->hotQ.resize(kHotTableFloats + (size_t)(kHotCandidates + 1) * kHotCandidateStep * 64));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (ipc_handle64) CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)ipc_handle64, h->hotQ.p));
    if (dev_ptr) *dev_ptr = h->hotQ.p;
    return YUE_OK;
}

int yue_hot_table_open(yue_t* h, const void* ipc_handle64, void** dev_ptr) {
    REQUIRE(h && ipc_handle64 && dev_ptr, YUE_E_ARG, "null argument");
    CK(cudaSetDevice(h->device));
    cudaIpcMemHandle_t hd;
    memcpy(&hd, ipc_handle64, sizeof(hd));
    const std::string key((const char*)ipc_handle64, sizeof(hd));
    for (size_t x = 0; x < h->ipc_keys.size(); ++x)
        if (h->ipc_keys[x] == key) { *dev_ptr = h->ipc_opened[x]; return YUE_OK; }     // the peer's table outlives its logs
    void* p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
    h->ipc_opened.push_back(p);
    h->ipc_keys.push_back(key);
    *dev_ptr = p;
    return YUE_OK;
}

int yue_enable_peer(yue_t* h, int peer_device) {
    REQUIRE(h, YUE_E_ARG, "null handle");
    CK(cudaSetDevice(h->device));
    if (peer_device == h->device) return YUE_OK;
    int can = 0;
    CK(cudaDeviceCanAccessPeer(&can, h->device, peer_device));
    REQUIRE(can, YUE_E_UNSUPPORTED, "device " + std::to_string(h->device) + " cannot access device " + std::to_string(peer_device) + " as a peer");
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return YUE_OK; }
    CK(e);
    return YUE_OK;
}

template <int V>
static cudaError_t launch_hot_gather_shared(yue_t* h) {
    hot_gather_shared_kernel<V><<<(h->n_hot + 7) / 8, 256, 0, h->stream>>>(h->Q.p, h->hot_base.p, h->hot_items.p, h->hot_dx.p, h->n_hot, h->ld,
                                                                           h->hot_nranks, h->hot_rank, hot_plane_floats(h->n_hot + kHotExtra));
    return cudaGetLastError();
}
template <int V>
static cudaError_t launch_hot_pull_shared(yue_t* h) {
    hot_pull_shared_kernel<V><<<(h->n_hot + 7) / 8, 256, 0, h->stream>>>(h->Q.p, h->hot_base.p, h->hot_items.p, h->hot_dx.p, h->n_hot, h->ld,
                                                                         hot_plane_floats(h->n_hot + kHotExtra));
    return cudaGetLastError();
}

int yue_hot_share(yue_t* h, int nranks, int rank, void* const* tables) {
    REQUIRE(h && h->have_log && h->have_factors, YUE_E_STATE, "set interactions and factors first");
    REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks && tables, YUE_E_ARG, "bad rank arguments");
    REQUIRE(h->ld == 32 || h->ld == 64 || h->ld == 128, YUE_E_UNSUPPORTED, "shared hot rows need num.factors = 32, 64 or 128");
    REQUIRE((uint64_t)h->n * h->ld * 4 < ((uint64_t)1 << 32), YUE_E_UNSUPPORTED, "catalog too large for the blocked kernel");
    CK(cudaSetDevice(h->device));
    if (int rc = q_rowmajor(h)) return rc;
    h->hot_nranks = nranks; h->hot_rank = rank;
    if (h->n_hot > 0) {
        CK(h->hotQ.resize(kHotTableFloats + (size_t)(kHotCandidates + 1) * kHotCandidateStep * 64));
        std::vector<unsigned long long> base((size_t)h->n_hot);
        for (int s = 0; s < h->n_hot; ++s) {
            const int owner = s % nranks;
            void* t = owner == rank ? (void*)h->hotQ.p : tables[owner];
            REQUIRE(t, YUE_E_ARG, "table of rank " + std::to_string(owner) + " is NULL");
            base[(size_t)s] = (unsigned long long)(uintptr_t)t;
        }
        CK(h->hot_base.resize(h->n_hot));
        CK(cudaMemcpyAsync(h->hot_base.p, base.data(), base.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, h->stream));
        switch (blk_width(h->ld)) {
            case 1: CK(launch_hot_gather_shared<1>(h)); break;
            case 2: CK(launch_hot_gather_shared<2>(h)); break;
            default: CK(launch_hot_gather_shared<4>(h)); break;
        }
        ++h->launches;
        CK(cudaStreamSynchronize(h->stream));       // base dies here; the caller's barrier then covers every rank's rows
    }
    h->hot_shared = true;
    return YUE_OK;
}

int yue_hot_pull(yue_t* h) {
    REQUIRE(h && h->hot_shared, YUE_E_STATE, "the hot rows are not shared");
    CK(cudaSetDevice(h->device));
    if (h->n_hot > 0) {
        switch (blk_width(h->ld)) {
            case 1: CK(launch_hot_pull_shared<1>(h)); break;
            case 2: CK(launch_hot_pull_shared<2>(h)); break;
            default: CK(launch_hot_pull_shared<4>(h)); break;
        }
        ++h->launches;
        h->tc.q_dirty = true;
    }
    CK(cudaStreamSynchronize(h->stream));
    h->hot_stale = false;
    return YUE_OK;
}

int yue_hot_unshare(yue_t* h) {
    if (int rc = yue_hot_pull(h)) return rc;
    h->hot_shared = false;
    return YUE_OK;
}

int yue_set_sgd_concurrency(yue_t* h, int n_warps, int n_ctas) {
    REQUIRE(h && n_warps >= 0 && n_ctas >= 0, YUE_E_ARG, "negative concurrency");
    h->sgd_warps_forced = n_warps;
    h->sgd_ctas_forced = std::min(n_ctas, h->sm_count);
    return YUE_OK;
}

static int ensure_exchange(yue_t* h) {
    if (int rc = ensure_snap(h)) return rc;
    CK(h->Qown.resize((size_t)h->n * h->ld));
    if (!h->stream2) {
        CK(cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&h->ev_pack, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_red, cudaEventDisableTiming));
    }
    return YUE_OK;
}
int yue_stream2(yue_t* h, void** cuda_stream) {
    REQUIRE(h && cuda_stream, YUE_E_ARG, "null argument");
    CK(cudaSetDevice(h->device));
    if (int rc = ensure_exchange(h)) return rc;
    *cuda_stream = (void*)h->stream2;
    return YUE_OK;
}
int yue_q_exchange_begin(yue_t* h) {
    REQUIRE(h && h->have_factors && h->have_snap, YUE_E_STATE, "call yue_q_snapshot first");
    REQUIRE(!h->exchange_pending, YUE_E_STATE, "an exchange is already in flight (yue_q_exchange_finish first)");
    CK(cudaSetDevice(h->device));
    if (int rc = ensure_exchange(h)) return rc;
    if (int rc = q_rowmajor(h)) return rc;
    const size_t n4 = (size_t)h->n * h->ld / 4;
    q_exchange_pack_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>((const float4*)h->Q.p, (const float4*)h->Qsnap.p, (float4*)h->Qdelta.p,
                                                                   (float4*)h->Qown.p, n4);
    ++h->launches;
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev_pack, h->stream));
    CK(cudaStreamWaitEvent(h->stream2, h->ev_pack, 0));
    h->exchange_pending = true;
    return YUE_OK;
}
int yue_q_exchange_reduce(yue_t* h) {
    REQUIRE(h && h->comm, YUE_E_STATE, "call yue_comm_init first");
    REQUIRE(h->exchange_pending, YUE_E_STATE, "call yue_q_exchange_begin first");
    CK(cudaSetDevice(h->device));
    const int rc = g_nccl.AllReduce(h->Qdelta.p, h->Qdelta.p, (size_t)h->n * h->ld, /*ncclFloat32*/ 7, /*ncclSum*/ 0, h->comm, h->stream2);
    if (rc != 0) return fail(h, YUE_E_NCCL, std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "error"));
    return YUE_OK;
}
int yue_q_exchange_reduce_peers(yue_t* h, int nranks, void* const* deltas) {
    REQUIRE(h && h->exchange_pending, YUE_E_STATE, "call yue_q_exchange_begin first");
    REQUIRE(nranks >= 1 && nranks <= 8 && deltas, YUE_E_ARG, "1..8 ranks");
    CK(cudaSetDevice(h->device));
    CK(h->Qsum.resize((size_t)h->n * h->ld));
    PeerDeltas src{};
    src.n = nranks;
    for (int r = 0; r < nranks; ++r) {
        src.p[r] = (const float4*)(deltas[r] ? deltas[r] : (void*)h->Qdelta.p);
    }
    const size_t n4 = (size_t)h->n * h->ld / 4;
    q_exchange_sum_peers_kernel<<<h->sm_count * 4, 256, 0, h->stream2>>>(src, (float4*)h->Qsum.p, n4);
    ++h->launches;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream2));     // the caller's barrier then tells every rank that its delta has been read
    h->sum_in_qsum = true;
    return YUE_OK;
}
int yue_q_exchange_finish(yue_t* h, int quiescent) {
    REQUIRE(h && h->exchange_pending, YUE_E_STATE, "no exchange in flight");
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(h->ev_red, h->stream2));
    CK(cudaStreamWaitEvent(h->stream, h->ev_red, 0));
    const size_t n4 = (size_t)h->n * h->ld / 4;
    q_exchange_apply_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>((float4*)h->Q.p, (float4*)h->Qsnap.p,
                                                                    (const float4*)(h->sum_in_qsum ? h->Qsum.p : h->Qdelta.p), (const float4*)h->Qown.p, h->have_delta_w ? h->delta_w.p : nullptr, h->ld / 4, n4, quiescent != 0);
    ++h->launches;
    CK(cudaGetLastError());
    h->exchange_pending = false;
    h->sum_in_qsum = false;
    h->tc.q_dirty = true;
    h->ilv_current = false;
    return YUE_OK;
}

// ---- result lines of evalRanking (host code) --------------------------------------------------------------------------
int yue_result_lines(const char* user_blob, const int64_t* user_off, const char* track_blob, const int64_t* track_off,
                     int64_t n_tracks, const int32_t* ids, const uint8_t* hits, int64_t B, int N,
                     char* out, int64_t out_cap, int64_t* out_len) {
    if (!user_blob || !user_off || !track_blob || !track_off || !ids || !hits || !out_len || B < 0 || N < 0 || n_tracks < 0) {
        g_create_error = "yue_result_lines: null or negative argument";
        return YUE_E_ARG;
    }
    const size_t nth = B < 4096 ? 1 : std::min<size_t>(16, std::max(1u, std::thread::hardware_concurrency()));
    std::vector<int64_t> first(nth + 1, 0);
    std::vector<int> bad(nth, 0);
    auto share = [&](size_t t) { return B * (int64_t)t / (int64_t)nth; };
    auto line_len = [&](int64_t b) {
        int64_t len = user_off[b + 1] - user_off[b] + 2;                   // name ':' ... '\n'
        for (int r = 0; r < N; ++r) {
            const int32_t id = ids[b * N + r];
            if (id < 0) continue;
            if (id >= n_tracks) return (int64_t)-1;
            len += track_off[id + 1] - track_off[id] + (hits[b * N + r] ? 1 : 0);
        }
        return len;
    };
    auto run = [&](auto fn) {
        std::vector<std::thread> th;
        for (size_t t = 1; t < nth; ++t) th.emplace_back(fn, t);
        fn(0);
        for (auto& x : th) x.join();
    };
    run([&](size_t t) {                                                     // pass 1: bytes per thread's share
        int64_t sum = 0;
        for (int64_t b = share(t); b < share(t + 1); ++b) { const int64_t l = line_len(b); if (l < 0) { bad[t] = 1; return; } sum += l; }
        first[t + 1] = sum;
    });
    for (size_t t = 0; t < nth; ++t) if (bad[t]) { g_create_error = "yue_result_lines: a ranked id is outside the catalog"; return YUE_E_ARG; }
    for (size_t t = 0; t < nth; ++t) first[t + 1] += first[t];
    *out_len = first[nth];
    if (!out || out_cap < first[nth]) { g_create_error = "yue_result_lines: output buffer too small"; return YUE_E_ARG; }
    run([&](size_t t) {                                                     // pass 2: the bytes
        char* w = out + first[t];
        for (int64_t b = share(t); b < share(t + 1); ++b) {
            const int64_t ul = user_off[b + 1] - user_off[b];
            memcpy(w, user_blob + user_off[b], (size_t)ul); w += ul;
            *w++ = ':';
            for (int r = 0; r < N; ++r) {
                const int32_t id = ids[b * N + r];
                if (id < 0) continue;
                const int64_t tl = track_off[id + 1] - track_off[id];
                memcpy(w, track_blob + track_off[id], (size_t)tl); w += tl;
                if (hits[b * N + r]) *w++ = '*';
            }
            *w++ = '\n';
        }
    });
    return YUE_OK;
}

// ---- measurement hooks ---------------------------------------------------------------------
int yue_timer_start(yue_t* h) { CK(cudaSetDevice(h->device)); CK(cudaEventRecord(h->ev0, h->stream)); return YUE_OK; }
int yue_timer_stop(yue_t* h, float* ms) {
    REQUIRE(ms, YUE_E_ARG, "null argument");
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(h->ev1, h->stream));
    CK(cudaEventSynchronize(h->ev1));
    CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    return YUE_OK;
}
int yue_rank_stats(yue_t* h, int64_t* fallback_rows, int64_t* spilled_rows) {
    REQUIRE(h, YUE_E_ARG, "null argument");
    if (fallback_rows) *fallback_rows = h->tc.last_fail;
    if (spilled_rows) *spilled_rows = h->tc.last_spill;
    return YUE_OK;
}
int yue_launch_count(yue_t* h, int64_t* n) { REQUIRE(h && n, YUE_E_ARG, "null argument"); *n = h->launches; return YUE_OK; }
int yue_flush_l2(yue_t* h) {
    CK(cudaSetDevice(h->device));
    const size_t bytes = std::max<size_t>(h->l2_bytes * 2, (size_t)256 << 20);
    CK(h->l2buf.resize(bytes));
    CK(cudaMemsetAsync(h->l2buf.p, 0x5a, bytes, h->stream));
    return YUE_OK;
}

