// yk_engine.cu -- libykgpu.so: host side of the engine + the C ABI of include/ykgpu.h.
//
// One scheduling cycle (yk_cycle) =
//   host  : Orderer (yk_orderer.hpp) produces the next batch of asks in schedule()-pass order
//   device: key kernel (float64 node score) -> stable radix sort by key over NodeID-rank order
//           -> gather into the sorted SoA view -> fused sweep kernel (batch x all nodes) -> fit bitmaps
//   commit: ordered, exact: ask i takes the minimum (key, NodeID) over {clean nodes whose bitmap bit is set}
//           U {nodes already committed to in this batch, re-scored}; see DESIGN.md "ordered commit".
// There is no CPU fallback for the sweep: without a CUDA device yk_create fails with YK_ERR_CUDA.
#include "../../include/ykgpu.h"

#include <cub/device/device_radix_sort.cuh>
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>
#include <x86intrin.h>

#include "yk_kernels.cuh"
#include "yk_lattice.cuh"
#include "yk_uniform.cuh"
#include "yk_commit.hpp"
#include "yk_lattice_host.hpp"
#include "yk_orderer.hpp"

namespace {

#ifndef YK_NPT
#define YK_NPT 2
#endif
constexpr int NPT = YK_NPT;       // sorted-node positions per sweep thread
constexpr int AC = 128;           // asks per sweep CTA chunk
constexpr int NODE_TILE = YK_SWEEP_THREADS * NPT;

inline size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

template <typename T>
struct Dev {
    T* p = nullptr; size_t n = 0;
    cudaError_t alloc(size_t count) {
        free();
        n = count;
        return cudaMalloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
    }
    void free() { if (p) cudaFree(p); p = nullptr; n = 0; }
    ~Dev() { free(); }
};
template <typename T>
struct Pin {
    T* p = nullptr; size_t n = 0;
    cudaError_t alloc(size_t count) {
        free();
        n = count;
        cudaError_t e = cudaMallocHost((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) memset(p, 0, std::max<size_t>(count, 1) * sizeof(T));
        return e;
    }
    void free() { if (p) cudaFreeHost(p); p = nullptr; n = 0; }
    T& operator[](size_t i) { return p[i]; }
    const T& operator[](size_t i) const { return p[i]; }
    ~Pin() { free(); }
};


double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// A helper thread that fills and launches the NEXT batch while the caller's thread commits the current one
// (the orderer state is only touched by one of the two at a time: fork before the commit, join after it).
struct Worker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, busy = false, quit = false;
    int device = 0;
    void start(int dev) {
        device = dev;
        th = std::thread([this] {
            cudaSetDevice(device);
            std::unique_lock<std::mutex> lk(m);
            for (;;) {
                cv.wait(lk, [this] { return has_job || quit; });
                if (quit) return;
                has_job = false;
                lk.unlock();
                job();
                lk.lock();
                busy = false;
                cv.notify_all();
            }
        });
    }
    void submit(std::function<void()> f) {
        std::lock_guard<std::mutex> lk(m);
        job = std::move(f); has_job = true; busy = true;
        cv.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [this] { return !busy; });
    }
    void stop() {
        if (!th.joinable()) return;
        { std::lock_guard<std::mutex> lk(m); quit = true; cv.notify_all(); }
        th.join();
    }
};

// One in-flight batch: its asks, device / pinned buffers and read-back events.  Two slots let the sweep and the
// read-back of batch k+1 run while the host commits batch k (both against the same epoch view, see run loop).
struct Slot {
    std::vector<uint32_t> asks;     // the batch, in commit order
    std::vector<uint32_t> reps;     // one representative ask per distinct signature = the rows the device sweeps
    std::vector<uint32_t> row_of;   // batch entry -> row
    yk::Orderer::Snap snap;
    Dev<uint32_t> d_batch, d_fit;
    Pin<uint32_t> h_batch, h_fit;
    Pin<int> h_err;                 // P2P: copy of the device error word after the flag waits
    std::vector<cudaEvent_t> ev;
    cudaEvent_t ev_s0 = nullptr, ev_s1 = nullptr;
    int B = 0, R = 0, W = 0, chunk = 0, nchunks = 0, rows = 0;   // B asks, R rows (all ranks), rows = this rank's shard
    uint32_t last_value = 0;        // P2P: sequence value signalled when this slot's previous content was published
};

// Signature numbers, kept up to date as asks are upserted: equal number <=> equal predicate signature (request vector,
// tolerations, required / forbidden labels, node name).  Open addressing on the 64-bit signature hash; a hit is always
// confirmed on the full signature of the entry's representative ask.  (A representative that was later overwritten with
// another signature just stops matching: the signature then gets a second number -- an extra swept row, never a wrong
// merge.)  Rebuilt from the present asks when it has handed out more than four numbers per ask slot.
struct SigTable {
    struct Ent { uint64_t h; uint32_t rep, id; };
    static constexpr uint32_t FREE = 0xFFFFFFFFu, TOMB = 0xFFFFFFFEu;
    std::vector<Ent> tab;
    std::vector<uint32_t> rep_slot;   // ask -> 1 + the slot it represents, 0 when it represents none
    uint32_t n = 0;
    void reset(size_t asks) {
        size_t cap = 1024;
        while (cap < 4 * asks) cap <<= 1;
        tab.assign(cap, Ent{0, FREE, 0});
        rep_slot.assign(asks, 0);
        n = 0;
    }
    // the ask's row is about to be overwritten: a number it represents is never handed out again (the asks that hold it
    // stay equal among themselves; the signature gets a fresh number next time it is seen)
    void retire(uint32_t ask) {
        if (rep_slot[ask]) { tab[rep_slot[ask] - 1].rep = TOMB; rep_slot[ask] = 0; }
    }
    uint32_t get(const yk::CommitTables& t, uint64_t h, uint32_t ask) {
        const size_t mask = tab.size() - 1;
        size_t x = (size_t)(h ^ (h >> 29)) & mask;
        for (;;) {
            Ent& e = tab[x];
            if (e.rep == FREE) { e.h = h; e.rep = ask; e.id = n++; rep_slot[ask] = (uint32_t)x + 1; return e.id; }
            if (e.rep != TOMB && e.h == h && yk::same_signature(t, e.rep, ask)) return e.id;
            x = (x + 1) & mask;
        }
    }
};

}  // namespace

struct yk_engine {
    std::mutex mu;
    yk_config cfg{};
    int D = 0;
    uint32_t maxN = 0, maxA = 0, maxP = 0, maxQ = 0, batch = 0;
    std::string err;
    yk_stats_t st{};
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    YkWeights w{};

    // ---- host tables (pinned: they are the H2D sources) ----
    Pin<int64_t> n_total, n_avail;             // [D][maxN]
    Pin<uint64_t> n_taint, n_label;
    Pin<uint32_t> n_flags;                     // bit0 schedulable, bit1 reserved (0 when absent)
    std::vector<uint32_t> n_rank;
    std::vector<uint8_t> n_present;
    uint32_t n_hi = 0;                         // 1 + highest node index in use
    bool nodes_stale = true, rank_stale = true;
    Pin<uint32_t> by_rank; uint32_t nlive = 0;
    bool ranks_unique = true;                // no two live nodes share a NodeID rank (checked where by_rank is rebuilt)

    Pin<int64_t> a_req;                        // [D][maxA]
    Pin<uint64_t> a_tol, a_need, a_deny;
    Pin<uint32_t> a_node;
    std::vector<int32_t> a_prio;
    std::vector<int64_t> a_create;
    std::vector<uint64_t> a_sig;    // signature hash of each ask's predicate inputs (yk::ask_signature)
    yk::RowShare share;
    bool share_rows = true;
    uint64_t split_min_pairs = 1ull << 25;   // multi-GPU: batches with fewer (row,node) pairs are swept whole on every rank
    std::vector<uint32_t> a_app, a_flags, a_gang, a_bound;
    std::vector<uint8_t> a_state;              // yk::ST_*, ST_ABSENT when not present
    uint32_t a_hi = 0;
    bool asks_stale = true;

    std::vector<uint32_t> p_queue; std::vector<int64_t> p_submit, p_alloc; std::vector<uint8_t> p_present;
    uint32_t nq = 0;
    std::vector<uint32_t> q_parent; std::vector<int64_t> q_guar, q_max, q_alloc; std::vector<uint8_t> q_sort;
    std::vector<int32_t> q_prio_offset; std::vector<uint8_t> q_prio_fence;   // queue properties priority.offset / priority.policy=fence
    std::vector<uint32_t> p_user, ul_queue, ul_user; std::vector<int64_t> ul_max, ul_alloc; uint32_t n_ul = 0;   // user / group limits

    // ---- device ----
    Dev<int64_t> d_total, d_avail; Dev<uint64_t> d_taint, d_label; Dev<uint32_t> d_flags, d_by_rank;
    Dev<int64_t> d_areq; Dev<uint64_t> d_atol, d_aneed, d_adeny; Dev<uint32_t> d_anode;
    Dev<uint64_t> d_key_in, d_key_out; Dev<uint32_t> d_val_in, d_val_out;
    Dev<uint8_t> d_cub; size_t cub_bytes = 0;
    Dev<int64_t> d_scap; Dev<uint64_t> d_staint, d_slabel; Dev<uint32_t> d_snode;
    Dev<int> d_flag;
    Slot slot[2];
    Worker worker;
    std::vector<uint32_t> pending;           // asks of the current cycle
    yk_stats_t wst{};                        // counters written by the worker thread, merged at join
    Dev<uint32_t> d_dirty_nodes; Dev<int64_t> d_dirty_vals; Dev<double> d_scores;
    size_t Wmax = 0;

    // pinned staging
    Pin<uint32_t> h_snode, h_dirty_nodes; Pin<uint64_t> h_skey; Pin<int64_t> h_dirty_vals;
    Pin<int> h_flag; Pin<double> h_scores;

    // ordered commit (host logic, csrc/yk_commit.hpp): working copy of the nodes, touched-node index, epoch state
    yk::Committer cm;
    Pin<uint32_t> h_order[2]; int cur = 0;   // node order (ascending (score, NodeID)), double-buffered
    Dev<uint32_t> d_order;
    int epochW = 0;                          // words per fit row in the current epoch
    uint32_t epoch_limit = 8192;             // an epoch ends before its touched-node count would pass this
    uint32_t epoch_floor = 8192, epoch_env = 0;
    bool prof = false;                       // YK_PROFILE_COMMIT: TSC split of the commit loop into st.dbg2[]
    bool no_spec = false;                    // debugging: never launch batch k+1 before batch k is committed
    int slots = 296;                         // resident sweep CTAs on this device (SMs x occupancy)

    yk::Orderer ord;
    // epoch rows: when the cycle's pending asks have few distinct predicate signatures, every signature is swept ONCE per
    // epoch (one launch, one read-back) and the batches of the epoch only index into those rows -- no per-batch device work
    static constexpr uint32_t EP_MAX = 1024;
    bool ep_rows = false; uint32_t ep_n = 0; bool ep_uploaded = false, ep_landed = true;
    std::vector<uint32_t> ep_reps;
    Dev<uint32_t> ep_d_batch, ep_d_fit; Pin<uint32_t> ep_h_batch, ep_h_fit;
    cudaEvent_t ep_ev = nullptr, ep_s0 = nullptr, ep_s1 = nullptr;
    uint32_t n_shapes = 0, n_sigs = 0;
    SigTable sigs; std::vector<uint32_t> ep_local, ep_seen; uint32_t ep_stamp = 0;
    // device-resident ordered commit (yk_lattice.h): node records, ping-pong node order, per-batch staging
    bool lt_allowed = true;                  // !YK_FLAG_HOST_COMMIT, single GPU
    int lt_force = 0;                        // YK_FLAG_DEVICE_COMMIT / YK_COMMIT=device: every eligible cycle commits on the device
    bool lt_auto = false;                    // the default: eligible cycles whose order is made of long uniform runs commit on the device
    bool lt_active = false;                  // this cycle runs (so far) on the device commit
    bool cycle_has_gang = false;             // some pending ask of this cycle is a gang member
    bool order_enqueued = false;             // device_order() of this cycle is already on the stream
    int lt_RS = 0; size_t lt_smem = 0;
    Dev<int64_t> d_rec; Dev<yklt::Ent> d_ord[2]; Dev<int> d_lt_cur, d_lt_hdr; Dev<int64_t> d_lt_ub;
    Dev<uint32_t> d_rank, d_lt_asks, d_lt_meta, d_lt_shp, d_lt_sig, d_lt_res;
    Dev<long long> d_lt_prof; bool lt_prof = false; uint64_t lt_total_subruns = 0;   // YK_PROFILE_LATTICE: SM clocks per kernel phase, printed by yk_destroy
    Pin<uint32_t> h_lt_asks, h_lt_meta, h_lt_shp, h_lt_sig, h_lt_res; Pin<int> h_lt_hdr; Pin<int64_t> h_lt_ub;
    std::vector<uint32_t> a_shape, a_sigid;
    std::vector<uint8_t> a_cause;               // per ask: 0, ST_SLOWPATH or ST_INVALID (yk::Tables::a_cause), kept by yk_asks_upsert
    cudaEvent_t ev_l0 = nullptr, ev_l1 = nullptr;
    // uniform runs (yk_uniform.h): allocated on first use; element buffers hold UN_EMAX generated elements
    bool hp_on = false; double hp[8] = {0, 0, 0, 0, 0, 0, 0, 0}; uint64_t hp_n = 0;
    bool un_hint = false;                       // this cycle's pending asks look like long uniform runs (auto commit: size the first batch for it)
    bool lt_plan_ready = false;                 // h_lt_meta/shp/sig and un_segs already describe slot[0]'s batch (built by the commit choice)
    bool un_alloc = false, un_ord_stale = false;   // un_ord_stale: uniform runs moved nodes since d_ord was last written
    const uint32_t* lt_shape_ids = nullptr;     // per ask: a number equal for equal request vectors (a_shape, or a_sigid: finer, still exact)
    int un_min = 2048;                          // shortest run that takes the uniform path (YK_UNIFORM_MIN)
    Dev<unsigned long long> d_un_ekey[2], d_un_bk, d_un_rkey[2], d_un_rrn[2];
    Dev<uint32_t> d_un_enode[2], d_un_cnt;
    Dev<ykun::Globals> d_un_g; Pin<ykun::Globals> h_un_g;
    Dev<uint8_t> d_un_cub; size_t un_cub_bytes = 0;
    std::vector<ykun::Segment> un_segs;
    Dev<uint32_t> pre_q; Dev<int64_t> pre_v; Dev<int32_t> pre_o;   // yk_preemption_search staging, grown on demand
    yk_allgather_fn xfn = nullptr; void* xctx = nullptr;
    // peer-to-peer exchange (see yk_peer_export): peers' slot buffers and sync blocks, mapped through CUDA IPC
    bool p2p = false;
    uint32_t seq = 0;
    Dev<uint32_t> d_sync;                    // [32]: ready[slot][rank] at slot*8+rank, consumed[slot][rank] at 16+slot*8+rank
    uint32_t* peer_fit[2][8] = {};
    uint32_t* peer_sync[8] = {};
    bool peer_open[8] = {};

    int fail(int code, const std::string& m) { err = m; return code; }
    int cuda_fail(cudaError_t e, const char* what) {
        err = std::string(what) + ": " + cudaGetErrorString(e);
        return YK_ERR_CUDA;
    }
};

#define CK(call)                                                     \
    do {                                                             \
        cudaError_t _e = (call);                                     \
        if (_e != cudaSuccess) return e->cuda_fail(_e, #call);       \
    } while (0)

namespace {

template <int D>
cudaError_t lattice_setup_d(size_t* smem) {
    *smem = sizeof(yklt::Shared<D>);
    return cudaFuncSetAttribute(yk_lattice_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)*smem);
}
cudaError_t lattice_setup(int D, size_t* smem) {
    switch (D) {
        case 1: return lattice_setup_d<1>(smem); case 2: return lattice_setup_d<2>(smem); case 3: return lattice_setup_d<3>(smem);
        case 4: return lattice_setup_d<4>(smem); case 5: return lattice_setup_d<5>(smem); case 6: return lattice_setup_d<6>(smem);
        case 7: return lattice_setup_d<7>(smem); default: return lattice_setup_d<8>(smem);
    }
}
void launch_lattice(int D, const yklt::Args& a, size_t smem, cudaStream_t s) {
    switch (D) {
        case 1: yk_lattice_kernel<1><<<1, yklt::THREADS, smem, s>>>(a); break;
        case 2: yk_lattice_kernel<2><<<1, yklt::THREADS, smem, s>>>(a); break;
        case 3: yk_lattice_kernel<3><<<1, yklt::THREADS, smem, s>>>(a); break;
        case 4: yk_lattice_kernel<4><<<1, yklt::THREADS, smem, s>>>(a); break;
        case 5: yk_lattice_kernel<5><<<1, yklt::THREADS, smem, s>>>(a); break;
        case 6: yk_lattice_kernel<6><<<1, yklt::THREADS, smem, s>>>(a); break;
        case 7: yk_lattice_kernel<7><<<1, yklt::THREADS, smem, s>>>(a); break;
        default: yk_lattice_kernel<8><<<1, yklt::THREADS, smem, s>>>(a); break;
    }
}

int upload_tables(yk_engine* e) {
    const int D = e->D;
    if (e->rank_stale) {
        std::vector<uint32_t> live;
        live.reserve(e->n_hi);
        for (uint32_t i = 0; i < e->n_hi; ++i) if (e->n_present[i]) live.push_back(i);
        std::sort(live.begin(), live.end(), [&](uint32_t a, uint32_t b) {
            if (e->n_rank[a] != e->n_rank[b]) return e->n_rank[a] < e->n_rank[b];
            return a < b;
        });
        e->nlive = (uint32_t)live.size();
        e->ranks_unique = true;
        for (size_t i = 1; i < live.size(); ++i) if (e->n_rank[live[i]] == e->n_rank[live[i - 1]]) e->ranks_unique = false;
        if (e->nlive) memcpy(e->by_rank.p, live.data(), sizeof(uint32_t) * e->nlive);
        if (e->nlive) CK(cudaMemcpyAsync(e->d_by_rank.p, e->by_rank.p, sizeof(uint32_t) * e->nlive, cudaMemcpyHostToDevice, e->stream));
        e->st.h2d_bytes += sizeof(uint32_t) * e->nlive;
        if (e->lt_allowed && e->n_hi) {   // the lattice commit orders ties by the rank itself
            CK(cudaMemcpyAsync(e->d_rank.p, e->n_rank.data(), sizeof(uint32_t) * e->n_hi, cudaMemcpyHostToDevice, e->stream));
            CK(cudaStreamSynchronize(e->stream));   // n_rank is pageable memory
            e->st.h2d_bytes += sizeof(uint32_t) * e->n_hi;
        }
        e->rank_stale = false;
    }
    if (e->nodes_stale && e->n_hi) {
        const size_t n = e->n_hi;
        for (int k = 0; k < D; ++k) {
            CK(cudaMemcpyAsync(e->d_total.p + (size_t)k * e->maxN, e->n_total.p + (size_t)k * e->maxN, 8 * n, cudaMemcpyHostToDevice, e->stream));
            CK(cudaMemcpyAsync(e->d_avail.p + (size_t)k * e->maxN, e->n_avail.p + (size_t)k * e->maxN, 8 * n, cudaMemcpyHostToDevice, e->stream));
        }
        CK(cudaMemcpyAsync(e->d_taint.p, e->n_taint.p, 8 * n, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->d_label.p, e->n_label.p, 8 * n, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->d_flags.p, e->n_flags.p, 4 * n, cudaMemcpyHostToDevice, e->stream));
        e->st.h2d_bytes += n * (16 * D + 20);
    }
    e->nodes_stale = false;
    if (e->asks_stale && e->a_hi) {
        const size_t n = e->a_hi;
        for (int k = 0; k < D; ++k)
            CK(cudaMemcpyAsync(e->d_areq.p + (size_t)k * e->maxA, e->a_req.p + (size_t)k * e->maxA, 8 * n, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->d_atol.p, e->a_tol.p, 8 * n, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->d_aneed.p, e->a_need.p, 8 * n, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->d_adeny.p, e->a_deny.p, 8 * n, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->d_anode.p, e->a_node.p, 4 * n, cudaMemcpyHostToDevice, e->stream));
        e->st.h2d_bytes += n * (8 * D + 28);
    }
    e->asks_stale = false;
    return YK_OK;
}

// grid.y (ask splits) is sized so that tiles x splits fills the resident CTA slots of the device exactly once
template <int D>
void launch_sweep_d(YkSweepArgs a, cudaStream_t s, int slots) {
    const int tiles = a.Np / NODE_TILE;
    int splits = std::max(1, slots / tiles);
    a.per = (a.rows + splits - 1) / splits;
    splits = (a.rows + a.per - 1) / a.per;
    dim3 grid((unsigned)tiles, (unsigned)splits);
    yk_sweep_kernel<D, NPT, AC><<<grid, YK_SWEEP_THREADS, 0, s>>>(a);
}
template <int D>
int sweep_slots_d(int sms) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, yk_sweep_kernel<D, NPT, AC>, YK_SWEEP_THREADS, 0) != cudaSuccess || per_sm < 1) per_sm = 2;
    return per_sm * sms;
}
int sweep_slots(int D, int sms) {
    switch (D) {
        case 1: return sweep_slots_d<1>(sms); case 2: return sweep_slots_d<2>(sms); case 3: return sweep_slots_d<3>(sms);
        case 4: return sweep_slots_d<4>(sms); case 5: return sweep_slots_d<5>(sms); case 6: return sweep_slots_d<6>(sms);
        case 7: return sweep_slots_d<7>(sms); default: return sweep_slots_d<8>(sms);
    }
}
void launch_sweep(int D, const YkSweepArgs& a, cudaStream_t s, int slots) {
    switch (D) {
        case 1: launch_sweep_d<1>(a, s, slots); break;
        case 2: launch_sweep_d<2>(a, s, slots); break;
        case 3: launch_sweep_d<3>(a, s, slots); break;
        case 4: launch_sweep_d<4>(a, s, slots); break;
        case 5: launch_sweep_d<5>(a, s, slots); break;
        case 6: launch_sweep_d<6>(a, s, slots); break;
        case 7: launch_sweep_d<7>(a, s, slots); break;
        default: launch_sweep_d<8>(a, s, slots); break;
    }
}

// Initial node order of a cycle, computed on the device: float64 score per node (yk_key_kernel), stable radix
// sort by key over NodeID-rank order = ascending (score, NodeID).  device_order() only enqueues (the lattice commit
// consumes the result on the stream); initial_order() also brings it to the host commit's working copy.
void setup_commit_tables(yk_engine* e) {
    yk::CommitTables& ct = e->cm.t;
    ct.D = e->D; ct.policy = e->cfg.policy; ct.w = e->w.w; ct.lda = e->maxA;
    ct.a_req = e->a_req.p; ct.a_tol = e->a_tol.p; ct.a_need = e->a_need.p; ct.a_deny = e->a_deny.p; ct.a_node = e->a_node.p;
    ct.a_gang = e->a_gang.data(); ct.a_app = e->a_app.data();
    e->cm.profile = e->prof;
}

int device_order(yk_engine* e) {
    const int nlive = (int)e->nlive;
    if (nlive == 0) return YK_OK;
    cudaStream_t s = e->stream;
    CK(cudaMemsetAsync(e->d_flag.p, 0, sizeof(int), s));
    CK(cudaEventRecord(e->ev0, s));
    yk_key_kernel<<<(nlive + 255) / 256, 256, 0, s>>>(e->D, e->cfg.policy, e->w, e->d_total.p, e->d_avail.p, e->maxN,
                                                     e->d_by_rank.p, nlive, e->d_key_in.p, e->d_val_in.p, e->d_flag.p);
    size_t tb = e->cub_bytes;
    CK(cub::DeviceRadixSort::SortPairs(e->d_cub.p, tb, e->d_key_in.p, e->d_key_out.p, e->d_val_in.p, e->d_val_out.p,
                                       nlive, 0, 64, s));
    CK(cudaEventRecord(e->ev1, s));
    CK(cudaMemcpyAsync(e->h_flag.p, e->d_flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    e->st.d2h_bytes += 4;
    e->st.other_launches += 11;   // key + cub radix sort (histogram, exclusive sum, 8 onesweep passes for 64-bit keys)
    return YK_OK;
}

int initial_order(yk_engine* e) {
    const int nlive = (int)e->nlive;
    if (nlive == 0) return YK_OK;
    cudaStream_t s = e->stream;
    if (!e->order_enqueued) {   // (after a hand-over from the device commit the order is computed again from the exported tables)
        int rc = device_order(e);
        if (rc) return rc;
    }
    e->order_enqueued = false;
    CK(cudaMemcpyAsync(e->h_order[0].p, e->d_val_out.p, sizeof(uint32_t) * (size_t)nlive, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(e->h_skey.p, e->d_key_out.p, sizeof(uint64_t) * (size_t)nlive, cudaMemcpyDeviceToHost, s));
    // while the device scores and sorts: the commit's working copy of the node table (host only)
    e->cm.build(e->n_hi, e->n_avail.p, e->n_total.p, e->maxN, e->n_taint.p, e->n_label.p, e->n_rank.data());
    CK(cudaStreamSynchronize(s));
    e->st.d2h_bytes += 12 * (size_t)nlive;
    if (e->h_flag[0]) return e->fail(YK_ERR_RANGE, "NaN node score (zero total on a weighted resource)");
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->st.sort_ms += ms;
    e->cur = 0;
    e->cm.set_order(e->h_order[0].p, e->h_skey.p, nlive);   // the cycle's initial order: (key, rank, node) per position
    return YK_OK;
}

// ---- uniform runs on the device (yk_uniform.h / yk_uniform.cuh) -------------------------------------------------------
constexpr size_t UN_EMAX = (size_t)4 << 20;   // generated elements per attempt at most (nodes x depth)

int un_ensure(yk_engine* e) {
    if (e->un_alloc) return YK_OK;
    const size_t N = e->maxN;
    for (int b = 0; b < 2; ++b) {
        CK(e->d_un_ekey[b].alloc(UN_EMAX)); CK(e->d_un_enode[b].alloc(UN_EMAX));
        CK(e->d_un_rkey[b].alloc(N)); CK(e->d_un_rrn[b].alloc(N));
    }
    CK(e->d_un_bk.alloc(N)); CK(e->d_un_cnt.alloc(N));
    CK(e->d_un_g.alloc(1)); CK(e->h_un_g.alloc(1));
    CK(cudaMemsetAsync(e->d_un_cnt.p, 0, sizeof(uint32_t) * std::max<size_t>(N, 1), e->stream));
    size_t t0 = 0, t1 = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, t0, e->d_un_ekey[0].p, e->d_un_ekey[1].p, e->d_un_enode[0].p, e->d_un_enode[1].p, (int)UN_EMAX, 0, 64, e->stream));
    CK(cub::DeviceRadixSort::SortPairs(nullptr, t1, e->d_un_rkey[0].p, e->d_un_rkey[1].p, e->d_un_rrn[0].p, e->d_un_rrn[1].p, (int)std::max<size_t>(N, 1), 0, 64, e->stream));
    e->un_cub_bytes = std::max(t0, t1);
    CK(e->d_un_cub.alloc(e->un_cub_bytes));
    e->un_alloc = true;
    return YK_OK;
}

template <int D>
cudaError_t un_attempt_d(yk_engine* e, const ykun::Args& a) {
    cudaStream_t s = e->stream;
    const int nb = (a.nlive + 255) / 256;
    ykun::un_reset_kernel<<<1, 1, 0, s>>>(a.g);
    ykun::un_depth_kernel<D><<<(unsigned)(((size_t)a.nlive * (size_t)a.L + 255) / 256), 256, 0, s>>>(a);
    ykun::un_brank_kernel<D><<<nb, 256, 0, s>>>(a);
    size_t tb = e->un_cub_bytes;
    cudaError_t rc = cub::DeviceRadixSort::SortPairs(e->d_un_cub.p, tb, a.ekey, const_cast<unsigned long long*>(a.skey), a.enode,
                                                     const_cast<uint32_t*>(a.snode), a.nlive * a.L, 0, 64, s);
    if (rc != cudaSuccess) return rc;
    ykun::un_select_kernel<D><<<(a.R + 255) / 256, 256, 0, s>>>(a);
    ykun::un_decide_kernel<<<1, 1, 0, s>>>(a);
    ykun::un_apply_rekey_kernel<D><<<nb, 256, 0, s>>>(a);   // leaves the new order entries (rank order) in rkey / rrn
    return cudaGetLastError();
}
cudaError_t un_attempt(yk_engine* e, const ykun::Args& a) {
    switch (e->D) {
        case 1: return un_attempt_d<1>(e, a); case 2: return un_attempt_d<2>(e, a); case 3: return un_attempt_d<3>(e, a);
        case 4: return un_attempt_d<4>(e, a); case 5: return un_attempt_d<5>(e, a); case 6: return un_attempt_d<6>(e, a);
        case 7: return un_attempt_d<7>(e, a); default: return un_attempt_d<8>(e, a);
    }
}

// The node order after uniform runs: only the windowed kernel reads it, so it is rebuilt (stable sort of the re-keyed entries,
// which un_apply_rekey_kernel left in rank order) when a windowed stretch follows, not after every run.
int un_reorder(yk_engine* e) {
    if (!e->un_ord_stale) return YK_OK;
    cudaStream_t s = e->stream;
    const int nlive = (int)e->nlive;
    size_t tb = e->un_cub_bytes;
    CK(cub::DeviceRadixSort::SortPairs(e->d_un_cub.p, tb, e->d_un_rkey[0].p, e->d_un_rkey[1].p, e->d_un_rrn[0].p, e->d_un_rrn[1].p, nlive, 0, 64, s));
    ykun::Args a{};
    a.ord[0] = e->d_ord[0].p; a.ord[1] = e->d_ord[1].p; a.cur = e->d_lt_cur.p; a.nlive = nlive;
    a.okey = e->d_un_rkey[1].p; a.orn = e->d_un_rrn[1].p;
    ykun::un_order_kernel<<<(nlive + 255) / 256, 256, 0, s>>>(a);
    CK(cudaGetLastError());
    e->st.other_launches += 11;
    e->un_ord_stale = false;
    return YK_OK;
}

// One uniform run: entries [off, off + R) of the staged batch (h_lt_asks; results land in d_lt_res at the same offset).
// status = ykun::U_DONE / U_STOPPED with *consumed entries decided, or U_FALLBACK: nothing was applied, the windowed kernel
// takes the run.
int lt_uniform(yk_engine* e, size_t off, size_t R, bool insensitive, bool has_gang, int* status, size_t* consumed) {
    *status = ykun::U_FALLBACK; *consumed = 0;
    const int nlive = (int)e->nlive;
    if (nlive == 0 || R == 0) return YK_OK;
    int rc = un_ensure(e);
    if (rc) return rc;
    cudaStream_t s = e->stream;
    const uint32_t ask = e->h_lt_asks[off];
    ykun::Args a{};
    a.policy = e->cfg.policy;
    for (int k = 0; k < 8; ++k) { a.w[k] = e->w.w[k]; a.req[k] = k < e->D ? e->a_req[(size_t)k * e->maxA + ask] : 0; }
    a.rec = e->d_rec.p; a.RS = e->lt_RS; a.ord[0] = e->d_ord[0].p; a.ord[1] = e->d_ord[1].p; a.cur = e->d_lt_cur.p;
    a.nlive = nlive; a.byrank = e->d_by_rank.p;   // live nodes by ascending (NodeID rank, index): upload_tables
    a.tol = e->a_tol[ask]; a.need = e->a_need[ask]; a.deny = e->a_deny[ask]; a.want = e->a_node[ask];
    a.R = (int)R; a.insensitive = insensitive ? 1 : 0; a.has_gang = has_gang ? 1 : 0;
    a.ekey = e->d_un_ekey[0].p; a.skey = e->d_un_ekey[1].p; a.enode = e->d_un_enode[0].p; a.snode = e->d_un_enode[1].p;
    a.bk = e->d_un_bk.p; a.cnt = e->d_un_cnt.p;
    a.rkey = e->d_un_rkey[0].p; a.okey = e->d_un_rkey[1].p; a.rrn = e->d_un_rrn[0].p; a.orn = e->d_un_rrn[1].p;
    a.res = e->d_lt_res.p + off; a.g = e->d_un_g.p;
    int L = ykun::first_depth((int)R, nlive);
    // no node takes the request more often than its TOTAL allows: beyond that depth nothing is ever cut
    int64_t capmax = 0;
    for (uint32_t i = 0; i < e->nlive; ++i) {
        const uint32_t n = e->by_rank[i];
        int64_t tot[8];
        for (int k = 0; k < e->D; ++k) tot[k] = e->n_total[(size_t)k * e->maxN + n];
        capmax = std::max(capmax, ykun::cap_of_d(e->D, true, tot, tot, a.req, (int64_t)R));
    }
    int Lmax = 1;
    while ((int64_t)Lmax < capmax) Lmax <<= 1;
    {   // a request with no weighted dimension leaves every key where it is: the run fills the first nodes (by key, NodeID) to
        // the brim, so the depth that matters is a node's whole capacity, not the mean share
        bool flat = true;
        for (int k = 0; k < e->D; ++k) if (e->w.w[k] != 0.0 && a.req[k] != 0) flat = false;
        if (flat) L = Lmax;
    }
    L = std::min(L, Lmax);
    for (;;) {
        if ((size_t)L * (size_t)nlive > UN_EMAX) return YK_OK;   // too deep for the element buffers: fallback
        a.L = L;
        CK(cudaEventRecord(e->ev_l0, s));
        CK(un_attempt(e, a));
        CK(cudaEventRecord(e->ev_l1, s));
        CK(cudaMemcpyAsync(e->h_un_g.p, e->d_un_g.p, sizeof(ykun::Globals), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        float ms = 0;
        cudaEventElapsedTime(&ms, e->ev_l0, e->ev_l1);
        e->st.lattice_ms += ms;
        e->st.lattice_launches += 1;
        e->st.other_launches += 16;   // 6 kernels of yk_uniform.cuh + one cub radix sort (histogram, exclusive sum, 8 onesweep passes)
        e->st.d2h_bytes += sizeof(ykun::Globals);
        const ykun::Globals& g = e->h_un_g[0];
        if (g.status == ykun::U_RETRY) {   // deeper; past Lmax only if a node's available exceeds its total (the buffers end it)
            e->st.uniform_retries++;
            L = L < Lmax ? (int)std::min<int64_t>((int64_t)L * 4, (int64_t)Lmax) : L * 4;
            continue;
        }
        if (g.status == ykun::U_NAN || g.status == ykun::U_FALLBACK) return YK_OK;
        if (g.nan) return e->fail(YK_ERR_RANGE, "NaN node score after commit");
        *status = g.status; *consumed = (size_t)g.consumed;
        e->un_ord_stale = true;
        e->st.uniform_runs++; e->st.uniform_asks += (uint64_t)g.consumed; e->st.uniform_elements += (uint64_t)L * (uint64_t)nlive;
        return YK_OK;
    }
}

// ---- device-resident ordered commit (yk_lattice.h) -------------------------------------------------------------------
// node records + order entries from the sorted keys; capacity bound and header reset
int lt_prepare(yk_engine* e) {
    const int nlive = (int)e->nlive;
    cudaStream_t s = e->stream;
    if (nlive)
        yk_lt_init_kernel<<<(nlive + 255) / 256, 256, 0, s>>>(e->D, e->d_total.p, e->d_avail.p, e->maxN, e->d_taint.p, e->d_label.p,
                                                             e->d_flags.p, e->d_rank.p, e->d_key_out.p, e->d_val_out.p, nlive,
                                                             e->d_rec.p, e->lt_RS, e->d_ord[0].p);
    CK(cudaGetLastError());
    for (int k = 0; k < 8; ++k) e->h_lt_ub[(size_t)k] = INT64_MAX;
    CK(cudaMemcpyAsync(e->d_lt_ub.p, e->h_lt_ub.p, 8 * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(e->d_lt_cur.p, 0, sizeof(int), s));
    CK(cudaMemsetAsync(e->d_lt_hdr.p, 0, yklt::H_WORDS * sizeof(int), s));
    e->st.other_launches += 1;
    memset(e->h_lt_hdr.p, 0, yklt::H_WORDS * sizeof(int));
    e->un_ord_stale = false;
    return YK_OK;
}

// One batch through the device commit: asks + their three words up (already in the pinned staging buffers), node indices +
// header back.  Uniform runs of at least un_min entries go through lt_uniform, the stretches between them through
// yk_lattice_kernel; h_lt_hdr[H_STATUS / H_CONSUMED] describe the whole batch afterwards.  Blocks until it is decided.
int lt_window(yk_engine* e, size_t off, size_t B, bool insensitive) {
    cudaStream_t s = e->stream;
    { const int rco = un_reorder(e); if (rco) return rco; }
    yklt::Args a{};
    a.policy = e->cfg.policy;
    for (int k = 0; k < 8; ++k) a.w[k] = e->w.w[k];
    a.rec = e->d_rec.p; a.RS = e->lt_RS; a.ord[0] = e->d_ord[0].p; a.ord[1] = e->d_ord[1].p; a.cur = e->d_lt_cur.p;
    a.nlive = (int)e->nlive;
    a.a_req = e->d_areq.p; a.lda = e->maxA; a.a_tol = e->d_atol.p; a.a_need = e->d_aneed.p; a.a_deny = e->d_adeny.p; a.a_node = e->d_anode.p;
    a.asks = e->d_lt_asks.p + off; a.meta = e->d_lt_meta.p + off; a.shp = e->d_lt_shp.p + off; a.sig = e->d_lt_sig.p + off; a.B = (int)B;
    a.res = e->d_lt_res.p + off; a.hdr = e->d_lt_hdr.p; a.ub = e->d_lt_ub.p; a.insensitive = insensitive ? 1 : 0;
    a.prof = e->lt_prof ? e->d_lt_prof.p : nullptr;
    CK(cudaEventRecord(e->ev_l0, s));
    launch_lattice(e->D, a, e->lt_smem, s);
    CK(cudaGetLastError());
    CK(cudaEventRecord(e->ev_l1, s));
    CK(cudaMemcpyAsync(e->h_lt_hdr.p, e->d_lt_hdr.p, yklt::H_WORDS * sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev_l0, e->ev_l1);
    e->st.lattice_ms += ms;
    e->st.lattice_launches += 1;
    e->st.d2h_bytes += yklt::H_WORDS * sizeof(int);
    return YK_OK;
}

int lt_batch(yk_engine* e, size_t B, bool insensitive) {
    cudaStream_t s = e->stream;
    // the segments (e->un_segs) were planned by the caller; only the windowed kernel reads the per-entry words
    bool staged = false;
    auto stage = [&]() -> int {
        if (staged) return YK_OK;
        CK(cudaMemcpyAsync(e->d_lt_asks.p, e->h_lt_asks.p, 4 * B, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(e->d_lt_meta.p, e->h_lt_meta.p, 4 * B, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(e->d_lt_shp.p, e->h_lt_shp.p, 4 * B, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(e->d_lt_sig.p, e->h_lt_sig.p, 4 * B, cudaMemcpyHostToDevice, s));
        e->st.h2d_bytes += 16 * B;
        staged = true;
        return YK_OK;
    };
    int status = yklt::ST_DONE;
    size_t done = 0;
    for (const ykun::Segment& sg : e->un_segs) {
        size_t consumed = 0;
        int st = yklt::ST_DONE;
        bool windowed = !sg.uniform;
        if (sg.uniform) {
            bool has_gang = false;
            for (int i = 0; i < sg.len && !has_gang; ++i) has_gang = (e->h_lt_meta[(size_t)sg.off + i] & yklt::M_GANG) != 0;
            int ust = ykun::U_FALLBACK;
            const int rc = lt_uniform(e, (size_t)sg.off, (size_t)sg.len, insensitive, has_gang, &ust, &consumed);
            if (rc) return rc;
            if (ust == ykun::U_FALLBACK) windowed = true;
            else st = ust == ykun::U_STOPPED ? yklt::ST_STOPPED : yklt::ST_DONE;
        }
        if (windowed) {
            const int rcs = stage();
            if (rcs) return rcs;
            const int rc = lt_window(e, (size_t)sg.off, (size_t)sg.len, insensitive);
            if (rc) return rc;
            st = e->h_lt_hdr[yklt::H_STATUS];
            consumed = (size_t)e->h_lt_hdr[yklt::H_CONSUMED];
            if (consumed > (size_t)sg.len) return e->fail(YK_ERR_CUDA, "lattice kernel returned a bad header");
        }
        done = (size_t)sg.off + consumed;
        status = st;
        if (st != yklt::ST_DONE || consumed < (size_t)sg.len) break;
    }
    e->h_lt_hdr[yklt::H_STATUS] = status;
    e->h_lt_hdr[yklt::H_CONSUMED] = (int)done;
    if (done) {
        CK(cudaMemcpyAsync(e->h_lt_res.p, e->d_lt_res.p, 4 * done, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        e->st.d2h_bytes += 4 * done;
    }
    return YK_OK;
}

// the records' availability back into the column-major device table and the host table (end of the cycle, or hand-over)
int lt_export(yk_engine* e) {
    const int nlive = (int)e->nlive;
    if (nlive == 0) return YK_OK;
    cudaStream_t s = e->stream;
    CK(cudaMemcpyAsync(e->h_flag.p, e->d_lt_cur.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const int cur = e->h_flag[0] & 1;
    yk_lt_export_kernel<<<(nlive + 255) / 256, 256, 0, s>>>(e->D, e->d_rec.p, e->lt_RS, e->d_ord[cur].p, nlive, e->d_avail.p, e->maxN);
    CK(cudaGetLastError());
    for (int k = 0; k < e->D; ++k)
        CK(cudaMemcpyAsync(e->n_avail.p + (size_t)k * e->maxN, e->d_avail.p + (size_t)k * e->maxN, 8 * (size_t)e->n_hi, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    e->st.d2h_bytes += 8 * (size_t)e->n_hi * e->D + 4;
    e->st.other_launches += 1;
    return YK_OK;
}

// ---- epochs -------------------------------------------------------------------------------------------
// An epoch is a run of batches swept against ONE sorted view (node order + cap columns as of the epoch start).
// Exactness does not need the view to be fresh: a node not touched since the epoch began has exactly the state
// the view holds, and every touched node is masked out of the bitmaps and handled from the working copy
// (DESIGN.md "ordered commit").  So the order is merged, the availability pushed to the device and the view
// regathered only when the touched set has grown enough to slow the commit down -- and because the sweeps of one
// epoch do not depend on each other's commits, the next batch's sweep and read-back overlap the current commit.
int begin_epoch(yk_engine* e) {
    const int nlive = (int)e->nlive;
    const int Np = (int)round_up((size_t)nlive, NODE_TILE);
    e->epochW = nlive ? Np / 32 : 0;
    e->cm.begin_epoch(e->epochW);
    if (nlive == 0) return YK_OK;
    cudaStream_t s = e->stream;
    CK(cudaMemcpyAsync(e->d_order.p, e->h_order[e->cur].p, sizeof(uint32_t) * (size_t)nlive, cudaMemcpyHostToDevice, s));
    e->st.h2d_bytes += sizeof(uint32_t) * (size_t)nlive;
    yk_gather_kernel<<<(Np + 255) / 256, 256, 0, s>>>(e->D, e->d_total.p, e->d_avail.p, e->maxN, e->d_taint.p, e->d_label.p,
                                                     e->d_flags.p, e->d_order.p, nlive, Np, e->d_scap.p, e->d_staint.p,
                                                     e->d_slabel.p, e->d_snode.p);
    CK(cudaGetLastError());
    e->st.other_launches += 1;
    if (e->ep_rows) {   // every distinct signature of the cycle against the fresh view: one launch, one read-back per epoch
        const int W = e->epochW, WS = W + 1, R = (int)e->ep_n;
        if (!e->ep_uploaded) {
            memcpy(e->ep_h_batch.p, e->ep_reps.data(), sizeof(uint32_t) * (size_t)R);
            CK(cudaMemcpyAsync(e->ep_d_batch.p, e->ep_h_batch.p, sizeof(uint32_t) * (size_t)R, cudaMemcpyHostToDevice, s));
            e->st.h2d_bytes += sizeof(uint32_t) * (size_t)R;
            e->ep_uploaded = true;
        }
        CK(cudaMemset2DAsync(e->ep_d_fit.p + W, sizeof(uint32_t) * (size_t)WS, 0xFF, sizeof(uint32_t), (size_t)R, s));
        CK(cudaEventRecord(e->ep_s0, s));
        YkSweepArgs a{};
        a.s_cap = e->d_scap.p; a.s_taint = e->d_staint.p; a.s_label = e->d_slabel.p; a.s_node = e->d_snode.p; a.Np = Np;
        a.a_req = e->d_areq.p; a.a_tol = e->d_atol.p; a.a_need = e->d_aneed.p; a.a_deny = e->d_adeny.p; a.a_node = e->d_anode.p;
        a.lda = e->maxA; a.batch = e->ep_d_batch.p; a.row0 = 0; a.rows = R;
        a.fit = e->ep_d_fit.p; a.W = W; a.WS = WS; a.n_peer = 0;
        launch_sweep(e->D, a, s, e->slots);
        CK(cudaEventRecord(e->ep_s1, s));
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(e->ep_h_fit.p, e->ep_d_fit.p, sizeof(uint32_t) * (size_t)R * WS, cudaMemcpyDeviceToHost, s));
        CK(cudaEventRecord(e->ep_ev, s));
        e->ep_landed = false;
        e->st.sweep_launches += 1;
        e->st.evaluations += (uint64_t)R * (uint64_t)nlive;
        e->st.rows_swept += (uint64_t)R;
        e->st.d2h_bytes += sizeof(uint32_t) * (size_t)R * WS;
    }
    return YK_OK;
}

// new node order = merge(previous order minus the touched nodes, touched nodes by new key); touched availability
// goes back to the column-major host table and to the device table.  `reorder` false = end of cycle (state only).
int end_epoch(yk_engine* e, bool reorder) {
    const int D = e->D, nlive = (int)e->nlive;
    const int nd = (int)e->cm.dirty_list.size();
    if (!nd) return YK_OK;
    const double t0 = now_ms();
    cudaStream_t s = e->stream;
    if (reorder) {
        e->cm.merge_order(e->h_order[e->cur ^ 1].p, nlive);
        e->cur ^= 1;
    }
    // staging is reused: the previous epoch's upload must have been consumed
    CK(cudaStreamSynchronize(s));
    for (int i0 = 0; i0 < nd; i0 += (int)e->h_dirty_nodes.n) {
        const int cnt = std::min<int>(nd - i0, (int)e->h_dirty_nodes.n);
        for (int i = 0; i < cnt; ++i) {
            const uint32_t n = e->cm.dirty_list[(size_t)(i0 + i)];
            e->h_dirty_nodes[(size_t)i] = n;
            for (int k = 0; k < D; ++k) {
                const int64_t v = e->cm.node(n).avail()[k];
                e->h_dirty_vals[(size_t)k * cnt + i] = v;
                e->n_avail[(size_t)k * e->maxN + n] = v;   // column-major host table stays authoritative between cycles
            }
        }
        CK(cudaMemcpyAsync(e->d_dirty_nodes.p, e->h_dirty_nodes.p, 4 * (size_t)cnt, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(e->d_dirty_vals.p, e->h_dirty_vals.p, 8 * (size_t)cnt * D, cudaMemcpyHostToDevice, s));
        yk_apply_avail_kernel<<<(cnt + 255) / 256, 256, 0, s>>>(D, e->d_avail.p, e->maxN, e->d_dirty_nodes.p, e->d_dirty_vals.p, cnt);
        CK(cudaGetLastError());
        e->st.h2d_bytes += (size_t)cnt * (4 + 8 * D);
        e->st.other_launches += 1;
        if (i0 + cnt < nd) CK(cudaStreamSynchronize(s));
    }
    e->st.host_ms[5] += now_ms() - t0;
    return YK_OK;
}

// Launch the device phase of one batch (already filled into sl.asks): sweep of this rank's rows against the epoch
// view, multi-GPU exchange, chunked read-back with one event per chunk.  Returns without waiting.
int produce(yk_engine* e, Slot& sl, yk_stats_t& st) {
    const int D = e->D;
    const int B = (int)sl.asks.size();
    const int nlive = (int)e->nlive;
    sl.B = B; sl.R = 0; sl.W = e->epochW; sl.rows = 0; sl.nchunks = 0;
    if (B == 0 || nlive == 0) return YK_OK;
    const double t0 = now_ms();
    if (e->ep_rows) {   // the rows of every signature were swept when the epoch began: the batch only points at them
        sl.row_of.resize((size_t)B);
        for (int i = 0; i < B; ++i) sl.row_of[(size_t)i] = e->ep_local[e->a_sigid[sl.asks[(size_t)i]]];
        sl.R = (int)e->ep_n;
        st.batches++;
        st.asks_swept += (uint64_t)B;
        st.host_ms[6] += now_ms() - t0;
        return YK_OK;
    }
    const int W = e->epochW, Np = W * 32, WS = W + 1;
    cudaStream_t s = e->stream;
    // one row per distinct predicate signature in the batch (yk_commit.hpp "shared rows")
    e->share.build(e->cm.t, e->a_sig.data(), sl.asks, e->share_rows, sl.reps, sl.row_of);
    const int R = (int)sl.reps.size();
    sl.R = R;
    memcpy(sl.h_batch.p, sl.reps.data(), sizeof(uint32_t) * (size_t)R);
    CK(cudaMemcpyAsync(sl.d_batch.p, sl.h_batch.p, sizeof(uint32_t) * (size_t)R, cudaMemcpyHostToDevice, s));
    st.h2d_bytes += sizeof(uint32_t) * (size_t)R;
    // this rank's shard of the rows (world == 1: all of them).  A sweep too small to pay for the exchange (shared rows:
    // a few dozen rows per batch) is not split at all: every rank sweeps every row locally and nothing is exchanged.
    // All ranks see the same R and nlive, so they take the same branch.
    const int G = std::max<int>(1, (int)e->cfg.world);
    const bool split = G > 1 && (uint64_t)R * (uint64_t)nlive >= e->split_min_pairs;
    const int world = split ? G : 1;
    const int my_rank = split ? (int)e->cfg.rank : 0;
    const int rows_per = (R + world - 1) / world;
    const int row0 = std::min(R, my_rank * rows_per);
    const int rows = std::min(R, row0 + rows_per) - row0;
    const int Bpad = rows_per * world;
    sl.rows = rows;
    // the last word of every row (first-fit position) starts at YK_NONE
    const int slot_id = (int)(&sl - e->slot);
    const bool p2p_on = G > 1 && e->p2p;   // peers can write into this rank's slots
    const bool p2p = split && p2p_on;      // ... and do, for this batch
    uint32_t value = 0;
    const long long spin_limit = 4000000000ll;   // ~2 s of SM clocks: a dead peer becomes YK_ERR_COMM, not a hang
    if (p2p_on) {
        // The slot's previous content must have been consumed by every rank before anybody overwrites it.  Batches that
        // are not split take part in this hand-shake too (not in the "rows ready" one): ranks are not in lock-step, and
        // a rank that is ahead must not publish the rows of a later, split batch into a slot this rank still reads.
        value = ++e->seq;
        yk_p2p_wait_kernel<<<1, 32, 0, s>>>(e->d_sync.p, G, 16 + slot_id * 8, sl.last_value, e->d_flag.p, spin_limit);
        sl.last_value = value;
        st.other_launches += 1;
    } else {
        // the last word of every row (first-fit position) starts at YK_NONE
        CK(cudaMemset2DAsync(sl.d_fit.p + W, sizeof(uint32_t) * (size_t)WS, 0xFF, sizeof(uint32_t), (size_t)Bpad, s));
    }
    CK(cudaEventRecord(sl.ev_s0, s));
    if (rows > 0) {
        YkSweepArgs a{};
        a.s_cap = e->d_scap.p; a.s_taint = e->d_staint.p; a.s_label = e->d_slabel.p; a.s_node = e->d_snode.p; a.Np = Np;
        a.a_req = e->d_areq.p; a.a_tol = e->d_atol.p; a.a_need = e->d_aneed.p; a.a_deny = e->d_adeny.p; a.a_node = e->d_anode.p;
        a.lda = e->maxA; a.batch = sl.d_batch.p; a.row0 = row0; a.rows = rows;
        a.fit = sl.d_fit.p; a.W = W; a.WS = WS;
        a.n_peer = p2p ? world : 0;
        for (int g = 0; g < 8; ++g) a.fit_peer[g] = p2p && g < world ? e->peer_fit[slot_id][g] : nullptr;
        launch_sweep(D, a, s, e->slots);
        st.sweep_launches += 1;
        st.evaluations += (uint64_t)rows * (uint64_t)nlive;
    }
    CK(cudaEventRecord(sl.ev_s1, s));
    CK(cudaGetLastError());
    if (p2p) {
        YkPeerSync ps{};
        YkPeerFit pf{};
        for (int g = 0; g < world; ++g) { ps.sync[g] = e->peer_sync[g]; pf.fit[g] = e->peer_fit[slot_id][g]; }
        if (rows > 0)
            yk_p2p_first_kernel<<<(rows + 255) / 256, 256, 0, s>>>(sl.d_fit.p, pf, world, my_rank, row0, rows, W, WS);
        yk_p2p_signal_kernel<<<1, 32, 0, s>>>(ps, world, slot_id * 8 + my_rank, value);            // my rows are in place
        yk_p2p_wait_kernel<<<1, 32, 0, s>>>(e->d_sync.p, world, slot_id * 8, value, e->d_flag.p, spin_limit);   // everybody's are
        CK(cudaGetLastError());
        st.other_launches += 3;
    } else if (world > 1) {
        if (!e->xfn) return e->fail(YK_ERR_COMM, "world > 1 but neither a peer-to-peer nor a callback exchange is set up");
        if (e->xfn(e->xctx, sl.d_fit.p, (uint64_t)WS * 4, (uint32_t)row0, (uint32_t)rows_per, (uint32_t)Bpad, (void*)s) != 0)
            return e->fail(YK_ERR_COMM, "exchange callback failed");
    }
    if (p2p_on) CK(cudaMemcpyAsync(sl.h_err.p, e->d_flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));   // flag waits timed out?
    // read-back in row chunks so the ordered commit overlaps the transfer
    sl.chunk = std::max(128, (R + (int)sl.ev.size() - 1) / (int)sl.ev.size());
    sl.nchunks = (R + sl.chunk - 1) / sl.chunk;
    for (int c = 0; c < sl.nchunks; ++c) {
        const size_t r0 = (size_t)c * sl.chunk, r1 = std::min<size_t>((size_t)R, r0 + sl.chunk);
        CK(cudaMemcpyAsync(sl.h_fit.p + r0 * WS, sl.d_fit.p + r0 * WS, sizeof(uint32_t) * (r1 - r0) * WS, cudaMemcpyDeviceToHost, s));
        CK(cudaEventRecord(sl.ev[(size_t)c], s));
    }
    if (p2p_on) {
        // consumed: wipe the slot (every word back to 0xFFFFFFFF, so first-fit words start at YK_NONE whatever the next
        // row layout is) and tell every rank it may publish into it again
        CK(cudaMemsetAsync(sl.d_fit.p, 0xFF, sl.d_fit.n * sizeof(uint32_t), s));
        YkPeerSync ps{};
        for (int g = 0; g < G; ++g) ps.sync[g] = e->peer_sync[g];
        yk_p2p_signal_kernel<<<1, 32, 0, s>>>(ps, G, 16 + slot_id * 8 + (int)e->cfg.rank, value);
        CK(cudaGetLastError());
        st.other_launches += 1;
    }
    st.d2h_bytes += sizeof(uint32_t) * (size_t)R * WS;
    st.batches++;
    st.asks_swept += (uint64_t)B;
    st.rows_swept += (uint64_t)R;
    st.host_ms[6] += now_ms() - t0;
    return YK_OK;
}

// wait until everything issued for the slot has landed (used before its buffers are reused or it is dropped)
int drain(yk_engine* e, Slot& sl) {
    if (sl.B > 0 && sl.nchunks > 0) CK(cudaEventSynchronize(sl.ev[(size_t)sl.nchunks - 1]));
    return YK_OK;
}

// Ordered commit of one batch from its (arriving) bitmaps: the logic is yk::Committer::commit_batch; this wrapper
// supplies the rows as the read-back chunks land and keeps the timing / counters.
int commit(yk_engine* e, Slot& sl, bool insensitive, std::vector<uint32_t>& result, size_t& consumed) {
    const int B = sl.B;
    const std::vector<uint32_t>& batch = sl.asks;
    result.assign((size_t)B, YK_NONE);
    consumed = 0;
    if (e->ep_rows && e->nlive != 0) {
        double t_wait = 0;
        const double t1 = now_ms();
        if (!e->ep_landed) {
            const cudaError_t ce = cudaEventSynchronize(e->ep_ev);
            if (ce != cudaSuccess) return e->cuda_fail(ce, "cudaEventSynchronize(epoch rows)");
            e->ep_landed = true;
            t_wait = now_ms() - t1;
            float ms_sweep = 0;
            cudaEventElapsedTime(&ms_sweep, e->ep_s0, e->ep_s1);
            e->st.sweep_ms += ms_sweep;
            e->st.last_sweep_ms = ms_sweep;
            e->st.last_sweep_pairs = (uint64_t)e->ep_n * (uint64_t)e->nlive;
        }
        const int R = sl.R;
        const int rc = e->cm.commit_batch(batch, sl.row_of.data(), e->ep_h_fit.p, insensitive, result, consumed, [R](int) { return R; });
        if (rc == -5) return e->fail(YK_ERR_RANGE, "NaN node score after commit");
        if (rc < 0) return e->fail(YK_ERR_CUDA, "commit aborted");
        const double t2 = now_ms();
        e->st.host_ms[3] += t_wait;
        e->st.host_ms[4] += (t2 - t1) - t_wait;
        e->st.commit_ms += (t2 - t1) - t_wait;
        return YK_OK;
    }
    if (e->nlive == 0 || sl.nchunks == 0) {   // no nodes: nothing fits
        consumed = insensitive ? (size_t)B : std::min<size_t>(1, (size_t)B);
        if (!insensitive && B > 0 && e->a_gang[batch[0]] != YK_NONE)
            while (consumed < (size_t)B && e->cm.same_gang(batch[0], batch[consumed])) ++consumed;
        return YK_OK;
    }
    double t_wait = 0;
    const double t1 = now_ms();
    int next_chunk = 0, wait_rc = YK_OK;
    auto wait = [&](int row) -> int {   // block until the chunk holding `row` has landed; -> rows landed so far
        while (row >= next_chunk * sl.chunk) {
            const double tw = now_ms();
            const cudaError_t ce = cudaEventSynchronize(sl.ev[(size_t)next_chunk]);
            t_wait += now_ms() - tw;
            if (ce != cudaSuccess) { wait_rc = e->cuda_fail(ce, "cudaEventSynchronize(read-back chunk)"); return -1; }
            ++next_chunk;
            if (e->p2p && sl.h_err[0]) {
                wait_rc = e->fail(YK_ERR_COMM, "peer-to-peer exchange timed out waiting for another rank");
                return -1;
            }
        }
        return std::min(sl.R, next_chunk * sl.chunk);
    };
    const int rc = e->cm.commit_batch(batch, sl.row_of.data(), sl.h_fit.p, insensitive, result, consumed, wait);
    if (rc == -5) return e->fail(YK_ERR_RANGE, "NaN node score after commit");
    if (rc < 0) return wait_rc ? wait_rc : e->fail(YK_ERR_CUDA, "commit aborted");
    // all read-back must have landed before the slot's buffers are reused
    {
        const double tw = now_ms();
        { int rcd = drain(e, sl); if (rcd) return rcd; }
        t_wait += now_ms() - tw;
    }
    const double t2 = now_ms();
    e->st.host_ms[3] += t_wait;
    e->st.host_ms[4] += (t2 - t1) - t_wait;
    e->st.commit_ms += (t2 - t1) - t_wait;
    float ms_sweep = 0;
    cudaEventElapsedTime(&ms_sweep, sl.ev_s0, sl.ev_s1);
    e->st.sweep_ms += ms_sweep;
    e->st.last_sweep_ms = ms_sweep;
    e->st.last_sweep_pairs = (uint64_t)sl.rows * (uint64_t)e->nlive;
    return YK_OK;
}

}  // namespace

// ======================================= C ABI =======================================
// idx[] = first, first+1, ... : the bulk-load shape; lets the upserts copy whole columns
static bool contiguous_run(const uint32_t* idx, uint32_t n) {
    for (uint32_t i = 1; i < n; ++i) if (idx[i] != idx[0] + i) return false;
    return n > 0;
}
// what the user of application p holds under every limit entry that applies to it moves by sign * request(ask)
static void user_held_add(yk_engine* e, uint32_t p, uint32_t ask, int sign) {
    if (!e->n_ul || e->p_user[p] == YK_NONE) return;
    for (uint32_t l = 0; l < e->n_ul; ++l) {
        if (e->ul_user[l] != e->p_user[p]) continue;
        for (uint32_t q = e->p_queue[p]; q != YK_NONE; q = e->q_parent[q])
            if (q == e->ul_queue[l]) {
                for (int k = 0; k < e->D; ++k) e->ul_alloc[(size_t)k * e->n_ul + l] += sign * e->a_req[(size_t)k * e->maxA + ask];
                break;
            }
    }
}

template <typename T>
static void copy_or_fill(T* dst, const T* src, uint32_t n, T dflt) {
    if (src) memcpy(dst, src, sizeof(T) * (size_t)n);
    else std::fill(dst, dst + n, dflt);
}

extern "C" {

uint32_t yk_abi_version(void) { return YK_ABI_VERSION; }

const char* yk_strerror(int s) {
    switch (s) {
        case YK_OK: return "ok";
        case YK_ERR_ARG: return "invalid argument";
        case YK_ERR_CUDA: return "CUDA error (no device, no sm_100a image, or launch/copy failure)";
        case YK_ERR_NOMEM: return "out of memory";
        case YK_ERR_STATE: return "invalid state";
        case YK_ERR_RANGE: return "value out of range (NaN node score)";
        case YK_ERR_COMM: return "multi-GPU exchange failed";
        default: return "unknown status";
    }
}

const char* yk_last_error(yk_engine* e) { return e ? e->err.c_str() : "null engine"; }

void yk_destroy(yk_engine* e) {
    if (!e) return;
    e->worker.stop();
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->hp_on && e->hp_n)
        fprintf(stderr, "[ykgpu] host ms per cycle (%llu cycles): prologue %.3f  upload+device_order %.3f  wait orderer setup %.3f  first fill + commit choice %.3f  "
                        "run %.3f  epoch end / export + sync %.3f  finish %.3f\n", (unsigned long long)e->hp_n, e->hp[0] / e->hp_n, e->hp[1] / e->hp_n,
                e->hp[2] / e->hp_n, e->hp[3] / e->hp_n, e->hp[4] / e->hp_n, e->hp[5] / e->hp_n, e->hp[6] / e->hp_n);
    if (e->lt_prof && e->d_lt_prof.p) {
        long long pf[16] = {0};
        if (cudaMemcpy(pf, e->d_lt_prof.p, sizeof(pf), cudaMemcpyDeviceToHost) == cudaSuccess) {
            static const char* nm[yklt::PF_N] = {"stage", "scan", "window", "bound", "lattice", "sort", "links+rows", "chain", "apply", "patch", "fullscan"};
            fprintf(stderr, "[ykgpu] lattice kernel, SM clocks per phase (%llu sub-runs):", (unsigned long long)e->lt_total_subruns);
            for (int k = 0; k < yklt::PF_N; ++k) fprintf(stderr, " %s=%lld", nm[k], pf[k]);
            fprintf(stderr, "\n");
        }
    }
    for (int g = 0; g < 8; ++g)
        if (e->peer_open[g]) { cudaIpcCloseMemHandle(e->peer_fit[0][g]); cudaIpcCloseMemHandle(e->peer_fit[1][g]); cudaIpcCloseMemHandle(e->peer_sync[g]); }
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->ev2) cudaEventDestroy(e->ev2);
    if (e->ep_ev) cudaEventDestroy(e->ep_ev);
    if (e->ep_s0) cudaEventDestroy(e->ep_s0);
    if (e->ep_s1) cudaEventDestroy(e->ep_s1);
    if (e->ev_l0) cudaEventDestroy(e->ev_l0);
    if (e->ev_l1) cudaEventDestroy(e->ev_l1);
    for (Slot& sl : e->slot) {
        for (auto ev : sl.ev) if (ev) cudaEventDestroy(ev);
        if (sl.ev_s0) cudaEventDestroy(sl.ev_s0);
        if (sl.ev_s1) cudaEventDestroy(sl.ev_s1);
    }
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

int yk_create(const yk_config* cfg, yk_engine** out) {
    if (!cfg || !out) return YK_ERR_ARG;
    *out = nullptr;
    if (cfg->abi_version != YK_ABI_VERSION || cfg->D < 1 || cfg->D > YK_MAX_D || cfg->policy > 1) return YK_ERR_ARG;
    if (!cfg->max_nodes || !cfg->max_asks || !cfg->max_apps || !cfg->max_queues) return YK_ERR_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return YK_ERR_CUDA;   // fail loudly: no CPU path
    if (cfg->device >= 0) { if (cudaSetDevice(cfg->device) != cudaSuccess) return YK_ERR_CUDA; }
    yk_engine* e = new (std::nothrow) yk_engine();
    if (!e) return YK_ERR_NOMEM;
    e->cfg = *cfg;
    e->share_rows = !(cfg->flags & YK_FLAG_NO_ROW_SHARING) && !getenv("YK_NO_ROW_SHARING");
    if (const char* sp = getenv("YK_SPLIT_MIN_PAIRS")) e->split_min_pairs = strtoull(sp, nullptr, 10);
    e->D = (int)cfg->D;
    e->maxN = cfg->max_nodes; e->maxA = cfg->max_asks; e->maxP = cfg->max_apps; e->maxQ = cfg->max_queues;
    e->batch = cfg->batch ? cfg->batch : 4096;
    for (int k = 0; k < 8; ++k) e->w.w[k] = k < e->D ? cfg->weights[k] : 0.0;
    const int D = e->D;
    const size_t N = e->maxN, A = e->maxA, Bm = e->batch;
    const size_t Npmax = round_up(N, NODE_TILE);
    e->Wmax = Npmax / 32;
    bool ok = true;
    auto T = [&](cudaError_t r) { if (r != cudaSuccess) { ok = false; e->err = cudaGetErrorString(r); } };
    T(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    T(cudaEventCreate(&e->ev0)); T(cudaEventCreate(&e->ev1)); T(cudaEventCreate(&e->ev2));
    T(e->n_total.alloc(N * D)); T(e->n_avail.alloc(N * D)); T(e->n_taint.alloc(N)); T(e->n_label.alloc(N)); T(e->n_flags.alloc(N));
    T(e->by_rank.alloc(N));
    T(e->a_req.alloc(A * D)); T(e->a_tol.alloc(A)); T(e->a_need.alloc(A)); T(e->a_deny.alloc(A)); T(e->a_node.alloc(A));
    T(e->d_total.alloc(N * D)); T(e->d_avail.alloc(N * D)); T(e->d_taint.alloc(N)); T(e->d_label.alloc(N)); T(e->d_flags.alloc(N));
    T(e->d_by_rank.alloc(N));
    T(e->d_areq.alloc(A * D)); T(e->d_atol.alloc(A)); T(e->d_aneed.alloc(A)); T(e->d_adeny.alloc(A)); T(e->d_anode.alloc(A));
    T(e->d_key_in.alloc(N)); T(e->d_key_out.alloc(N)); T(e->d_val_in.alloc(N)); T(e->d_val_out.alloc(N));
    if (ok) {
        size_t tb = 0;
        T(cub::DeviceRadixSort::SortPairs(nullptr, tb, e->d_key_in.p, e->d_key_out.p, e->d_val_in.p, e->d_val_out.p, (int)N, 0, 64, e->stream));
        e->cub_bytes = tb;
        T(e->d_cub.alloc(tb));
    }
    T(e->d_scap.alloc(Npmax * D)); T(e->d_staint.alloc(Npmax)); T(e->d_slabel.alloc(Npmax)); T(e->d_snode.alloc(Npmax));
    const size_t Bpad = Bm + std::max<uint32_t>(cfg->world, 1);   // rows rounded up to a multiple of world
    T(e->d_flag.alloc(1));
    T(e->h_order[0].alloc(N)); T(e->h_order[1].alloc(N)); T(e->d_order.alloc(N));
    for (Slot& sl : e->slot) {
        T(sl.d_batch.alloc(Bm)); T(sl.d_fit.alloc(Bpad * (e->Wmax + 1)));
        T(sl.h_batch.alloc(Bm)); T(sl.h_fit.alloc(Bm * (e->Wmax + 1))); T(sl.h_err.alloc(1));
        sl.ev.assign(16, nullptr);
        for (auto& ev : sl.ev) T(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        T(cudaEventCreate(&sl.ev_s0)); T(cudaEventCreate(&sl.ev_s1));
    }
    T(e->d_sync.alloc(32));
    if (ok) {
        T(cudaMemset(e->d_sync.p, 0, 32 * sizeof(uint32_t)));
        for (Slot& sl : e->slot) T(cudaMemset(sl.d_fit.p, 0xFF, sl.d_fit.n * sizeof(uint32_t)));
    }
    e->epoch_floor = std::max<uint32_t>(2 * e->batch, 4096);
    if (const char* v = getenv("YK_EPOCH_NODES")) e->epoch_env = (uint32_t)std::max(1, atoi(v));   // tuning / debugging knob
    e->no_spec = getenv("YK_NO_SPECULATION") != nullptr;
    e->prof = getenv("YK_PROFILE_COMMIT") != nullptr;
    if (ok) { int dev = 0; cudaGetDevice(&dev); e->worker.start(dev); }
    T(e->d_dirty_nodes.alloc(N)); T(e->d_dirty_vals.alloc(N * D)); T(e->d_scores.alloc(N));
    // device-resident ordered commit
    e->lt_allowed = !(cfg->flags & YK_FLAG_HOST_COMMIT) && cfg->world <= 1;
    e->lt_auto = true;
    if (cfg->flags & YK_FLAG_DEVICE_COMMIT) e->lt_force = 1;
    if (const char* cm = getenv("YK_COMMIT")) {
        if (!strcmp(cm, "host")) e->lt_allowed = false;
        if (!strcmp(cm, "device")) e->lt_force = 1;
        if (!strcmp(cm, "auto")) { e->lt_auto = true; e->lt_force = 0; e->lt_allowed = !(cfg->flags & YK_FLAG_HOST_COMMIT) && cfg->world <= 1; }
    }
    e->lt_RS = (2 * D + 3 + 3) / 4 * 4;
    T(e->d_rec.alloc(N * (size_t)e->lt_RS)); T(e->d_ord[0].alloc(N)); T(e->d_ord[1].alloc(N)); T(e->d_rank.alloc(N));
    T(e->d_lt_cur.alloc(1)); T(e->d_lt_hdr.alloc(yklt::H_WORDS)); T(e->d_lt_ub.alloc(8));
    T(e->d_lt_asks.alloc(A)); T(e->d_lt_meta.alloc(A)); T(e->d_lt_shp.alloc(A)); T(e->d_lt_sig.alloc(A)); T(e->d_lt_res.alloc(A));
    T(e->h_lt_asks.alloc(A)); T(e->h_lt_meta.alloc(A)); T(e->h_lt_shp.alloc(A)); T(e->h_lt_sig.alloc(A)); T(e->h_lt_res.alloc(A)); T(e->h_lt_hdr.alloc(yklt::H_WORDS)); T(e->h_lt_ub.alloc(8));
    T(cudaEventCreate(&e->ev_l0)); T(cudaEventCreate(&e->ev_l1));
    T(e->ep_d_batch.alloc(yk_engine::EP_MAX)); T(e->ep_h_batch.alloc(yk_engine::EP_MAX));
    T(e->ep_d_fit.alloc((size_t)yk_engine::EP_MAX * (e->Wmax + 1))); T(e->ep_h_fit.alloc((size_t)yk_engine::EP_MAX * (e->Wmax + 1)));
    T(cudaEventCreateWithFlags(&e->ep_ev, cudaEventDisableTiming)); T(cudaEventCreate(&e->ep_s0)); T(cudaEventCreate(&e->ep_s1));
    e->lt_prof = getenv("YK_PROFILE_LATTICE") != nullptr;
    e->hp_on = getenv("YK_PROFILE_HOST") != nullptr;
    if (const char* um = getenv("YK_UNIFORM_MIN")) e->un_min = atoi(um);   // 0: no uniform-run path
    T(e->d_lt_prof.alloc(16));
    if (ok) T(cudaMemset(e->d_lt_prof.p, 0, 16 * sizeof(long long)));
    if (ok) T(lattice_setup(D, &e->lt_smem));
    T(e->h_snode.alloc(N)); T(e->h_skey.alloc(N));
    T(e->h_dirty_nodes.alloc(N)); T(e->h_dirty_vals.alloc(N * D)); T(e->h_flag.alloc(1)); T(e->h_scores.alloc(N));
    if (ok) {   // does this binary carry an image the device can run?
        cudaFuncAttributes fa;
        T(cudaFuncGetAttributes(&fa, yk_key_kernel));
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        e->slots = sweep_slots(D, sms);
    }
    if (!ok) { yk_destroy(e); return YK_ERR_CUDA; }
    e->n_rank.assign(N, 0); e->n_present.assign(N, 0);
    e->a_shape.assign(A, 0); e->a_sigid.assign(A, 0); e->a_cause.assign(A, 0);
    e->sigs.reset(A);
    e->a_sig.assign(A, 0); e->a_prio.assign(A, 0); e->a_create.assign(A, 0); e->a_app.assign(A, 0); e->a_flags.assign(A, 0);
    e->a_gang.assign(A, YK_NONE); e->a_bound.assign(A, YK_NONE); e->a_state.assign(A, yk::ST_ABSENT);
    e->p_queue.assign(e->maxP, 0); e->p_submit.assign(e->maxP, 0); e->p_present.assign(e->maxP, 0); e->p_user.assign(e->maxP, YK_NONE);
    e->p_alloc.assign((size_t)e->maxP * D, 0);
    // default queue tree: root only would have no leaf for apps; root + one leaf "root.default"
    e->nq = 0;
    
    *out = e;
    return YK_OK;
}

int yk_nodes_upsert(yk_engine* e, uint32_t n, const uint32_t* idx, const int64_t* total, const int64_t* avail,
                    const uint64_t* taint, const uint64_t* label, const uint32_t* name_rank, const uint32_t* flags) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && (!idx || !total || !avail || !name_rank)) return e->fail(YK_ERR_ARG, "yk_nodes_upsert: null array");
    for (uint32_t i = 0; i < n; ++i) if (idx[i] >= e->maxN) return e->fail(YK_ERR_ARG, "yk_nodes_upsert: index beyond max_nodes");
    if (contiguous_run(idx, n)) {   // whole-column copies
        const uint32_t x0 = idx[0];
        for (int k = 0; k < e->D; ++k) {
            memcpy(&e->n_total[(size_t)k * e->maxN + x0], total + (size_t)k * n, sizeof(int64_t) * (size_t)n);
            memcpy(&e->n_avail[(size_t)k * e->maxN + x0], avail + (size_t)k * n, sizeof(int64_t) * (size_t)n);
        }
        copy_or_fill<uint64_t>(&e->n_taint[x0], taint, n, 0);
        copy_or_fill<uint64_t>(&e->n_label[x0], label, n, 0);
        copy_or_fill<uint32_t>(&e->n_flags[x0], flags, n, YK_NODE_SCHEDULABLE);
        for (uint32_t i = 0; i < n && !e->rank_stale; ++i)
            if (!e->n_present[x0 + i] || e->n_rank[x0 + i] != name_rank[i]) e->rank_stale = true;
        memcpy(&e->n_rank[x0], name_rank, sizeof(uint32_t) * (size_t)n);
        std::fill(e->n_present.begin() + x0, e->n_present.begin() + x0 + n, 1);
        e->n_hi = std::max(e->n_hi, x0 + n);
        e->nodes_stale = true;
        return YK_OK;
    }
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t x = idx[i];
        for (int k = 0; k < e->D; ++k) {
            e->n_total[(size_t)k * e->maxN + x] = total[(size_t)k * n + i];
            e->n_avail[(size_t)k * e->maxN + x] = avail[(size_t)k * n + i];
        }
        e->n_taint[x] = taint ? taint[i] : 0;
        e->n_label[x] = label ? label[i] : 0;
        e->n_flags[x] = flags ? flags[i] : YK_NODE_SCHEDULABLE;
        if (!e->n_present[x] || e->n_rank[x] != name_rank[i]) e->rank_stale = true;
        e->n_rank[x] = name_rank[i];
        e->n_present[x] = 1;
        e->n_hi = std::max(e->n_hi, x + 1);
    }
    e->nodes_stale = true;
    return YK_OK;
}

int yk_nodes_remove(yk_engine* e, uint32_t n, const uint32_t* idx) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && !idx) return e->fail(YK_ERR_ARG, "yk_nodes_remove: null array");
    for (uint32_t i = 0; i < n; ++i) {
        if (idx[i] >= e->maxN) return e->fail(YK_ERR_ARG, "yk_nodes_remove: index beyond max_nodes");
        if (e->n_present[idx[i]]) { e->n_present[idx[i]] = 0; e->n_flags[idx[i]] = 0; e->rank_stale = true; e->nodes_stale = true; }
    }
    return YK_OK;
}

int yk_queues_set(yk_engine* e, uint32_t q, const uint32_t* parent, const int64_t* guaranteed, const int64_t* max,
                  const int64_t* allocated, const uint8_t* sort) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (!q || q > e->maxQ || !parent) return e->fail(YK_ERR_ARG, "yk_queues_set: bad queue count");
    if (parent[0] != YK_NONE) return e->fail(YK_ERR_ARG, "yk_queues_set: queue 0 must be the root");
    for (uint32_t i = 1; i < q; ++i) if (parent[i] >= i) return e->fail(YK_ERR_ARG, "yk_queues_set: parent[i] must be < i");
    const int D = e->D;
    // applications keep pointing at queue indices: a tree that no longer has them (or turned their leaf into a parent) is
    // refused rather than silently re-homing them
    for (uint32_t p = 0; p < e->maxP; ++p) {
        if (!e->p_present[p]) continue;
        if (e->p_queue[p] >= q) return e->fail(YK_ERR_STATE, "yk_queues_set: an application sits in a queue the new tree does not have (remove or move it first)");
        for (uint32_t i = 1; i < q; ++i)
            if (parent[i] == e->p_queue[p]) return e->fail(YK_ERR_STATE, "yk_queues_set: an application sits in a queue the new tree makes a parent");
    }
    e->nq = q;
    e->q_parent.assign(parent, parent + q);
    e->q_guar.assign((size_t)q * D, -1); e->q_max.assign((size_t)q * D, -1); e->q_alloc.assign((size_t)q * D, 0);
    if (guaranteed) e->q_guar.assign(guaranteed, guaranteed + (size_t)q * D);
    if (max) e->q_max.assign(max, max + (size_t)q * D);
    if (allocated) e->q_alloc.assign(allocated, allocated + (size_t)q * D);
    else   // what the present applications hold stays accounted: their allocations are summed up the new tree
        for (uint32_t p = 0; p < e->maxP; ++p) {
            if (!e->p_present[p]) continue;
            for (uint32_t qq = e->p_queue[p]; qq != YK_NONE; qq = e->q_parent[qq])
                for (int k = 0; k < D; ++k) e->q_alloc[(size_t)k * q + qq] += e->p_alloc[(size_t)k * e->maxP + p];
        }
    e->q_sort.assign(q, 0);
    if (sort) e->q_sort.assign(sort, sort + q);
    e->q_prio_offset.assign(q, 0); e->q_prio_fence.assign(q, 0);   // defaults; yk_queues_priority sets them
    for (uint32_t i = 0; i < q; ++i)
        if (e->q_sort[i] > 1) return e->fail(YK_ERR_ARG, "yk_queues_set: unknown application sort policy");
    return YK_OK;
}

int yk_queues_priority(yk_engine* e, uint32_t q, const int32_t* offset, const uint8_t* fence) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (q != e->nq) return e->fail(YK_ERR_ARG, "yk_queues_priority: queue count differs from yk_queues_set");
    e->q_prio_offset.assign(q, 0); e->q_prio_fence.assign(q, 0);
    if (offset) e->q_prio_offset.assign(offset, offset + q);
    if (fence) for (uint32_t i = 0; i < q; ++i) e->q_prio_fence[i] = fence[i] ? 1 : 0;
    return YK_OK;
}

int yk_apps_upsert(yk_engine* e, uint32_t n, const uint32_t* idx, const uint32_t* queue, const int64_t* submit) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && (!idx || !queue || !submit)) return e->fail(YK_ERR_ARG, "yk_apps_upsert: null array");
    for (uint32_t i = 0; i < n; ++i) {
        if (idx[i] >= e->maxP) return e->fail(YK_ERR_ARG, "yk_apps_upsert: index beyond max_apps");
        if (queue[i] >= e->nq) return e->fail(YK_ERR_ARG, "yk_apps_upsert: unknown queue (call yk_queues_set first)");
    }
    for (uint32_t i = 0; i < n; ++i) {
        if (!e->p_present[idx[i]]) for (int k = 0; k < e->D; ++k) e->p_alloc[(size_t)k * e->maxP + idx[i]] = 0;
        e->p_queue[idx[i]] = queue[i]; e->p_submit[idx[i]] = submit[i]; e->p_present[idx[i]] = 1;
    }
    return YK_OK;
}

int yk_apps_user(yk_engine* e, uint32_t n, const uint32_t* idx, const uint32_t* user) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && (!idx || !user)) return e->fail(YK_ERR_ARG, "yk_apps_user: null array");
    for (uint32_t i = 0; i < n; ++i) if (idx[i] >= e->maxP) return e->fail(YK_ERR_ARG, "yk_apps_user: index beyond max_apps");
    for (uint32_t i = 0; i < n; ++i) e->p_user[idx[i]] = user[i];
    return YK_OK;
}

int yk_user_limits_set(yk_engine* e, uint32_t n, const uint32_t* queue, const uint32_t* user, const int64_t* max, const int64_t* held) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && (!queue || !user || !max)) return e->fail(YK_ERR_ARG, "yk_user_limits_set: null array");
    for (uint32_t i = 0; i < n; ++i) if (queue[i] >= e->nq) return e->fail(YK_ERR_ARG, "yk_user_limits_set: unknown queue (call yk_queues_set first)");
    const int D = e->D;
    e->n_ul = n;
    e->ul_queue.assign(queue, queue + n); e->ul_user.assign(user, user + n);
    e->ul_max.assign(max, max + (size_t)n * D);
    if (held) e->ul_alloc.assign(held, held + (size_t)n * D); else e->ul_alloc.assign((size_t)n * D, 0);
    return YK_OK;
}

int yk_apps_remove(yk_engine* e, uint32_t n, const uint32_t* idx) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && !idx) return e->fail(YK_ERR_ARG, "yk_apps_remove: null array");
    for (uint32_t i = 0; i < n; ++i) {
        if (idx[i] >= e->maxP) return e->fail(YK_ERR_ARG, "yk_apps_remove: index beyond max_apps");
        e->p_present[idx[i]] = 0;
    }
    return YK_OK;
}

// what keeps an ask out of the passes whatever the cluster looks like (yk::Tables::a_cause): the slow-path flag, or a request
// that is not strictly greater than zero ([EXT] preAllocateCheck)
static uint8_t ask_cause(const yk_engine* e, uint32_t x) {
    if (e->a_flags[x] & 1u) return yk::ST_SLOWPATH;
    bool pos = false;
    for (int k = 0; k < e->D; ++k) {
        const int64_t v = e->a_req[(size_t)k * e->maxA + x];
        if (v < 0) return yk::ST_INVALID;
        if (v > 0) pos = true;
    }
    return pos ? 0 : yk::ST_INVALID;
}

int yk_asks_upsert(yk_engine* e, uint32_t a, const uint32_t* idx, const int64_t* req, const uint64_t* tol,
                   const uint64_t* need, const uint64_t* deny, const int32_t* prio, const int64_t* create_seq,
                   const uint32_t* app, const uint32_t* required_node, const uint32_t* flags, const uint32_t* gang) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (a && (!idx || !req || !create_seq || !app)) return e->fail(YK_ERR_ARG, "yk_asks_upsert: null array");
    for (uint32_t i = 0; i < a; ++i) {
        if (idx[i] >= e->maxA) return e->fail(YK_ERR_ARG, "yk_asks_upsert: index beyond max_asks");
        if (app[i] >= e->maxP || !e->p_present[app[i]]) return e->fail(YK_ERR_ARG, "yk_asks_upsert: unknown application");
        if (required_node && required_node[i] != YK_NONE && required_node[i] >= e->maxN)
            return e->fail(YK_ERR_ARG, "yk_asks_upsert: required_node beyond max_nodes");
        if (e->a_state[idx[i]] == yk::ST_ALLOCATED) return e->fail(YK_ERR_STATE, "yk_asks_upsert: ask holds an allocation (release it first)");
    }
    yk::CommitTables sv;   // just enough of a view for the signature hash
    sv.D = e->D; sv.lda = e->maxA; sv.a_req = e->a_req.p; sv.a_tol = e->a_tol.p; sv.a_need = e->a_need.p; sv.a_deny = e->a_deny.p; sv.a_node = e->a_node.p;
    if (contiguous_run(idx, a)) {   // whole-column copies, then the signature hashes in one sequential pass
        const uint32_t x0 = idx[0];
        for (int k = 0; k < e->D; ++k) memcpy(&e->a_req[(size_t)k * e->maxA + x0], req + (size_t)k * a, sizeof(int64_t) * (size_t)a);
        copy_or_fill<uint64_t>(&e->a_tol[x0], tol, a, 0);
        copy_or_fill<uint64_t>(&e->a_need[x0], need, a, 0);
        copy_or_fill<uint64_t>(&e->a_deny[x0], deny, a, 0);
        copy_or_fill<uint32_t>(&e->a_node[x0], required_node, a, YK_NONE);
        copy_or_fill<int32_t>(&e->a_prio[x0], prio, a, 0);
        memcpy(&e->a_create[x0], create_seq, sizeof(int64_t) * (size_t)a);
        memcpy(&e->a_app[x0], app, sizeof(uint32_t) * (size_t)a);
        copy_or_fill<uint32_t>(&e->a_flags[x0], flags, a, 0);
        copy_or_fill<uint32_t>(&e->a_gang[x0], gang, a, YK_NONE);
        std::fill(e->a_state.begin() + x0, e->a_state.begin() + x0 + a, (uint8_t)yk::ST_PENDING);
        std::fill(e->a_bound.begin() + x0, e->a_bound.begin() + x0 + a, YK_NONE);
        // (the rows [x0, x0+a) were overwritten above: numbers they represented are retired first)
        const bool full = x0 == 0 && a >= e->a_hi;
        if (full) e->sigs.reset(e->maxA);
        else for (uint32_t i = 0; i < a; ++i) e->sigs.retire(x0 + i);
        for (uint32_t i = 0; i < a; ++i) e->a_sig[x0 + i] = yk::ask_signature(sv, x0 + i);
        for (uint32_t i = 0; i < a; ++i) e->a_cause[x0 + i] = ask_cause(e, x0 + i);
        e->a_hi = std::max(e->a_hi, x0 + a);
        if (!full && e->sigs.n > 2 * e->maxA) {   // too many stale numbers: renumber every present ask
            e->sigs.reset(e->maxA);
            for (uint32_t y = 0; y < e->a_hi; ++y) if (e->a_state[y] != yk::ST_ABSENT) e->a_sigid[y] = e->sigs.get(sv, e->a_sig[y], y);
        } else {
            for (uint32_t i = 0; i < a; ++i) e->a_sigid[x0 + i] = e->sigs.get(sv, e->a_sig[x0 + i], x0 + i);
        }
        e->asks_stale = true;
        return YK_OK;
    }
    for (uint32_t i = 0; i < a; ++i) {
        const uint32_t x = idx[i];
        for (int k = 0; k < e->D; ++k) e->a_req[(size_t)k * e->maxA + x] = req[(size_t)k * a + i];
        e->a_tol[x] = tol ? tol[i] : 0;
        e->a_need[x] = need ? need[i] : 0;
        e->a_deny[x] = deny ? deny[i] : 0;
        e->a_node[x] = required_node ? required_node[i] : YK_NONE;
        e->a_sig[x] = yk::ask_signature(sv, x);
        e->sigs.retire(x);
        if (e->sigs.n > 2 * e->maxA) {   // too many stale numbers: renumber the present asks
            e->sigs.reset(e->maxA);
            for (uint32_t y = 0; y < e->a_hi; ++y) if (y != x && e->a_state[y] != yk::ST_ABSENT) e->a_sigid[y] = e->sigs.get(sv, e->a_sig[y], y);
        }
        e->a_sigid[x] = e->sigs.get(sv, e->a_sig[x], x);
        e->a_prio[x] = prio ? prio[i] : 0;
        e->a_create[x] = create_seq[i];
        e->a_app[x] = app[i];
        e->a_flags[x] = flags ? flags[i] : 0;
        e->a_cause[x] = ask_cause(e, x);
        e->a_gang[x] = gang ? gang[i] : YK_NONE;
        e->a_state[x] = yk::ST_PENDING;
        e->a_bound[x] = YK_NONE;
        e->a_hi = std::max(e->a_hi, x + 1);
    }
    e->asks_stale = true;
    return YK_OK;
}

int yk_asks_remove(yk_engine* e, uint32_t a, const uint32_t* idx) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (a && !idx) return e->fail(YK_ERR_ARG, "yk_asks_remove: null array");
    for (uint32_t i = 0; i < a; ++i) {
        if (idx[i] >= e->maxA) return e->fail(YK_ERR_ARG, "yk_asks_remove: index beyond max_asks");
        if (e->a_state[idx[i]] == yk::ST_ALLOCATED) return e->fail(YK_ERR_STATE, "yk_asks_remove: ask holds an allocation (use yk_release)");
    }
    for (uint32_t i = 0; i < a; ++i) e->a_state[idx[i]] = yk::ST_ABSENT;
    return YK_OK;
}

int yk_release(yk_engine* e, uint32_t n, const uint32_t* idx) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && !idx) return e->fail(YK_ERR_ARG, "yk_release: null array");
    for (uint32_t i = 0; i < n; ++i)
        if (idx[i] >= e->maxA || e->a_state[idx[i]] != yk::ST_ALLOCATED) return e->fail(YK_ERR_STATE, "yk_release: ask holds no allocation");
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t a = idx[i], node = e->a_bound[a];
        for (int k = 0; k < e->D; ++k) {
            const int64_t r = e->a_req[(size_t)k * e->maxA + a];
            if (node != YK_NONE && e->n_present[node]) e->n_avail[(size_t)k * e->maxN + node] += r;
            for (uint32_t q = e->p_queue[e->a_app[a]]; q != YK_NONE; q = e->q_parent[q]) e->q_alloc[(size_t)k * e->nq + q] -= r;
            e->p_alloc[(size_t)k * e->maxP + e->a_app[a]] -= r;
        }
        user_held_add(e, e->a_app[a], a, -1);
        e->a_state[a] = yk::ST_ABSENT;
        e->a_bound[a] = YK_NONE;
    }
    e->nodes_stale = true;
    return YK_OK;
}

}  // extern "C" (reopened after yk_cycle)

// ---- one cycle ---------------------------------------------------------------------------------------------------
namespace {

struct Cycle {
    uint32_t max_bindings = 0;
    yk_binding* out = nullptr;
    uint32_t n = 0;                 // bindings so far
    std::vector<uint32_t> result;
};

// Decided entries [0, consumed) of a batch: orderer bookkeeping + bindings out.  `failed` = the batch ended on an ask /
// gang that found no node in a placement-sensitive order (the orderer is rewound to just before it).
void settle(yk_engine* e, Cycle& c, Slot& A, Slot* later, bool later_forked, size_t consumed, bool ins, bool& failed) {
    failed = false;
    const std::vector<uint32_t>& result = c.result;
    if (!ins && consumed > 0 && result[consumed - 1] == YK_NONE) {
        const double t_r = now_ms();
        size_t j = consumed - 1;   // first entry of the failed ask / gang
        while (j > 0 && e->a_gang[A.asks[j]] != YK_NONE && e->a_gang[A.asks[j - 1]] == e->a_gang[A.asks[j]] &&
               e->a_app[A.asks[j - 1]] == e->a_app[A.asks[j]] && result[j - 1] == YK_NONE) --j;
        // the speculated fill is undone even when it produced no batch: it may still have marked asks (headroom skips)
        e->ord.rewind(A.snap, later_forked && later ? &later->snap : nullptr, A.asks, j);
        e->st.host_ms[2] += now_ms() - t_r;
        failed = true;
    }
    for (size_t i = 0; i < consumed; ++i) {
        const uint32_t a = A.asks[i];
        if (result[i] == YK_NONE) {
            if (ins) e->ord.fail_in_place(a);
            e->st.nofit++;
            continue;
        }
        e->ord.confirm(a);
        e->a_bound[a] = result[i];
        c.out[c.n].ask = a; c.out[c.n].node = result[i];
        ++c.n;
        e->st.allocations++;
    }
}

// fill one batch; YK_ERR_ARG when a gang cannot fit any batch
int fill_batch(yk_engine* e, size_t& bsz, size_t bmax, size_t cap_user, Slot& sl, yk_stats_t& st) {
    sl.asks.clear(); sl.B = 0; sl.nchunks = 0;
    if (cap_user == 0) return YK_OK;
    const double t_f = now_ms();
    e->ord.fill(bsz, cap_user, sl.asks, sl.snap);
    st.host_ms[2] += now_ms() - t_f;
    if (e->ord.oversize_gang) {
        if (bsz < bmax) { bsz = bmax; e->ord.fill(bsz, cap_user, sl.asks, sl.snap); }
        if (e->ord.oversize_gang)
            return e->fail(YK_ERR_ARG, "yk_cycle: a gang has more members than the sweep batch (raise yk_config.batch)");
    }
    return YK_OK;
}

// The cycle on the device commit.  slot[0] already holds the first batch.  Returns with handoff = true (and slot[0]
// holding the next, not yet committed batch) when the rest of the cycle belongs to the host commit.
int run_lattice(yk_engine* e, Cycle& c, bool& handoff) {
    handoff = false;
    const bool ins = e->ord.insensitive;
    Slot& A = e->slot[0];
    size_t bsz = ins ? (size_t)e->maxA : (size_t)e->batch;
    const size_t bmax = bsz;
    int rc = lt_prepare(e);
    if (rc) return rc;
    bool first = true;
    while (!A.asks.empty()) {
        const size_t B = A.asks.size();
        memcpy(e->h_lt_asks.p, A.asks.data(), 4 * B);
        if (!e->lt_plan_ready) {
            yklt::build_meta(e->cm.t, e->lt_shape_ids, e->a_sigid.data(), A.asks, e->h_lt_meta.p, e->h_lt_shp.p, e->h_lt_sig.p);
            ykun::plan_segments(e->h_lt_meta.p, e->h_lt_shp.p, e->h_lt_sig.p, (int)B, e->un_min > 0 ? e->un_min : (int)B + 1, e->un_segs);
        }
        e->lt_plan_ready = false;
        size_t consumed = 0;
        int status = yklt::ST_DONE;
        if (e->nlive == 0) {   // no nodes: nothing fits
            c.result.assign(B, YK_NONE);
            consumed = ins ? B : 1;
            if (!ins && e->a_gang[A.asks[0]] != YK_NONE)
                while (consumed < B && e->cm.same_gang(A.asks[0], A.asks[consumed])) ++consumed;
            if (!ins) status = yklt::ST_STOPPED;
        } else {
            rc = lt_batch(e, B, ins);
            if (rc) return rc;
            if (first && e->h_flag[0]) {
                // the batch was decided on an order holding a NaN key and none of it is returned: the node records it
                // changed must not be exported, so the tables keep what they held before the cycle
                e->lt_active = false;
                return e->fail(YK_ERR_RANGE, "NaN node score (zero total on a weighted resource)");
            }
            status = e->h_lt_hdr[yklt::H_STATUS];
            consumed = (size_t)e->h_lt_hdr[yklt::H_CONSUMED];
            if (status == yklt::ST_NAN) return e->fail(YK_ERR_RANGE, "NaN node score after commit");
            if (consumed > B) return e->fail(YK_ERR_CUDA, "lattice kernel returned a bad header");
            c.result.assign(e->h_lt_res.p, e->h_lt_res.p + B);
        }
        first = false;
        e->st.lattice_asks += consumed;
        e->st.batches++;
        bool failed = false;
        if (status == yklt::ST_HANDOFF) {
            e->ord.unfill(A.snap, A.asks, consumed);   // the undecided tail goes back to the orderer
            bool f2 = false;
            A.asks.resize(consumed);
            c.result.resize(consumed);
            settle(e, c, A, nullptr, false, consumed, true /* no failure cut: every decided entry stands */, f2);
            // (settle with ins = true calls fail_in_place for NONE entries, which is what a placement-insensitive order
            //  wants; a placement-sensitive batch never carries a NONE before a hand-over: the kernel stops there instead)
            e->st.lattice_handoffs++;
            handoff = true;
            return YK_OK;
        }
        settle(e, c, A, nullptr, false, consumed, ins, failed);
        if (!failed && consumed < B) return e->fail(YK_ERR_CUDA, "lattice kernel ended a batch early without a failure");
        bsz = failed ? std::max<size_t>(std::min<size_t>(64, bmax), bsz / 4) : std::min<size_t>(bmax, bsz * 2);
        rc = fill_batch(e, bsz, bmax, (size_t)c.max_bindings - c.n, A, e->st);
        if (rc) return rc;
    }
    return YK_OK;
}

// The cycle on the sweep + host commit path.  slot[0] holds the first batch (filled, not yet launched); the host commit's
// working copy and the epoch view are set up here.
int run_host(yk_engine* e, Cycle& c) {
    int rc = initial_order(e);
    if (rc) return rc;
    e->cm.set_pending(e->pending);   // smallest pending request per dimension: nodes below it are retired from the walk
    // epoch length: long enough that order merges / view refreshes (and the pipeline bubble they cost) stay rare on big
    // clusters, short enough that the touched set does not slow the walk: 5/8 of the nodes, at least two batches
    e->epoch_limit = e->epoch_env ? e->epoch_env : std::max<uint32_t>(e->epoch_floor, (uint32_t)((uint64_t)e->nlive * 5 / 8));
    // Few-signature cycles (epoch rows) under the fair sort, no gangs: the sweeps cost nothing per batch, so what an epoch end buys
    // (a shorter touched index) is worth less than what it costs (order merge, view refresh, a pipeline bubble): measured on
    // config 2, 6.5 -> 5.8 ms with one epoch for the whole cycle; gang cycles (roll-backs walk the touched index) lose.
    if (!e->epoch_env && e->ep_rows && !e->cycle_has_gang && e->cfg.policy == YK_POLICY_FAIR)
        e->epoch_limit = std::max<uint32_t>(e->epoch_limit, 2u * e->nlive);
    rc = begin_epoch(e);
    if (rc) return rc;
    size_t bsz = e->batch;
    const size_t bmax = e->batch;
    const bool ins = e->ord.insensitive;
    // fill + launch one batch into a slot; B == 0 afterwards means the orderer has nothing (more) to offer
    auto next_batch = [&](Slot& sl, size_t cap_user, yk_stats_t& st) -> int {
        const int rcf = fill_batch(e, bsz, bmax, cap_user, sl, st);
        if (rcf) return rcf;
        return produce(e, sl, st);
    };
    auto merge_worker_stats = [&]() {
        yk_stats_t& w = e->wst;
        e->st.h2d_bytes += w.h2d_bytes; e->st.d2h_bytes += w.d2h_bytes; e->st.batches += w.batches;
        e->st.asks_swept += w.asks_swept; e->st.rows_swept += w.rows_swept;
        e->st.sweep_launches += w.sweep_launches; e->st.evaluations += w.evaluations; e->st.other_launches += w.other_launches;
        e->st.host_ms[7] += w.host_ms[2] + w.host_ms[6];   // orderer + launch time hidden behind the commit
        w = yk_stats_t{};
    };
    int cur = 0;
    rc = produce(e, e->slot[0], e->st);
    if (rc) return rc;
    while (e->slot[cur].B > 0) {
        Slot& A = e->slot[cur];
        Slot& Nx = e->slot[cur ^ 1];
        // speculate the next batch on the same epoch view unless this batch may fill the epoch
        Nx.asks.clear(); Nx.B = 0; Nx.nchunks = 0;
        const bool room = e->cm.dirty_list.size() + (size_t)A.B < (size_t)e->epoch_limit;
        const size_t left = (size_t)c.max_bindings - c.n;
        bool forked = false;
        int rc_next = YK_OK;
        if (room && !e->no_spec && left > (size_t)A.B) {
            const size_t cap = left - (size_t)A.B;
            e->worker.submit([&, cap] { rc_next = next_batch(Nx, cap, e->wst); });
            forked = true;
        }
        size_t consumed = 0;
        rc = commit(e, A, ins, c.result, consumed);
        if (forked) { e->worker.wait(); merge_worker_stats(); }
        if (rc) return rc;
        bool failed = false;
        settle(e, c, A, &Nx, forked, consumed, ins, failed);
        if (rc_next) return rc_next;   // this batch's bindings stand; the speculated one never ran
        if (failed && Nx.B > 0) {   // the speculated batch was built on an order that did not happen: drop it
            rc = drain(e, Nx);
            if (rc) return rc;
            Nx.asks.clear(); Nx.B = 0; Nx.nchunks = 0;
        }
        if (failed) { Nx.asks.clear(); Nx.B = 0; Nx.nchunks = 0; }
        // after a failure in a placement-sensitive order, probe with short batches until placements resume
        bsz = failed ? std::max<size_t>(std::min<size_t>(64, e->batch), bsz / 4) : std::min<size_t>(e->batch, bsz * 2);
        if (Nx.B == 0 && c.n < c.max_bindings) {
            // nothing in flight: the epoch may end here (merge order, refresh the device view) before the next batch
            if (e->cm.dirty_list.size() * 2 >= (size_t)e->epoch_limit || failed) {
                rc = end_epoch(e, true);
                if (rc) return rc;
                rc = begin_epoch(e);
                if (rc) return rc;
            }
            rc = next_batch(Nx, (size_t)c.max_bindings - c.n, e->st);
            if (rc) return rc;
        }
        cur ^= 1;
    }
    return YK_OK;
}

}  // namespace

extern "C" int yk_cycle(yk_engine* e, uint32_t max_bindings, yk_binding* out, uint32_t* n_out, uint32_t* slow, uint32_t slow_cap,
             uint32_t* n_slow) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (!n_out || (max_bindings && !out)) return e->fail(YK_ERR_ARG, "yk_cycle: null output");
    *n_out = 0;
    if (n_slow) *n_slow = 0;
    if (e->nq == 0) return e->fail(YK_ERR_STATE, "yk_cycle: no queues configured (yk_queues_set)");
    for (uint32_t p = 0; p < e->maxP; ++p)
        if (e->p_present[p] && e->p_queue[p] >= e->nq) return e->fail(YK_ERR_STATE, "yk_cycle: an application sits in a queue that no longer exists");
    const double t_start = now_ms();
    double hp_t = t_start;   // YK_PROFILE_HOST: where the host time of the cycle goes (printed by yk_destroy)
    auto hp = [&](int k) { if (e->hp_on) { const double t = now_ms(); e->hp[k] += t - hp_t; hp_t = t; } };
    // the orderer's per-cycle setup (host only) runs on the helper thread while this thread uploads stale tables and
    // starts the initial node order on the device
    std::vector<uint32_t>& pending = e->pending;
    double begin_ms = 0;
    bool gang_too_big = false;
    setup_commit_tables(e);
    // device commit: forced (every eligible cycle), or automatic (cycles whose asks come in long uniform runs: yk_uniform.h)
    const bool force_lattice = e->lt_allowed && e->lt_force && e->cfg.policy == YK_POLICY_FAIR;
    const bool auto_lattice = e->lt_allowed && !e->lt_force && e->lt_auto && e->un_min > 0 && e->cfg.policy == YK_POLICY_FAIR;
    e->worker.submit([&] {
        const double t_b = now_ms();
        pending.clear();
        pending.reserve(e->a_hi);
        bool any_gang = false;
        // (longest run of one signature id among consecutive pending asks, in index order: the hint for the automatic commit choice)
        size_t sig_run = 0, sig_longest = 0;
        uint32_t sig_prev = YK_NONE;
        for (uint32_t a = 0; a < e->a_hi; ++a) {
            uint8_t& st = e->a_state[a];
            if (st == yk::ST_ABSENT || st == yk::ST_ALLOCATED) continue;
            st = yk::ST_PENDING;   // failed / skipped asks are tried again every cycle, like the reference
            if (!e->p_present[e->a_app[a]]) continue;
            pending.push_back(a);
            any_gang = any_gang || e->a_gang[a] != YK_NONE;
            if (auto_lattice) {
                const uint32_t g = e->a_sigid[a];
                if (g == sig_prev) ++sig_run; else { sig_longest = std::max(sig_longest, sig_run); sig_run = 1; sig_prev = g; }
            }
        }
        sig_longest = std::max(sig_longest, sig_run);
        e->cycle_has_gang = any_gang;
        if (any_gang) {   // a gang that no batch can hold is an argument error: found before anything is committed
            std::unordered_map<uint64_t, uint32_t> members;
            for (uint32_t a : pending)
                if (e->a_gang[a] != YK_NONE && ++members[((uint64_t)e->a_app[a] << 32) | e->a_gang[a]] > e->batch) gang_too_big = true;
        }
        yk::Tables& t = e->ord.t;
        t.D = e->D; t.maxA = e->maxA; t.maxP = e->maxP; t.nq = e->nq;
        t.a_req = e->a_req.p; t.a_prio = e->a_prio.data(); t.a_create = e->a_create.data(); t.a_app = e->a_app.data();
        t.a_flags = e->a_flags.data(); t.a_cause = e->a_cause.data(); t.a_gang = e->a_gang.data(); t.a_state = e->a_state.data();
        t.p_queue = e->p_queue.data(); t.p_submit = e->p_submit.data(); t.p_present = e->p_present.data();
        t.q_parent = e->q_parent.data(); t.q_guar = e->q_guar.data(); t.q_max = e->q_max.data(); t.q_alloc = e->q_alloc.data(); t.p_alloc = e->p_alloc.data();
        t.q_sort = e->q_sort.data();
        t.q_prio_offset = e->q_prio_offset.data(); t.q_prio_fence = e->q_prio_fence.data();
        t.p_user = e->p_user.data(); t.n_ul = e->n_ul; t.ul_queue = e->ul_queue.data(); t.ul_user = e->ul_user.data();
        t.ul_max = e->ul_max.data(); t.ul_alloc = e->ul_alloc.data();
        if (!gang_too_big) e->ord.begin_cycle(pending);
        e->ep_rows = false;
        if (!gang_too_big && e->share_rows && e->cfg.world <= 1 && !getenv("YK_NO_EPOCH_ROWS")) {
            // how many distinct signatures do the pending asks have?  Few: every one is swept once per epoch (ep_local =
            // its row), no per-batch device work at all
            if (e->ep_seen.size() < e->sigs.n) { e->ep_seen.assign(e->sigs.n + 1024, 0); e->ep_local.assign(e->sigs.n + 1024, 0); e->ep_stamp = 0; }
            if (++e->ep_stamp == 0) { std::fill(e->ep_seen.begin(), e->ep_seen.end(), 0); e->ep_stamp = 1; }
            e->ep_reps.clear();
            uint32_t ns = 0;
            for (uint32_t a : pending) {
                const uint32_t id = e->a_sigid[a];
                if (e->ep_seen[id] != e->ep_stamp) {
                    e->ep_seen[id] = e->ep_stamp;
                    if (ns < yk_engine::EP_MAX) { e->ep_local[id] = ns; e->ep_reps.push_back(a); }
                    if (++ns > yk_engine::EP_MAX) break;
                }
            }
            e->n_sigs = ns;
            e->ep_rows = ns > 0 && ns <= yk_engine::EP_MAX && (uint64_t)ns * 8 <= pending.size();
            e->ep_n = ns;
        }
        // a hint only (it sizes the first batch, never decides): asks are usually upserted application by application, so a long
        // run of one signature in index order promises one in the orderer's order
        e->un_hint = !gang_too_big && auto_lattice && pending.size() >= (size_t)e->un_min && sig_longest >= (size_t)e->un_min;
        if (!gang_too_big && force_lattice) {   // request-vector numbers for the lattice kernel's windows
            yklt::assign_shapes(e->cm.t, pending, e->a_shape, &e->n_shapes);
            e->lt_shape_ids = e->a_shape.data();
        }
        e->ep_uploaded = false; e->ep_landed = true;
        begin_ms = now_ms() - t_b;
    });
    hp(0);
    int rc = upload_tables(e);
    // the device scores and sorts the nodes while the helper thread still sets the orderer up
    e->order_enqueued = false;
    if (!rc) { rc = device_order(e); e->order_enqueued = rc == YK_OK && e->nlive > 0; }
    const double t_a = now_ms();
    hp(1);
    e->worker.wait();
    hp(2);
    e->st.host_ms[0] += t_a - t_start;
    e->st.host_ms[1] += begin_ms;
    if (rc) return rc;
    if (gang_too_big) return e->fail(YK_ERR_ARG, "yk_cycle: a gang has more members than the sweep batch (raise yk_config.batch)");

    Cycle c;
    c.max_bindings = max_bindings; c.out = out;
    // the first batch decides which commit the cycle starts on
    const bool ins = e->ord.insensitive;
    bool lattice = false;
    size_t bsz0 = e->batch;
    if (force_lattice) {
        const yklt::Eligibility el = yklt::eligible(e->cm.t, e->n_hi, e->n_present.data(), e->n_total.p, e->maxN, e->n_rank.data(), pending, &e->ranks_unique, &e->cycle_has_gang);
        lattice = el.ok;
        if (lattice && ins) bsz0 = e->maxA;   // the whole static order in one launch
    }
    if (auto_lattice && e->un_hint && ins) bsz0 = e->maxA;
    e->lt_plan_ready = false;
    rc = fill_batch(e, bsz0, std::max<size_t>(bsz0, e->batch), max_bindings, e->slot[0], e->st);
    if (!rc && auto_lattice && pending.size() >= (size_t)e->un_min && e->slot[0].asks.size() >= (size_t)e->un_min) {
        // Automatic: the device commit decides a uniform run (one request vector, one predicate signature) by a grid-wide sort,
        // everything else through a sequential chain that one host core still does faster (profiles/r2_lattice_*).  So the
        // cycle starts on the device exactly when the order is made of long uniform runs.  Cheap screen first -- the
        // longest run of one signature id in the first batch -- and only then the eligibility test and the shape numbers.
        const std::vector<uint32_t>& as = e->slot[0].asks;
        size_t longest = 0, run = 1;
        for (size_t i = 1; i <= as.size(); ++i) {
            if (i < as.size() && e->a_sigid[as[i]] == e->a_sigid[as[i - 1]]) { ++run; continue; }
            longest = std::max(longest, run);
            run = 1;
        }
        if (longest >= (size_t)e->un_min) {
            const yklt::Eligibility el = yklt::eligible(e->cm.t, e->n_hi, e->n_present.data(), e->n_total.p, e->maxN, e->n_rank.data(), pending, &e->ranks_unique, &e->cycle_has_gang);
            if (el.ok) {
                // signature ids double as shape numbers: equal signatures request equal vectors; two signatures with one request
                // only make the (rare, here) windowed stretches see one more shape
                e->lt_shape_ids = e->a_sigid.data();
                if (ins && e->slot[0].asks.size() < pending.size() && bsz0 < (size_t)e->maxA) {   // the whole static order in one batch
                    e->ord.unfill(e->slot[0].snap, e->slot[0].asks, 0);
                    size_t b = e->maxA;
                    rc = fill_batch(e, b, e->maxA, max_bindings, e->slot[0], e->st);
                }
                if (!rc) {
                    const size_t B0 = e->slot[0].asks.size();
                    yklt::build_meta(e->cm.t, e->lt_shape_ids, e->a_sigid.data(), e->slot[0].asks, e->h_lt_meta.p, e->h_lt_shp.p, e->h_lt_sig.p);
                    ykun::plan_segments(e->h_lt_meta.p, e->h_lt_shp.p, e->h_lt_sig.p, (int)B0, e->un_min, e->un_segs);
                    // measured costs (profiles/r2b_*, r2_lattice_*): a uniform run ~0.25 ms whatever its length (16 launches, one
                    // round trip), a windowed ask ~0.35 us, an ask on the host commit ~0.08 us
                    double dev_us = 0;
                    for (const ykun::Segment& sg : e->un_segs) dev_us += sg.uniform ? 250.0 : 0.35 * sg.len;
                    lattice = dev_us < 0.7 * 0.08 * (double)B0;
                    e->lt_plan_ready = lattice;
                }
            }
        }
    }
    if (!rc && !lattice && e->slot[0].asks.size() > e->batch) {   // the first fill was sized for the device commit
        e->ord.unfill(e->slot[0].snap, e->slot[0].asks, 0);
        size_t b = e->batch;
        rc = fill_batch(e, b, e->batch, max_bindings, e->slot[0], e->st);
    }
    e->lt_active = false;
    hp(3);
    if (!rc) {
        if (lattice) {
            e->lt_active = true;
            e->order_enqueued = false;   // consumed by lt_prepare; a hand-over sorts again from the exported tables
            e->st.lattice_cycles++;
            bool handoff = false;
            rc = run_lattice(e, c, handoff);
            if (!rc) {
                const int rce = lt_export(e);   // node tables current again, host and device
                e->lt_active = false;
                rc = rce;
            }
            if (!rc) {
                const int* h = e->h_lt_hdr.p;
                e->lt_total_subruns += (uint64_t)h[yklt::H_SUBRUNS];
                e->st.lattice_subruns += (uint64_t)h[yklt::H_SUBRUNS]; e->st.lattice_fullscans += (uint64_t)h[yklt::H_FULLSCANS];
                e->st.lattice_sorts += (uint64_t)h[yklt::H_SORTS]; e->st.lattice_elements += (uint64_t)h[yklt::H_ELEMS];
                e->st.lattice_quick += (uint64_t)h[yklt::H_QUICK];
            }
            if (!rc && handoff && c.n < max_bindings) {
                size_t b = e->batch;
                rc = fill_batch(e, b, e->batch, (size_t)max_bindings - c.n, e->slot[0], e->st);
                if (!rc) rc = run_host(e, c);
            }
        } else {
            rc = run_host(e, c);
        }
    }
    hp(4);
    // ---- always: leave host and device node tables current, persist what was bound, no ask left in flight ----
    int rc_end = YK_OK;
    if (e->lt_active) { rc_end = lt_export(e); e->lt_active = false; }
    else rc_end = end_epoch(e, false);
    e->cm.begin_epoch(e->epochW);   // nothing touched any more
    for (int k = 0; k < 4; ++k) { e->st.dbg[k] += e->cm.dbg[k]; e->cm.dbg[k] = 0; }
    for (int k = 0; k < 6; ++k) { e->st.prof[k] += e->cm.prof[k]; e->cm.prof[k] = 0; }
    if (cudaStreamSynchronize(e->stream) != cudaSuccess && !rc && !rc_end) rc_end = e->fail(YK_ERR_CUDA, "cudaStreamSynchronize at the end of the cycle");
    hp(5);
    if (rc) {
        // the cycle broke off: the bindings made so far stand (they are returned), every ask still in flight is pending
        // again, and the queue / application accounting is rebuilt from exactly the bindings returned
        e->worker.wait();
        for (Slot& sl : e->slot) { if (sl.B > 0 && sl.nchunks > 0) cudaEventSynchronize(sl.ev[(size_t)sl.nchunks - 1]); sl.asks.clear(); sl.B = 0; sl.nchunks = 0; }
        for (uint32_t a : pending) if (e->a_state[a] == yk::ST_TENTATIVE) e->a_state[a] = yk::ST_PENDING;
        for (uint32_t i = 0; i < c.n; ++i) {
            const uint32_t a = out[i].ask;
            for (int k = 0; k < e->D; ++k) {
                const int64_t r = e->a_req[(size_t)k * e->maxA + a];
                for (uint32_t q = e->p_queue[e->a_app[a]]; q != YK_NONE; q = e->q_parent[q]) e->q_alloc[(size_t)k * e->nq + q] += r;
                e->p_alloc[(size_t)k * e->maxP + e->a_app[a]] += r;
            }
            user_held_add(e, e->a_app[a], a, +1);
        }
    } else {
        e->ord.finish();
    }
    for (uint32_t a : e->ord.slow_list) {
        if (slow && n_slow && *n_slow < slow_cap) slow[(*n_slow)++] = a;
    }
    for (uint32_t a : pending) if (e->a_state[a] == yk::ST_SKIPPED) e->st.skipped++;
    *n_out = c.n;
    e->st.cycles++;
    hp(6);
    e->hp_n++;
    e->st.total_ms += now_ms() - t_start;
    return rc ? rc : rc_end;
}

extern "C" {

int yk_ask_states(yk_engine* e, uint32_t n, const uint32_t* idx, uint8_t* out) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && (!idx || !out)) return e->fail(YK_ERR_ARG, "yk_ask_states: null array");
    for (uint32_t i = 0; i < n; ++i) {
        if (idx[i] >= e->maxA) return e->fail(YK_ERR_ARG, "yk_ask_states: index beyond max_asks");
        out[i] = e->a_state[idx[i]];
    }
    return YK_OK;
}

int yk_nodes_available(yk_engine* e, uint32_t n, const uint32_t* idx, int64_t* out) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && (!idx || !out)) return e->fail(YK_ERR_ARG, "yk_nodes_available: null array");
    for (uint32_t i = 0; i < n; ++i) {
        if (idx[i] >= e->maxN) return e->fail(YK_ERR_ARG, "yk_nodes_available: index beyond max_nodes");
        for (int k = 0; k < e->D; ++k) out[(size_t)k * n + i] = e->n_avail[(size_t)k * e->maxN + idx[i]];
    }
    return YK_OK;
}

static int evaluate_phase(yk_engine* e, uint32_t ask, uint32_t node, int allocate) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (ask >= e->maxA || node >= e->maxN) return e->fail(YK_ERR_ARG, "yk_evaluate: index out of range");
    if (e->a_state[ask] == yk::ST_ABSENT || !e->n_present[node]) return YK_FAIL_ABSENT;
    int rc = upload_tables(e);
    if (rc) return rc;
    yk_evaluate_kernel<<<1, 32, 0, e->stream>>>(e->D, e->d_total.p, e->d_avail.p, e->maxN, e->d_taint.p, e->d_label.p,
                                                e->d_flags.p, e->d_areq.p, e->d_atol.p, e->d_aneed.p, e->d_adeny.p,
                                                e->d_anode.p, e->maxA, ask, node, allocate, e->d_flag.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(e->h_flag.p, e->d_flag.p, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->st.other_launches++;
    return e->h_flag[0];
}

int yk_evaluate(yk_engine* e, uint32_t ask, uint32_t node) { return evaluate_phase(e, ask, node, 1); }
int yk_evaluate_reserve(yk_engine* e, uint32_t ask, uint32_t node) { return evaluate_phase(e, ask, node, 0); }

int yk_node_scores(yk_engine* e, uint32_t n, const uint32_t* idx, double* out) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (n && (!idx || !out)) return e->fail(YK_ERR_ARG, "yk_node_scores: null array");
    if (n > e->maxN) return e->fail(YK_ERR_ARG, "yk_node_scores: more indices than max_nodes");
    for (uint32_t i = 0; i < n; ++i) if (idx[i] >= e->maxN) return e->fail(YK_ERR_ARG, "yk_node_scores: index beyond max_nodes");
    if (!n) return YK_OK;
    int rc = upload_tables(e);
    if (rc) return rc;
    memcpy(e->h_snode.p, idx, 4 * (size_t)n);
    CK(cudaMemcpyAsync(e->d_val_in.p, e->h_snode.p, 4 * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    yk_score_kernel<<<(n + 255) / 256, 256, 0, e->stream>>>(e->D, e->cfg.policy, e->w, e->d_total.p, e->d_avail.p, e->maxN,
                                                           e->d_val_in.p, (int)n, e->d_scores.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(e->h_scores.p, e->d_scores.p, 8 * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    memcpy(out, e->h_scores.p, 8 * (size_t)n);
    e->st.other_launches++;
    return YK_OK;
}

int yk_preemption_search(yk_engine* e, uint32_t nq, const uint32_t* ask, const uint32_t* node, const uint32_t* voff,
                         const int64_t* vreq, const uint32_t* start, int32_t* out) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (nq && (!ask || !node || !voff || !start || !out)) return e->fail(YK_ERR_ARG, "yk_preemption_search: null array");
    if (!nq) return YK_OK;
    const uint32_t nv = voff[nq];
    if (nv && !vreq) return e->fail(YK_ERR_ARG, "yk_preemption_search: null victim_req");
    for (uint32_t i = 0; i < nq; ++i) {
        if (ask[i] >= e->maxA || node[i] >= e->maxN || e->a_state[ask[i]] == yk::ST_ABSENT || !e->n_present[node[i]])
            return e->fail(YK_ERR_ARG, "yk_preemption_search: unknown ask or node");
        if (voff[i] > voff[i + 1]) return e->fail(YK_ERR_ARG, "yk_preemption_search: victim_off must be non-decreasing");
    }
    int rc = upload_tables(e);
    if (rc) return rc;
    const int D = e->D;
    // device buffers are kept between calls and only grow (a cudaMalloc per call costs more than the search)
    Dev<uint32_t>& d_q = e->pre_q; Dev<int64_t>& d_v = e->pre_v; Dev<int32_t>& d_o = e->pre_o;
    if (d_q.n < (size_t)nq * 4 + 1) CK(d_q.alloc(((size_t)nq * 4 + 1) * 2));
    if (d_v.n < (size_t)std::max<uint32_t>(nv, 1) * D) CK(d_v.alloc((size_t)std::max<uint32_t>(nv, 1) * D * 2));
    if (d_o.n < nq) CK(d_o.alloc((size_t)nq * 2));
    cudaStream_t s = e->stream;
    CK(cudaMemcpyAsync(d_q.p, ask, 4 * (size_t)nq, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_q.p + nq, node, 4 * (size_t)nq, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_q.p + 2 * (size_t)nq, voff, 4 * ((size_t)nq + 1), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_q.p + 3 * (size_t)nq + 1, start, 4 * (size_t)nq, cudaMemcpyHostToDevice, s));
    if (nv) CK(cudaMemcpyAsync(d_v.p, vreq, 8 * (size_t)nv * D, cudaMemcpyHostToDevice, s));
    const int threads = 128, warps_per_block = threads / 32;
    yk_preempt_kernel<<<(nq + warps_per_block - 1) / warps_per_block, threads, 0, s>>>(
        D, e->d_total.p, e->d_avail.p, e->maxN, e->d_taint.p, e->d_label.p, e->d_flags.p, e->d_areq.p, e->d_atol.p,
        e->d_aneed.p, e->d_adeny.p, e->d_anode.p, e->maxA, (int)nq, d_q.p, d_q.p + nq, d_q.p + 2 * (size_t)nq, d_v.p,
        std::max<uint32_t>(nv, 1), d_q.p + 3 * (size_t)nq + 1, d_o.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d_o.p, 4 * (size_t)nq, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    e->st.other_launches++;
    return YK_OK;
}

int yk_set_exchange(yk_engine* e, yk_allgather_fn fn, void* ctx) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    e->xfn = fn; e->xctx = ctx;
    return YK_OK;
}

int yk_peer_export(yk_engine* e, yk_peer_handles* out) {
    if (!e || !out) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)out->blob[0], e->slot[0].d_fit.p));
    CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)out->blob[1], e->slot[1].d_fit.p));
    CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)out->blob[2], e->d_sync.p));
    return YK_OK;
}

int yk_peer_import(yk_engine* e, uint32_t peer, const yk_peer_handles* in) {
    if (!e || !in) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    if (peer >= 8 || peer >= e->cfg.world || peer == e->cfg.rank) return e->fail(YK_ERR_ARG, "yk_peer_import: bad peer rank");
    if (e->peer_open[peer]) return e->fail(YK_ERR_STATE, "yk_peer_import: peer already imported");
    cudaIpcMemHandle_t h[3];
    memcpy(h, in->blob, sizeof(h));
    void* p0 = nullptr; void* p1 = nullptr; void* p2 = nullptr;
    CK(cudaIpcOpenMemHandle(&p0, h[0], cudaIpcMemLazyEnablePeerAccess));
    CK(cudaIpcOpenMemHandle(&p1, h[1], cudaIpcMemLazyEnablePeerAccess));
    CK(cudaIpcOpenMemHandle(&p2, h[2], cudaIpcMemLazyEnablePeerAccess));
    e->peer_fit[0][peer] = (uint32_t*)p0; e->peer_fit[1][peer] = (uint32_t*)p1; e->peer_sync[peer] = (uint32_t*)p2;
    e->peer_open[peer] = true;
    return YK_OK;
}

int yk_peer_enable(yk_engine* e) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    const uint32_t world = e->cfg.world, rank = e->cfg.rank;
    if (world < 2 || world > 8) return e->fail(YK_ERR_ARG, "yk_peer_enable: world must be 2..8");
    for (uint32_t p = 0; p < world; ++p)
        if (p != rank && !e->peer_open[p]) return e->fail(YK_ERR_STATE, "yk_peer_enable: a peer has not been imported");
    e->peer_fit[0][rank] = e->slot[0].d_fit.p; e->peer_fit[1][rank] = e->slot[1].d_fit.p; e->peer_sync[rank] = e->d_sync.p;
    for (Slot& sl : e->slot) CK(cudaMemset(sl.d_fit.p, 0xFF, sl.d_fit.n * sizeof(uint32_t)));   // slots start wiped
    e->p2p = true;
    return YK_OK;
}

int yk_stats(yk_engine* e, yk_stats_t* out) {
    if (!e || !out) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    *out = e->st;
    return YK_OK;
}

int yk_stats_reset(yk_engine* e) {
    if (!e) return YK_ERR_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    e->st = yk_stats_t{};
    return YK_OK;
}

}  // extern "C"
