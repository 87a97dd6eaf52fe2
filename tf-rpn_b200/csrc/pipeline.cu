// pipeline.cu -- host-buffer steps of the hot path, pipelined over PCIe.
//
// This is the call site the reference drives from Keras' generator thread (utils/train_utils.py:67-82,
// trainer.py:48-49,64-69): every step a padded host batch goes in and (bbox_deltas, bbox_labels) come
// out; predictor.py:48-60 does the same with the head outputs.  Dense, a C2 step would move ~11 MB each way
// while its kernels take ~0.05 ms, so this file (a) keeps several steps in flight and (b) moves fewer bytes.
//
// (a) Each in-flight step owns a SLOT: device + page-locked staging, its own copy-in / proposal / copy-out
//     streams, events.  The target kernels of all slots share one stream (they share the handle's workspace).
//     Results are bit-identical to the separate calls: images are independent and the counter RNG is keyed by
//     the global image index.  A depth-1 pipeline is the synchronous step (tfrpn_rpn_step_host): chunked over
//     images so that its own copies overlap its kernels, dense in both directions.
//
// (b) Measured at C2 (profiles/r2d_*, r2_scale/): 11.1 MB in / 11.5 MB out -> 3.6 / 3.1 MB per step.
//   two-phase proposals   rpn_reg is 80 % of the input bytes and NMS decodes ~560 of its 8649 rows per image.
//                         Only the scores are copied; a rank launch returns the entry index of the first ranks;
//                         the rows of the first `gather_rows` ranks are gathered ON THE HOST from the caller's
//                         tensor -- page-locked or pageable, read in place -- into a compact block that follows
//                         in one copy; the NMS launch reads rows by rank.  SM-issued loads of single rows over
//                         PCIe run at ~0.4-0.6 G rows/s (tools/src/pcie_rows.cu, pcie_gather.cu): as slow as
//                         copying the whole tensor, which is why the host gathers when it has the cores
//                         (gather_rows_kernel is the device-side variant for hosts that have not).
//   compact bbox_deltas   exactly zero outside the <= total_pos sampled positives (train_utils.py:137): only those
//                         rows come back and host threads scatter them into the dense array when the step is
//                         retired (optionally bbox_labels too, as codes of its entries != -1).
//
// Host stages run on a SERVICE THREAD (polls the rank-copy events, gathers, enqueues the tail of the step) and a
// WORKER POOL (gather, scatter, staging copies): cudaLaunchHostFunc costs ~150 us of stream time per call on this
// box and serialises across streams (tools/src/hostfunc_lat.cu).  Device time stamps of every stage:
// TFRPN_PIPE_TRACE=1 + tfrpn_pipeline_trace (tools/pipe_trace.py).
#include <sched.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <chrono>

#include "common.cuh"

namespace tfrpn {
size_t targets_workspace_bytes(int B, int N, int G);  // targets.cu
int launch_targets(tfrpn_handle h, const float* anchors, const float* gt_boxes, const int32_t* gt_labels, int B, int N,
                   int G, const tfrpn_target_cfg* cfg, float* deltas, float* labels, int32_t* pos_idx,
                   float* pos_deltas, int32_t* lbl_code, const tfrpn_target_debug* dbg, tfrpn_stream s);
int scatter_rows_to_host_enqueue(int32_t* prev_idx, int prev_tp, const int32_t* idx, const float* rows, int tp, int B, int N,
                                 float* dense_host_dev_alias, int stride_prev, cudaStream_t st);
int proposals_enqueue(tfrpn_handle h, const float* rpn_reg, const float* rpn_cls, const float* anchors, int B, int N,
                      const tfrpn_proposal_cfg* cfg, float* out_boxes, float* out_scores, int32_t* valid,
                      int32_t* keep_idx_or_null, unsigned long long* rows_fetched_or_null, cudaStream_t st);   // proposals.cu
// the two-phase flow (proposals.cu): ranks from the scores, rows gathered by the host, NMS over the gathered rows
int proposals_rank_cap();
bool proposals_two_phase_applies(int B, int N, const tfrpn_proposal_cfg* cfg);
int proposals_rank_enqueue(tfrpn_handle h, const float* rpn_cls, int B, int N, const tfrpn_proposal_cfg* cfg,
                           int32_t* rank_idx, int32_t* rank_n, int32_t* rank_more, cudaStream_t st);
int proposals_presorted_enqueue(tfrpn_handle h, const float* rpn_reg_or_null, const float* reg_compact, int compact_rows,
                                int compact_stride, const float* rpn_cls, const float* anchors, int B, int N,
                                const tfrpn_proposal_cfg* cfg, int32_t* rank_idx, int32_t* rank_n, int32_t* rank_more,
                                float* out_boxes, float* out_scores, int32_t* valid, int32_t* keep_idx_or_null,
                                int32_t* redo_flags, unsigned int* mask_ws_or_null, cudaStream_t st);
size_t proposals_mask_bytes(int B, int rows);
int proposals_redo_enqueue(tfrpn_handle h, const float* rpn_reg, const float* rpn_cls, const float* anchors, int B, int N,
                           const tfrpn_proposal_cfg* cfg, float* out_boxes, float* out_scores, int32_t* valid,
                           int32_t* keep_idx_or_null, const int32_t* redo_flags, unsigned long long* rows_fetched_or_null,
                           cudaStream_t st);
int proposals_gather_enqueue(const float* reg_pinned_dev, const int32_t* rank_idx, const int32_t* rank_n, int B, int N,
                             int rows, float* dst, int stride, unsigned long long* counter_or_null, cudaStream_t st);
}

namespace {

constexpr int MAX_CHUNKS = 8;
constexpr int MAX_DEPTH = 16;
constexpr int COMPACT_MAX_POS = 256;   // sparse result form is used when total_pos_bboxes <= this ...
constexpr int COMPACT_MAX_Q = 512;     // ... and total_pos_bboxes + total_neg_bboxes <= this

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

bool is_pinned(const void* p) {
    cudaPointerAttributes attr;
    bool r = cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    return r;
}

// ---- host worker pool -------------------------------------------------------------------------------
// run(chunks, f) calls f(0) .. f(chunks - 1) on the pool's threads and the calling thread and returns when
// all are done.  Callers: the CUDA host-function thread (row gather, delta expansion) and the submitting
// thread (staging copies of pageable inputs); one job at a time.  Workers spin briefly for the next job
// (jobs arrive every ~50 us while a pipeline is busy) and then sleep on a condition variable.
class HostPool {
    struct Job {
        const std::function<void(int)>* fn;
        int chunks;
        std::atomic<int> next{0}, done{0};
    };
    std::vector<std::thread> workers_;
    std::mutex run_mu_, mu_;
    std::condition_variable cv_;
    std::shared_ptr<Job> cur_;             // guarded by mu_
    std::atomic<unsigned long long> gen_{0};
    std::atomic<bool> stop_{false};

    static void relax() {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#else
        std::this_thread::yield();
#endif
    }
    static void work(Job& j) {
        for (;;) {
            const int c = j.next.fetch_add(1, std::memory_order_relaxed);
            if (c >= j.chunks) return;
            (*j.fn)(c);
            j.done.fetch_add(1, std::memory_order_release);
        }
    }
    void loop() {
        unsigned long long seen = 0;
        for (;;) {
            int spins = 0;
            while (gen_.load(std::memory_order_acquire) == seen && !stop_.load(std::memory_order_relaxed)) {
                if (++spins < 20000) { relax(); continue; }
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return gen_.load(std::memory_order_acquire) != seen || stop_.load(); });
            }
            if (stop_.load()) return;
            std::shared_ptr<Job> j;
            {
                std::lock_guard<std::mutex> lk(mu_);
                seen = gen_.load(std::memory_order_acquire);
                j = cur_;
            }
            if (j) work(*j);
        }
    }

  public:
    explicit HostPool(int threads) {
        for (int i = 1; i < threads; ++i) workers_.emplace_back([this] { loop(); });
    }
    ~HostPool() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_.store(true);
        }
        cv_.notify_all();
        for (auto& t : workers_) t.join();
    }
    void run(int chunks, const std::function<void(int)>& f) {
        if (chunks <= 0) return;
        if (workers_.empty() || chunks == 1) { for (int c = 0; c < chunks; ++c) f(c); return; }
        std::lock_guard<std::mutex> one(run_mu_);
        auto j = std::make_shared<Job>();
        j->fn = &f; j->chunks = chunks;
        {
            std::lock_guard<std::mutex> lk(mu_);
            cur_ = j;
            gen_.fetch_add(1, std::memory_order_release);
        }
        cv_.notify_all();
        work(*j);
        while (j->done.load(std::memory_order_acquire) < chunks) relax();
        std::lock_guard<std::mutex> lk(mu_);
        cur_.reset();
    }
    // memcpy split over the pool (pageable staging copies of a few MB)
    void copy(void* dst, const void* src, size_t bytes) {
        const size_t piece = 256 * 1024;
        const int chunks = (int)((bytes + piece - 1) / piece);
        if (chunks <= 1) { memcpy(dst, src, bytes); return; }
        run(chunks, [&](int c) {
            const size_t o = (size_t)c * piece;
            memcpy(static_cast<char*>(dst) + o, static_cast<const char*>(src) + o, bytes - o < piece ? bytes - o : piece);
        });
    }
};

// Staging layout of a slot; the device and the pinned block mirror each other.  Inputs are contiguous
// and results are contiguous, so a step whose host buffers ARE the slot's pinned block (acquired mode)
// is one H2D and one D2H copy -- on this link several copies per direction cost 30 % of the duplex
// rate (tools/src/pcie_pattern.cu: 309 us vs 231 us per C2 step).
struct Layout {
    size_t gt, gl, cls, small_end, reg, in_end; // inputs: the small ones first, the head's regression output last
    size_t d, l, ob, os, v, k, pc, rf, dense_end;   // results (pc: rows of rpn_reg pulled; rf: redo flags)
    size_t comp, comp_end;                      // sparse targets (label codes, row indices, rows: packed at submit)
    size_t pci;                                 // device side: row indices the slot's dense host array still holds (device expansion)
    size_t ri, rn, rm, rank_end, rc, mk, total; // two-phase: rank indices / counts / more flags (D2H), compact rows (H2D), NMS matrix
};

// everything the later stages of the step in flight need (filled by pipe_submit, read by the service thread)
struct Step {
    bool do_t = false, do_p = false, acquired = false, compact = false, two_phase = false, sparse_labels = false;
    bool device_expand = false;         // the dense bbox_deltas host array is kept up to date by a kernel (no host scatter)
    bool reg_pinned = false;            // the caller's rpn_reg is page-locked: the device can read it (redo pulls rows)
    bool device_gather = false;         // the rows are gathered by a kernel reading the page-locked tensor (no host stage)
    int B = 0, N = 0, G = 0, P = 0, GR = 0, total_pos = 0, Q = 0;
    Layout L = {};
    size_t cl = 0, ci = 0, cd = 0;      // sparse targets inside [L.comp, L.comp_end): label codes (B,Q), row indices (B,total_pos), rows
    const float* anchors = nullptr;
    tfrpn_proposal_cfg pcfg = {};
    const float* reg_host = nullptr;    // the caller's rpn_reg (any host memory): source of the row gather
    const float* reg_dev = nullptr;     // its device alias when page-locked
    float* dense_dst = nullptr;         // where the dense bbox_deltas go: the slot's own array, or the caller's buffer
};

struct Slot {
    char* dev = nullptr; size_t dev_bytes = 0;
    char* pin = nullptr; size_t pin_bytes = 0;
    cudaStream_t s_in = nullptr, s_prop = nullptr, s_out = nullptr;   // this slot's copy-in, proposal and copy-out streams
    cudaEvent_t ev_gt = nullptr, ev_prop = nullptr, ev_done = nullptr, ev_rank = nullptr;
    cudaEvent_t ev_in[MAX_CHUNKS] = {}, ev_tgt[MAX_CHUNKS] = {};
    long long ticket = -1;          // ticket in flight in this slot (-1 = free)
    cudaEvent_t tr[8] = {};         // TFRPN_PIPE_TRACE: timing events (h2d, targets, proposals, d2h: begin / end)
    float tr_ms[8] = {};            // ... of the last step retired from this slot, ms since the pipeline was created
    long long tr_ticket = -1;
    float gather_ms = 0.f, expand_ms = 0.f;   // host time of the two service stages (tracing)
    Step step;
    // service thread -> submitting thread
    std::atomic<int> svc_pending{0};   // stages the service thread still owes for the step in flight
    int svc_rc = 0;
    char svc_err[256] = "";
    long long gathered = 0;            // rows of rpn_reg gathered for the step in flight
    bool pulled = false;               // the redo kernel counts the rows it pulls from the pinned tensor at L.pc
    float* labels_dst = nullptr;       // where the dense bbox_labels go: the slot's own array, or the caller's buffer
    // incremental expansion of the sparse targets into the slot's own dense arrays
    bool dense_clean = false;          // pin + L.d holds zeros except the rows listed in prev_idx, pin + L.l holds -1
    int pB = 0, pN = 0, pTP = 0, pQ = 0;   //   except the entries coded in prev_lbl
    size_t p_off_d = 0;
    std::vector<int32_t> prev_idx, prev_lbl;
    bool dev_clean = false;            // ... or the same invariant with the row list kept on the device (L.pci): device expansion
    int dB = 0, dN = 0;
    size_t d_off_d = 0;
    struct Copy { void* dst; const void* src; size_t bytes; } copies[8 + 2 * MAX_CHUNKS];
    int n_copies = 0;
    void defer(void* d, const void* s, size_t b) { copies[n_copies].dst = d; copies[n_copies].src = s; copies[n_copies].bytes = b; ++n_copies; }
};

// A stage of a step that runs on the host between two device stages.  CUDA host functions would be the
// obvious tool, but one costs ~150 us of stream time on this box and they run one at a time
// (tools/src/hostfunc_lat.cu), i.e. 300 us per step.  Instead one service thread per pipeline polls the
// stage's event (cudaEventQuery), does the host work on the worker pool and enqueues what follows.
enum { STAGE_GATHER = 0 };
struct StageJob { int kind; Slot* slot; };

}  // namespace

struct tfrpn_pipe {
    tfrpn_handle h = nullptr;
    int depth = 1;
    cudaStream_t s_tgt = nullptr;   // target kernels of every slot (they share the handle's workspace)
    cudaEvent_t ev_after = nullptr;
    bool trace = false;             // TFRPN_PIPE_TRACE=1 (read when the handle was created)
    cudaEvent_t ev_base = nullptr;  // time origin of the trace
    std::unique_ptr<HostPool> pool;
    // service threads (jobs of different slots are independent; each job stays with the thread that took it)
    std::thread svc[2];
    int n_svc = 0;
    std::mutex svc_mu;
    std::condition_variable svc_cv;
    std::deque<StageJob> svc_inbox;
    bool svc_stop = false;
    Slot slots[MAX_DEPTH];
    long long next_ticket = 0;
    int acq_B = 0, acq_N = 0, acq_G = 0, acq_P = 0;   // shape of the slot handed out by the last acquire()
    bool acq_live = false;
    long long last_h2d = 0, last_d2h = 0;             // bytes copied by the last submitted step
    long long last_pulled = 0;                        // bytes of rpn_reg rows gathered / pulled for the last RETIRED step
    // TFRPN_PIPE_OPT_STABLE_OUTPUTS: the caller promises that the bbox_deltas arrays it passes to submit() are written by
    // this pipeline only, so an array seen before still holds zeros plus the rows of its last step (no 4*B*N*4-byte memset)
    bool stable_outputs = false;
    struct CallerDense { float* ptr; int B, N, TP; std::vector<int32_t> idx; };
    std::vector<CallerDense> caller_dense;            // most recent first, at most 64 arrays
    int gather_rows = 640;                            // rows of rpn_reg per image the two-phase transfer sends (adapts)
    bool gather_adapt = true;
    bool device_gather = false;                       // page-locked tensors: gather on the device instead of the host
    bool sparse_labels = false;                       // bbox_labels returns as codes (scattered by host threads) instead of densely
    bool device_expand = false;                       // acquired slots: a kernel scatters the bbox_deltas rows into the pinned array
};

namespace tfrpn {

static Layout make_layout(int B, int N, int G, int P) {
    Layout L;
    size_t o = 0;
    L.gt = o;  o += align256((size_t)B * G * 16);
    L.gl = o;  o += align256((size_t)B * G * 4);
    L.cls = o; o += align256((size_t)B * N * 4);
    L.small_end = o;
    L.reg = o; o += align256((size_t)B * N * 16);
    L.in_end = o;
    L.d = o;   o += align256((size_t)B * N * 16);
    L.l = o;   o += align256((size_t)B * N * 4);
    L.ob = o;  o += align256((size_t)B * P * 16);
    L.os = o;  o += align256((size_t)B * P * 4);
    L.v = o;   o += align256((size_t)B * 4);
    L.k = o;   o += align256((size_t)B * P * 4);
    L.pc = o;  o += 256;
    L.rf = o;  o += align256((size_t)B * 4);
    L.dense_end = o;
    L.comp = o; o += align256((size_t)B * COMPACT_MAX_Q * 4) + align256((size_t)B * COMPACT_MAX_POS * 4) +
                     align256((size_t)B * COMPACT_MAX_POS * 16);
    L.comp_end = o;
    L.pci = o; o += align256((size_t)B * COMPACT_MAX_POS * 4);
    L.ri = o;  o += align256((size_t)B * proposals_rank_cap() * 4);
    L.rn = o;  o += align256((size_t)B * 4);
    L.rm = o;  o += align256((size_t)B * 4);
    L.rank_end = o;
    L.rc = o;  o += align256((size_t)B * proposals_rank_cap() * 16);   // sized for the cap: gather_rows adapts
    L.mk = o;  o += align256(proposals_mask_bytes(B, proposals_rank_cap()));   // (device side only)
    L.total = o;
    return L;
}

// Rows of rpn_reg gathered per image.  NMS consumes candidates in rounds of 128 ranks; 640 covers the ~560 +- 30
// ranks a C2-like image needs for 300 proposals.  The count adapts: when more than 1/16 of a step's images had to
// be redone (their NMS wanted more rows), the pipeline gathers 128 rows more from then on (up to the rank cap).
static int initial_gather_rows(tfrpn_handle h) {
    int r = h->opts.pipe_gather_rows > 0 ? h->opts.pipe_gather_rows : 640;
    return r > proposals_rank_cap() ? proposals_rank_cap() : r;
}

static void svc_push(tfrpn_pipe* p, int kind, Slot* s) {
    {
        std::lock_guard<std::mutex> lk(p->svc_mu);
        p->svc_inbox.push_back({kind, s});
    }
    p->svc_cv.notify_one();
}

// ---- host stage 1: the candidate rows of rpn_reg, in rank order, into the slot's pinned compact block ----
static void gather_rows(tfrpn_pipe* p, Slot& s) {
    const Step& st = s.step;
    const int32_t* n_of = reinterpret_cast<const int32_t*>(s.pin + st.L.rn);
    const int32_t* idx_of = reinterpret_cast<const int32_t*>(s.pin + st.L.ri);
    float* dst_of = reinterpret_cast<float*>(s.pin + st.L.rc);
    const int cap = proposals_rank_cap(), rows = st.GR, N = st.N, B = st.B;
    constexpr int PIECE = 4;        // images per chunk
    std::atomic<long long> total{0};
    p->pool->run((B + PIECE - 1) / PIECE, [&](int c) {
        constexpr int AHEAD = 24;
        long long mine = 0;
        for (int b = c * PIECE; b < B && b < (c + 1) * PIECE; ++b) {
            const int n = n_of[b] < rows ? n_of[b] : rows;
            const int32_t* idx = idx_of + (size_t)b * cap;
            const float* src = st.reg_host + (size_t)b * N * 4;
            float* dst = dst_of + (size_t)b * rows * 4;
            for (int r = 0; r < n && r < AHEAD; ++r) __builtin_prefetch(src + (size_t)idx[r] * 4, 0, 0);
            for (int r = 0; r < n; ++r) {
                if (r + AHEAD < n) __builtin_prefetch(src + (size_t)idx[r + AHEAD] * 4, 0, 0);
                memcpy(dst + (size_t)r * 4, src + (size_t)idx[r] * 4, 16);
            }
            mine += n;
        }
        total.fetch_add(mine, std::memory_order_relaxed);
    });
    s.gathered = total.load();
}

// ---- host stage 2: the sparse targets into the dense (B,N,4) bbox_deltas and (B,N) bbox_labels host arrays ----
static void expand_targets(tfrpn_pipe* p, Slot& s, float* labels_dst) {
    const Step& st = s.step;
    float* own_dense = reinterpret_cast<float*>(s.pin + st.L.d);
    const bool own = st.dense_dst == own_dense;
    const int B = st.B, N = st.N, TP = st.total_pos, Q = st.Q, pTP = s.pTP, pQ = s.pQ;
    // (a dense bbox_labels copy overwrites the slot's label array: the sparse bookkeeping restarts, pQ = 0 means "not -1-filled")
    const bool reuse = own && s.dense_clean && s.pB == B && s.pN == N && s.p_off_d == st.L.d && (!st.sparse_labels || s.pQ > 0);
    const int32_t* idx = reinterpret_cast<const int32_t*>(s.pin + st.ci);
    const float* rows = reinterpret_cast<const float*>(s.pin + st.cd);
    const int32_t* codes = reinterpret_cast<const int32_t*>(s.pin + st.cl);
    const int32_t* prev = reuse ? s.prev_idx.data() : nullptr;
    const int32_t* prev_l = reuse ? s.prev_lbl.data() : nullptr;
    float* dense = st.dense_dst;
    int prev_tp = pTP;
    tfrpn_pipe::CallerDense* known = nullptr;
    if (!own && p->stable_outputs) {   // a caller's array this pipeline filled before: reset only the rows it wrote then
        for (auto& cd : p->caller_dense)
            if (cd.ptr == dense && cd.B == B && cd.N == N) { known = &cd; break; }
        if (known) { prev = known->idx.data(); prev_tp = known->TP; }
    }
    constexpr int PIECE = 2;        // images per chunk
    p->pool->run((B + PIECE - 1) / PIECE, [&](int c) {
        const int b0 = c * PIECE, nb = (B - b0 < PIECE) ? B - b0 : PIECE;
        tfrpn_expand_targets_host(idx + (size_t)b0 * TP, rows + (size_t)b0 * TP * 4, nb, N, TP,
                                  prev ? prev + (size_t)b0 * prev_tp : nullptr, prev_tp, dense + (size_t)b0 * N * 4);
        if (st.sparse_labels)
            tfrpn_expand_labels_host(codes + (size_t)b0 * Q, nb, N, Q, prev_l ? prev_l + (size_t)b0 * pQ : nullptr, pQ,
                                     labels_dst + (size_t)b0 * N);
    });
    if (own) {
        s.prev_idx.assign(idx, idx + (size_t)B * TP);
        s.prev_lbl.assign(codes, codes + (size_t)B * Q);
        s.pB = B; s.pN = N; s.pTP = TP; s.pQ = Q; s.p_off_d = st.L.d;
        s.dense_clean = true;
    } else if (p->stable_outputs) {
        if (known) {
            known->TP = TP;
            known->idx.assign(idx, idx + (size_t)B * TP);
        } else {
            if (p->caller_dense.size() >= 64) p->caller_dense.pop_back();
            p->caller_dense.insert(p->caller_dense.begin(), tfrpn_pipe::CallerDense{dense, B, N, TP, std::vector<int32_t>(idx, idx + (size_t)B * TP)});
        }
    }
}

// The tail of a step: [two-phase: compact rows H2D, NMS over them, redo of flagged images] -> results D2H.
// Called by the submitting thread, or by the service thread once the rows have been gathered.
static int enqueue_tail(tfrpn_pipe* p, Slot& s) {
    tfrpn_handle h = p->h;
    const Step& st = s.step;
    const Layout& L = st.L;
    char* d = s.dev;
    char* pin = s.pin;
    const int B = st.B, N = st.N, GR = st.GR;
    auto mark = [&](int i, cudaStream_t stream) { if (p->trace) cudaEventRecord(s.tr[i], stream); };
    if (st.two_phase) {
        const float* cls = reinterpret_cast<const float*>(d + L.cls);
        int32_t* ri = reinterpret_cast<int32_t*>(d + L.ri);
        int32_t* rn = reinterpret_cast<int32_t*>(d + L.rn);
        int32_t* rm = reinterpret_cast<int32_t*>(d + L.rm);
        int32_t* rf = reinterpret_cast<int32_t*>(d + L.rf);
        float* ob = reinterpret_cast<float*>(d + L.ob);
        float* os = reinterpret_cast<float*>(d + L.os);
        int32_t* v = reinterpret_cast<int32_t*>(d + L.v);
        int32_t* k = reinterpret_cast<int32_t*>(d + L.k);
        unsigned long long* pc = reinterpret_cast<unsigned long long*>(d + L.pc);   // (zeroed by pipe_submit)
        if (st.device_gather) {
            if (int rc = proposals_gather_enqueue(st.reg_dev, ri, rn, B, N, GR, reinterpret_cast<float*>(d + L.rc), GR, pc, s.s_prop))
                return rc;
        } else {
            TFRPN_CHECK_CUDA(cudaMemcpyAsync(d + L.rc, pin + L.rc, (size_t)B * GR * 16, cudaMemcpyHostToDevice, s.s_prop));
        }
        if (int rc = proposals_presorted_enqueue(h, nullptr, reinterpret_cast<const float*>(d + L.rc), GR, GR, cls, st.anchors,
                                                 B, N, &st.pcfg, ri, rn, rm, ob, os, v, k, rf, reinterpret_cast<unsigned int*>(d + L.mk), s.s_prop)) return rc;
        // images whose NMS ran out of gathered rows (rare): the unfiltered kernel redoes them, reading the rows it
        // needs straight from the caller's page-locked tensor; a pageable tensor is handled when the step is retired
        if (st.reg_pinned) {
            if (int rc = proposals_redo_enqueue(h, st.reg_dev, cls, st.anchors, B, N, &st.pcfg, ob, os, v, k, rf, pc, s.s_prop))
                return rc;
        }
    }
    if (st.do_p) {
        mark(5, s.s_prop);
        TFRPN_CHECK_CUDA(cudaEventRecord(s.ev_prop, s.s_prop));
        TFRPN_CHECK_CUDA(cudaStreamWaitEvent(s.s_out, s.ev_prop, 0));
    }
    mark(6, s.s_out);
    // results: ONE D2H copy of the contiguous range [labels | proposal results | redo flags | compact rows] when the
    // deltas travel in compact form; otherwise dense targets (acquired: one range; caller buffers: copied per chunk
    // by pipe_submit) and the small proposal results
    if (st.compact) {
        const size_t lo = !st.sparse_labels ? L.l : (st.do_p ? L.ob : L.rf);
        const size_t hi = st.device_expand ? L.dense_end : st.cd + (size_t)B * st.total_pos * 16;
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(pin + lo, d + lo, hi - lo, cudaMemcpyDeviceToHost, s.s_out));
    } else if (st.acquired) {
        const size_t lo = st.do_t ? L.d : L.ob, hi = st.do_p ? L.dense_end : L.ob;
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(pin + lo, d + lo, hi - lo, cudaMemcpyDeviceToHost, s.s_out));
    } else if (st.do_p) {   // the small proposal results come back in ONE D2H copy through pinned staging
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(pin + L.ob, d + L.ob, L.dense_end - L.ob, cudaMemcpyDeviceToHost, s.s_out));
    }
    mark(7, s.s_out);
    TFRPN_CHECK_CUDA(cudaEventRecord(s.ev_done, s.s_out));
    return 0;
}

static void svc_fail(Slot& s, int rc) {
    s.svc_rc = rc;
    snprintf(s.svc_err, sizeof(s.svc_err), "%s", tfrpn_last_error());
    s.svc_pending.store(0, std::memory_order_release);   // nothing more will happen for this step
}

static void service_loop(tfrpn_pipe* p) {
    cudaSetDevice(p->h->device);
    std::vector<StageJob> pending;
    for (;;) {
        {
            std::unique_lock<std::mutex> lk(p->svc_mu);
            if (pending.empty()) p->svc_cv.wait(lk, [&] { return p->svc_stop || !p->svc_inbox.empty(); });
            if (p->svc_stop && pending.empty() && p->svc_inbox.empty()) return;
            // (with two threads a thread that already holds a job leaves the inbox to the other one)
            while (!p->svc_inbox.empty() && (p->n_svc == 1 || pending.empty())) {
                pending.push_back(p->svc_inbox.front());
                p->svc_inbox.pop_front();
            }
        }
        bool progress = false;
        for (size_t i = 0; i < pending.size();) {
            Slot& s = *pending[i].slot;
            const cudaError_t q = cudaEventQuery(s.ev_rank);
            if (q == cudaErrorNotReady) { ++i; continue; }
            const int kind = pending[i].kind;
            pending.erase(pending.begin() + i);
            progress = true;
            if (q != cudaSuccess) { svc_fail(s, cuda_fail(q, "pipeline service thread: cudaEventQuery")); continue; }
            if (s.svc_rc != 0) continue;   // an earlier stage of this step failed
            const auto t0 = std::chrono::steady_clock::now();
            (void)kind;
            gather_rows(p, s);
            s.gather_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
            if (int rc = enqueue_tail(p, s)) { svc_fail(s, rc); continue; }
            s.svc_pending.fetch_sub(1, std::memory_order_release);
        }
        if (!progress) {
#if defined(__x86_64__) || defined(__i386__)
            __builtin_ia32_pause();
#endif
        }
    }
}

static int slot_finish(tfrpn_pipe* p, Slot& s);

void pipe_destroy(tfrpn_pipe* p) {
    if (!p) return;
    DeviceGuard guard(p->h->device);
    for (int i = 0; i < p->depth; ++i) slot_finish(p, p->slots[i]);
    if (p->n_svc > 0) {
        {
            std::lock_guard<std::mutex> lk(p->svc_mu);
            p->svc_stop = true;
        }
        p->svc_cv.notify_all();
        for (int i = 0; i < p->n_svc; ++i) if (p->svc[i].joinable()) p->svc[i].join();
    }
    for (int i = 0; i < p->depth; ++i)
        for (cudaStream_t s : {p->slots[i].s_in, p->slots[i].s_prop, p->slots[i].s_out})
            if (s) cudaStreamSynchronize(s);
    if (p->s_tgt) { cudaStreamSynchronize(p->s_tgt); cudaStreamDestroy(p->s_tgt); }
    if (p->ev_after) cudaEventDestroy(p->ev_after);
    if (p->ev_base) cudaEventDestroy(p->ev_base);
    for (int i = 0; i < p->depth; ++i) {
        Slot& s = p->slots[i];
        for (cudaStream_t st : {s.s_in, s.s_prop, s.s_out}) if (st) cudaStreamDestroy(st);
        if (s.dev) cudaFree(s.dev);
        if (s.pin) cudaFreeHost(s.pin);
        for (cudaEvent_t e : {s.ev_gt, s.ev_prop, s.ev_done, s.ev_rank}) if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : s.tr) if (e) cudaEventDestroy(e);
        for (int c = 0; c < MAX_CHUNKS; ++c) {
            if (s.ev_in[c]) cudaEventDestroy(s.ev_in[c]);
            if (s.ev_tgt[c]) cudaEventDestroy(s.ev_tgt[c]);
        }
    }
    cudaGetLastError();
    delete p;
}

static int pipe_create(tfrpn_handle h, int depth, tfrpn_pipe** out) {
    if (!h || !out) return fail(TFRPN_ERR_BAD_ARG, "pipeline_create: null pointer");
    if (depth < 1 || depth > MAX_DEPTH) return fail(TFRPN_ERR_BAD_ARG, "pipeline_create: depth must be 1..%d", MAX_DEPTH);
    TFRPN_ENTER(h);
    tfrpn_pipe* p = new tfrpn_pipe();
    p->h = h;
    p->depth = depth;
    const char* lws = getenv("LOCAL_WORLD_SIZE");
    const int local_ranks = lws && atoi(lws) > 0 ? atoi(lws) : 1;
    int threads = h->opts.host_threads;
    if (threads <= 0) {
        // default: half of this process's share of the cores it may run on, at most 8 -- the data loader and the
        // other ranks of a multi-GPU job (torchrun exports LOCAL_WORLD_SIZE) need theirs
        int hw = (int)std::thread::hardware_concurrency();
        cpu_set_t set;
        if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) hw = CPU_COUNT(&set);
        const int share = hw / local_ranks;
        threads = share / 2 < 1 ? 1 : (share / 2 > 8 ? 8 : share / 2);
    }
    // TFRPN_PIPE_GATHER = host | device (default: host when the pool has >= 4 threads, else device)
    p->device_gather = h->opts.pipe_gather == 2 || (h->opts.pipe_gather == 0 && threads < 4);
    // bbox_labels is -1 except <= total_pos + total_neg entries per image: as codes it is 65 KB instead of 2.2 MB per C2
    // step, but the host then scatters 2 x 16 k floats per step into DRAM-resident arrays (~45 us on 8 threads), which
    // costs a lone GPU more than the DMA it saves.  Worth it when many GPUs share the host's PCIe / memory bandwidth.
    p->sparse_labels = h->opts.pipe_sparse_labels > 0;
    (void)local_ranks;
    // TFRPN_PIPE_EXPAND = host (default) | device: who scatters the compact bbox_deltas rows into the dense host array.
    // Measured (profiles/r2_scale/e2e_policies_8gpu.txt): a lone GPU loses with the device variant (its 2 x 8 k posted
    // 16-byte writes per step share the PCIe small-request path: targets-only 96 instead of 56 us per step), and with
    // 8 ranks on one host every variant ends at ~250 us per half-step -- that box moves ~90 GB/s between all GPUs and
    // host memory, whoever issues the transfers -- so the host scatter stays the default.
    p->device_expand = h->opts.pipe_expand == 2;
    if (depth == 1) threads = threads > 2 ? 2 : threads;   // a synchronous step only uses the pool for staging copies
    p->pool.reset(new HostPool(threads > 16 ? 16 : threads));
    p->gather_rows = initial_gather_rows(h);
    p->gather_adapt = h->opts.pipe_gather_rows <= 0;   // an explicit TFRPN_PIPE_GATHER_ROWS is kept as given
    cudaError_t e = cudaStreamCreateWithFlags(&p->s_tgt, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_after, cudaEventDisableTiming);
    for (int i = 0; i < depth && e == cudaSuccess; ++i) {
        Slot& s = p->slots[i];
        for (cudaStream_t* st : {&s.s_in, &s.s_prop, &s.s_out})
            if (e == cudaSuccess) e = cudaStreamCreateWithFlags(st, cudaStreamNonBlocking);
        for (cudaEvent_t* ev : {&s.ev_gt, &s.ev_prop, &s.ev_done, &s.ev_rank})
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
        for (int c = 0; c < MAX_CHUNKS && e == cudaSuccess; ++c) {
            e = cudaEventCreateWithFlags(&s.ev_in[c], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.ev_tgt[c], cudaEventDisableTiming);
        }
    }
    p->trace = h->opts.pipe_trace;
    if (p->trace && e == cudaSuccess) {
        e = cudaEventCreate(&p->ev_base);
        if (e == cudaSuccess) e = cudaEventRecord(p->ev_base, p->s_tgt);
        for (int i = 0; i < depth; ++i)
            for (cudaEvent_t& ev : p->slots[i].tr) if (e == cudaSuccess) e = cudaEventCreate(&ev);
    }
    if (e != cudaSuccess) { pipe_destroy(p); return cuda_fail(e, "pipeline_create"); }
    if (depth > 1) {
        // TFRPN_SVC_THREADS=2: one thread gathers while the other enqueues the tail of its step.  Measured at C2: no
        // consistent gain (the worker pool, i.e. host memory latency, is the limit: 570-770 k images/s either way).
        p->n_svc = h->opts.svc_threads >= 2 ? 2 : 1;
        for (int i = 0; i < p->n_svc; ++i) p->svc[i] = std::thread(service_loop, p);
    }
    *out = p;
    return 0;
}

static int redo_flagged_on_host(tfrpn_pipe* p, Slot& s);

// block until the step in `slot` has landed in the caller's buffers
static int slot_finish(tfrpn_pipe* p, Slot& s) {
    if (s.ticket < 0) return 0;
    // the service thread first (it may still have to enqueue the tail of the step, i.e. record ev_done)
    for (int spins = 0; s.svc_pending.load(std::memory_order_acquire) > 0; ++spins) {
        if (spins < 4000) {
#if defined(__x86_64__) || defined(__i386__)
            __builtin_ia32_pause();
#endif
        } else {
            std::this_thread::yield();
        }
    }
    const Step& st = s.step;
    const long long ticket = s.ticket;
    s.ticket = -1;
    if (s.svc_rc != 0) {
        const int rc = s.svc_rc;
        s.svc_rc = 0;
        return fail(rc, "%s", s.svc_err);
    }
    TFRPN_CHECK_CUDA(cudaEventSynchronize(s.ev_done));
    if (p->trace) {
        for (int i = 0; i < 8; ++i)
            if (cudaEventElapsedTime(&s.tr_ms[i], p->ev_base, s.tr[i]) != cudaSuccess) { s.tr_ms[i] = -1.0f; cudaGetLastError(); }
        s.tr_ticket = ticket;
    }
    if (st.two_phase) {
        const int32_t* flags = reinterpret_cast<const int32_t*>(s.pin + st.L.rf);
        int redone = 0;
        for (int b = 0; b < st.B; ++b) redone += flags[b] != 0;
        if (redone && !st.reg_pinned) if (int rc = redo_flagged_on_host(p, s)) return rc;
        if (p->gather_adapt && redone * 16 > st.B && p->gather_rows < proposals_rank_cap())
            p->gather_rows = p->gather_rows + 128 > proposals_rank_cap() ? proposals_rank_cap() : p->gather_rows + 128;
    }
    if (st.compact && !st.device_expand) {   // the retiring thread waits here anyway: it scatters the sparse targets (worker pool)
        const auto t0 = std::chrono::steady_clock::now();
        expand_targets(p, s, s.labels_dst);
        s.expand_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    for (int i = 0; i < s.n_copies; ++i) p->pool->copy(s.copies[i].dst, s.copies[i].src, s.copies[i].bytes);
    s.n_copies = 0;
    p->last_pulled = 0;
    if (s.pulled) {
        p->last_pulled = 16LL * (long long)*reinterpret_cast<const unsigned long long*>(s.pin + st.L.pc);
        s.pulled = false;
    }
    if (st.two_phase) p->last_pulled += 16LL * s.gathered;
    return 0;
}

struct StepArgs {
    const float* anchors_dev;
    // target half (skipped when gt_boxes is null)
    const float* gt_boxes; const int32_t* gt_labels; int B, N, G; const tfrpn_target_cfg* tcfg;
    float* deltas; float* labels;
    // proposal half (skipped when rpn_reg is null)
    const float* rpn_reg; const float* rpn_cls; const tfrpn_proposal_cfg* pcfg;
    float* out_boxes; float* out_scores; int32_t* valid; int32_t* keep_idx;
};

static int slot_reserve(tfrpn_pipe* p, Slot& s, size_t total) {
    if (total <= s.dev_bytes && total <= s.pin_bytes) return 0;
    // growing frees the old buffers: nothing of this pipeline may still be using them
    for (int i = 0; i < p->depth; ++i) if (int rc = slot_finish(p, p->slots[i])) return rc;
    if (int rc = grow_buffer(&s.dev, &s.dev_bytes, total, s.s_out, false)) return rc;
    if (int rc = grow_buffer(&s.pin, &s.pin_bytes, total, s.s_out, true)) return rc;
    s.dense_clean = false;   // new host block: nothing is known about its contents
    return 0;
}

// `acquired`: the caller's buffers are the slot's own pinned block (tfrpn_pipeline_acquire).
static int pipe_submit(tfrpn_pipe* p, const StepArgs& a, bool acquired, bool order_after, cudaStream_t after,
                       long long* ticket_out) {
    const bool do_t = a.gt_boxes != nullptr, do_p = a.rpn_reg != nullptr;
    if (!do_t && !do_p) return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit: neither half given");
    if (!a.anchors_dev) return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit: anchors_dev is null");
    if (a.B <= 0 || a.N <= 0) return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit: bad shape");
    if (do_t && (!a.gt_labels || !a.tcfg || !a.deltas || !a.labels || a.G <= 0))
        return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit: target half needs gt_labels, cfg, deltas, labels and G >= 1");
    if (do_p && (!a.rpn_cls || !a.pcfg || !a.out_boxes || !a.out_scores || !a.valid || a.pcfg->post_nms_topn <= 0))
        return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit: proposal half needs rpn_cls, cfg, out_boxes, out_scores, valid");
    if (do_p && a.pcfg->pre_nms_topn <= 0) return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit: pre_nms_topn must be > 0");
    if (do_p) if (int rc = check_iou_threshold("pipeline_submit", a.pcfg->nms_iou_threshold)) return rc;
    tfrpn_handle h = p->h;
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, a.anchors_dev, "pipeline_submit: anchors_dev");
    const int B = a.B, N = a.N, G = a.G > 0 ? a.G : 1;
    const int P = acquired ? p->acq_P : (do_p ? a.pcfg->post_nms_topn : 1);
    const int GR = p->gather_rows;
    Slot& s = p->slots[p->next_ticket % p->depth];
    if (!acquired) {
        if (int rc = slot_finish(p, s)) return rc;     // slot still busy with ticket - depth: retire it first
        if (int rc = slot_reserve(p, s, make_layout(B, N, G, P).total)) return rc;
    }
    const Layout L = make_layout(B, N, G, P);
    if (do_t) {
        char* ws;
        if (int rc = ensure_workspace(h, targets_workspace_bytes(B, N, G), p->s_tgt, &ws)) return rc;
    }
    char* d = s.dev;
    char* pin = s.pin;
    auto h2d = [&](size_t off, const void* src, size_t bytes) -> int {
        if (!is_pinned(src)) { p->pool->copy(pin + off, src, bytes); src = pin + off; }
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(d + off, src, bytes, cudaMemcpyHostToDevice, s.s_in));
        return 0;
    };
    auto d2h = [&](void* dst, size_t off, size_t bytes) -> int {
        if (is_pinned(dst)) {
            TFRPN_CHECK_CUDA(cudaMemcpyAsync(dst, d + off, bytes, cudaMemcpyDeviceToHost, s.s_out));
        } else {
            TFRPN_CHECK_CUDA(cudaMemcpyAsync(pin + off, d + off, bytes, cudaMemcpyDeviceToHost, s.s_out));
            s.defer(dst, pin + off, bytes);
        }
        return 0;
    };

    if (order_after) {   // everything of this step is ordered after the caller's prior work on `after`
        TFRPN_CHECK_CUDA(cudaEventRecord(p->ev_after, after));
        for (cudaStream_t st : {s.s_in, p->s_tgt, s.s_prop, s.s_out}) TFRPN_CHECK_CUDA(cudaStreamWaitEvent(st, p->ev_after, 0));
    }
    s.n_copies = 0;
    auto mark = [&](int i, cudaStream_t st) { if (p->trace) cudaEventRecord(s.tr[i], st); };
    if (p->trace) for (int i = 0; i < 8; ++i) cudaEventRecord(s.tr[i], s.s_in);   // halves that do not run read as 0-length
    mark(0, s.s_in);
    // bbox_deltas returns in compact form (2.8 MB of results instead of 11.5 MB per C2 step: the deltas are exactly
    // zero outside the <= total_pos sampled positives, utils/train_utils.py:137) and the service thread scatters the
    // rows into the dense host array -- the slot's own (acquired: kept consistent incrementally) or the caller's.
    const bool several = p->depth > 1;   // a depth-1 pipeline is the synchronous step: chunked instead (below)
    const bool compact = several && do_t && !h->opts.pipe_dense && a.tcfg->total_pos <= COMPACT_MAX_POS &&
                         a.tcfg->total_pos + a.tcfg->total_neg <= COMPACT_MAX_Q;
    // The incremental expansion relies on the slot's dense deltas region still holding zeros plus the previous
    // step's rows.  Any step that is not an acquired compact step of the SAME layout may write into that region
    // (dense results, or the inputs / results of another (B,N,G,P) layout): forget the invariant.
    const bool device_expand = compact && acquired && p->device_expand && !p->sparse_labels;
    if (!(compact && acquired && !device_expand && s.pB == B && s.pN == N && s.p_off_d == L.d)) s.dense_clean = false;
    if (!(device_expand && s.dB == B && s.dN == N && s.d_off_d == L.d)) s.dev_clean = false;
    // Two-phase proposals (see the header of this file).  TFRPN_PIPE_DENSE_IN=1 copies the whole rpn_reg tensor.
    const bool two_phase = several && do_p && !h->opts.pipe_dense_in && proposals_two_phase_applies(B, N, a.pcfg);
    // A synchronous step is chunked over images so that copies overlap its own kernels; with several steps in
    // flight the overlap comes from the neighbouring steps and fewer, larger copies win.
    int chunks = !several ? (B >= 32 ? 4 : (B >= 8 ? 2 : 1)) : 1;
    if (h->opts.pipe_chunks > 0 && !several) chunks = h->opts.pipe_chunks;
    chunks = chunks < 1 ? 1 : (chunks > MAX_CHUNKS ? MAX_CHUNKS : chunks);

    Step& st = s.step;
    st = Step();
    st.do_t = do_t; st.do_p = do_p; st.acquired = acquired; st.compact = compact; st.two_phase = two_phase;
    st.B = B; st.N = N; st.G = G; st.P = P; st.GR = GR; st.total_pos = do_t ? a.tcfg->total_pos : 0;
    st.device_expand = device_expand;
    st.sparse_labels = compact && p->sparse_labels;
    st.Q = st.sparse_labels ? a.tcfg->total_pos + a.tcfg->total_neg : 0;
    st.L = L; st.anchors = a.anchors_dev;
    st.cl = L.comp;                                              // packed with this step's quotas: one D2H range
    st.ci = st.cl + (((size_t)B * st.Q * 4 + 15) & ~(size_t)15);
    st.cd = st.ci + (((size_t)B * st.total_pos * 4 + 15) & ~(size_t)15);
    s.labels_dst = acquired ? reinterpret_cast<float*>(pin + L.l) : a.labels;
    if (do_p) st.pcfg = *a.pcfg;
    st.reg_host = a.rpn_reg;
    // a caller's dense buffer (page-locked or not: the rows are written by host threads) is zeroed and filled in place
    st.dense_dst = acquired ? reinterpret_cast<float*>(pin + L.d) : a.deltas;
    if (two_phase) {
        cudaPointerAttributes attr;
        st.reg_pinned = cudaPointerGetAttributes(&attr, a.rpn_reg) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
                        attr.devicePointer != nullptr;
        cudaGetLastError();
        st.reg_dev = st.reg_pinned ? static_cast<const float*>(attr.devicePointer) : nullptr;
    }
    // who gathers: host threads when the pool has enough of them (lower latency, one bulk copy), else the device
    st.device_gather = two_phase && st.reg_pinned && p->device_gather;
    s.pulled = two_phase && st.reg_pinned;
    s.gathered = 0;
    s.gather_ms = s.expand_ms = 0.f;
    s.svc_rc = 0;
    s.svc_pending.store(two_phase && !st.device_gather ? 1 : 0, std::memory_order_release);

    p->last_h2d = p->last_d2h = 0;
    if (acquired) {
        // one copy for all (copied) inputs of the halves that run
        const size_t lo = do_t ? L.gt : L.cls, hi = do_p ? (two_phase ? L.small_end : L.in_end) : L.cls;
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(d + lo, pin + lo, hi - lo, cudaMemcpyHostToDevice, s.s_in));
        p->last_h2d = (long long)(hi - lo);
    } else {
        if (do_t) {
            if (int rc = h2d(L.gt, a.gt_boxes, (size_t)B * G * 16)) return rc;
            if (int rc = h2d(L.gl, a.gt_labels, (size_t)B * G * 4)) return rc;
            p->last_h2d += (long long)B * G * 20;
        }
        if (two_phase) {
            if (int rc = h2d(L.cls, a.rpn_cls, (size_t)B * N * 4)) return rc;
            p->last_h2d += (long long)B * N * 4;
        }
    }
    mark(1, s.s_in);
    TFRPN_CHECK_CUDA(cudaEventRecord(s.ev_gt, s.s_in));
    if (do_t) TFRPN_CHECK_CUDA(cudaStreamWaitEvent(p->s_tgt, s.ev_gt, 0));
    if (do_p) TFRPN_CHECK_CUDA(cudaStreamWaitEvent(s.s_prop, s.ev_gt, 0));
    if (do_t) mark(2, p->s_tgt);
    if (do_p) mark(4, s.s_prop);
    if (two_phase) {   // ranks from the scores, and their indices back to the host; the service thread takes over from there
        if (int rc = proposals_rank_enqueue(h, reinterpret_cast<const float*>(d + L.cls), B, N, a.pcfg,
                                            reinterpret_cast<int32_t*>(d + L.ri), reinterpret_cast<int32_t*>(d + L.rn),
                                            reinterpret_cast<int32_t*>(d + L.rm), s.s_prop)) return rc;
        if (st.reg_pinned) TFRPN_CHECK_CUDA(cudaMemsetAsync(d + L.pc, 0, 8, s.s_prop));   // rows the device pulls itself
        if (!st.device_gather) {
            TFRPN_CHECK_CUDA(cudaMemcpyAsync(pin + L.ri, d + L.ri, L.rank_end - L.ri, cudaMemcpyDeviceToHost, s.s_prop));
            TFRPN_CHECK_CUDA(cudaEventRecord(s.ev_rank, s.s_prop));
            p->last_h2d += (long long)B * GR * 16;
            p->last_d2h += (long long)(L.rank_end - L.ri);
        }
    }
    for (int c = 0; c < chunks; ++c) {
        const int lo = (int)((long long)B * c / chunks), hi = (int)((long long)B * (c + 1) / chunks), nb = hi - lo;
        if (nb == 0) continue;
        if (do_p && !two_phase) {
            if (!acquired) {
                if (int rc = h2d(L.reg + (size_t)lo * N * 16, a.rpn_reg + (size_t)lo * N * 4, (size_t)nb * N * 16)) return rc;
                if (int rc = h2d(L.cls + (size_t)lo * N * 4, a.rpn_cls + (size_t)lo * N, (size_t)nb * N * 4)) return rc;
                p->last_h2d += (long long)nb * N * 20;
                TFRPN_CHECK_CUDA(cudaEventRecord(s.ev_in[c], s.s_in));
                TFRPN_CHECK_CUDA(cudaStreamWaitEvent(s.s_prop, s.ev_in[c], 0));
            }
            if (int rc = proposals_enqueue(h, reinterpret_cast<const float*>(d + L.reg) + (size_t)lo * N * 4,
                                           reinterpret_cast<const float*>(d + L.cls) + (size_t)lo * N, a.anchors_dev, nb, N,
                                           a.pcfg, reinterpret_cast<float*>(d + L.ob) + (size_t)lo * P * 4,
                                           reinterpret_cast<float*>(d + L.os) + (size_t)lo * P,
                                           reinterpret_cast<int32_t*>(d + L.v) + lo,
                                           reinterpret_cast<int32_t*>(d + L.k) + (size_t)lo * P, nullptr, s.s_prop)) return rc;
        }
        if (do_t) {
            tfrpn_target_cfg cc = *a.tcfg;
            cc.image_offset = a.tcfg->image_offset + lo;
            if (compact) {   // (compact => one chunk)
                if (int rc = launch_targets(h, a.anchors_dev, reinterpret_cast<const float*>(d + L.gt),
                                            reinterpret_cast<const int32_t*>(d + L.gl), nb, N, G, &cc, nullptr,
                                            st.sparse_labels ? nullptr : reinterpret_cast<float*>(d + L.l),
                                            reinterpret_cast<int32_t*>(d + st.ci), reinterpret_cast<float*>(d + st.cd),
                                            st.sparse_labels ? reinterpret_cast<int32_t*>(d + st.cl) : nullptr, nullptr,
                                            p->s_tgt)) return rc;
                if (device_expand) {
                    float* dense = reinterpret_cast<float*>(pin + L.d);   // (UVA: a cudaHostAlloc pointer is its own device alias)
                    int32_t* pci = reinterpret_cast<int32_t*>(d + L.pci);
                    if (!s.dev_clean) {   // first use of this layout: the whole array is zeroed once, over PCIe
                        TFRPN_CHECK_CUDA(cudaMemsetAsync(dense, 0, (size_t)B * N * 16, p->s_tgt));
                        TFRPN_CHECK_CUDA(cudaMemsetAsync(pci, 0xFF, (size_t)B * COMPACT_MAX_POS * 4, p->s_tgt));
                    }
                    if (int rc = scatter_rows_to_host_enqueue(pci, COMPACT_MAX_POS, reinterpret_cast<int32_t*>(d + st.ci),
                                                              reinterpret_cast<float*>(d + st.cd), a.tcfg->total_pos, B, N, dense,
                                                              COMPACT_MAX_POS, p->s_tgt)) return rc;
                    s.dev_clean = true; s.dB = B; s.dN = N; s.d_off_d = L.d;
                }
            } else if (int rc = tfrpn_rpn_targets(h, a.anchors_dev, reinterpret_cast<const float*>(d + L.gt) + (size_t)lo * G * 4,
                                           reinterpret_cast<const int32_t*>(d + L.gl) + (size_t)lo * G, nb, N, G, &cc,
                                           reinterpret_cast<float*>(d + L.d) + (size_t)lo * N * 4,
                                           reinterpret_cast<float*>(d + L.l) + (size_t)lo * N, nullptr, p->s_tgt)) return rc;
            mark(3, p->s_tgt);
            TFRPN_CHECK_CUDA(cudaEventRecord(s.ev_tgt[c], p->s_tgt));
            TFRPN_CHECK_CUDA(cudaStreamWaitEvent(s.s_out, s.ev_tgt[c], 0));
            if (!acquired && !compact) {
                if (int rc = d2h(a.deltas + (size_t)lo * N * 4, L.d + (size_t)lo * N * 16, (size_t)nb * N * 16)) return rc;
                if (int rc = d2h(a.labels + (size_t)lo * N, L.l + (size_t)lo * N * 4, (size_t)nb * N * 4)) return rc;
                p->last_d2h += (long long)nb * N * 20;
            }
        }
    }
    // bytes of the result copy enqueue_tail makes
    if (compact && !acquired && !st.sparse_labels) s.defer(a.labels, pin + L.l, (size_t)B * N * 4);
    if (compact) p->last_d2h += (long long)((device_expand ? L.dense_end + (size_t)2 * B * a.tcfg->total_pos * 16 : st.cd + (size_t)B * a.tcfg->total_pos * 16) -
                                            (!st.sparse_labels ? L.l : (do_p ? L.ob : L.rf)));   // (device expansion: + the rows written over PCIe)
    else if (acquired) p->last_d2h += (long long)((do_p ? L.dense_end : L.ob) - (do_t ? L.d : L.ob));
    else if (do_p) p->last_d2h += (long long)(L.dense_end - L.ob);
    if (!acquired) {   // results that land in the slot's pinned block are copied out when the step is retired
        if (do_p) {
            s.defer(a.out_boxes, pin + L.ob, (size_t)B * P * 16);
            s.defer(a.out_scores, pin + L.os, (size_t)B * P * 4);
            s.defer(a.valid, pin + L.v, (size_t)B * 4);
            if (a.keep_idx) s.defer(a.keep_idx, pin + L.k, (size_t)B * P * 4);
        }
    }
    s.ticket = p->next_ticket++;
    if (ticket_out) *ticket_out = s.ticket;
    if (two_phase && !st.device_gather) svc_push(p, STAGE_GATHER, &s);   // ... which ends by calling enqueue_tail
    else if (int rc = enqueue_tail(p, s)) return rc;
    return 0;
}

// Two-phase step whose rpn_reg is pageable (the device cannot read it): images that raised their redo flag get
// their whole reg rows copied now and the unfiltered kernel run for them, synchronously.  Rare by construction
// (NMS needed more than the gathered rows of an image).
static int redo_flagged_on_host(tfrpn_pipe* p, Slot& s) {
    const Step& st = s.step;
    const Layout& L = st.L;
    const int32_t* flags = reinterpret_cast<const int32_t*>(s.pin + L.rf);
    bool any = false;
    for (int b = 0; b < st.B; ++b) any = any || flags[b] != 0;
    if (!any) return 0;
    tfrpn_handle h = p->h;
    char* d = s.dev;
    char* pin = s.pin;
    for (int b = 0; b < st.B; ++b) {
        if (!flags[b]) continue;
        const size_t off = L.reg + (size_t)b * st.N * 16;
        memcpy(pin + off, st.reg_host + (size_t)b * st.N * 4, (size_t)st.N * 16);
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(d + off, pin + off, (size_t)st.N * 16, cudaMemcpyHostToDevice, s.s_prop));
    }
    if (int rc = proposals_redo_enqueue(h, reinterpret_cast<const float*>(d + L.reg), reinterpret_cast<const float*>(d + L.cls),
                                        st.anchors, st.B, st.N, &st.pcfg, reinterpret_cast<float*>(d + L.ob),
                                        reinterpret_cast<float*>(d + L.os), reinterpret_cast<int32_t*>(d + L.v),
                                        reinterpret_cast<int32_t*>(d + L.k), reinterpret_cast<const int32_t*>(d + L.rf),
                                        nullptr, s.s_prop)) return rc;
    TFRPN_CHECK_CUDA(cudaMemcpyAsync(pin + L.ob, d + L.ob, L.dense_end - L.ob, cudaMemcpyDeviceToHost, s.s_prop));
    TFRPN_CHECK_CUDA(cudaStreamSynchronize(s.s_prop));
    return 0;
}

static int pipe_wait(tfrpn_pipe* p, long long ticket) {
    if (ticket < 0 || ticket >= p->next_ticket) return fail(TFRPN_ERR_BAD_ARG, "pipeline_wait: unknown ticket %lld", ticket);
    Slot& s = p->slots[ticket % p->depth];
    if (s.ticket != ticket) return 0;     // already retired (waited for, or its slot was reused)
    return slot_finish(p, s);
}

}  // namespace tfrpn

using namespace tfrpn;

extern "C" int tfrpn_pipeline_create(tfrpn_handle h, int depth, tfrpn_pipeline* out) { return pipe_create(h, depth, out); }

extern "C" int tfrpn_pipeline_destroy(tfrpn_pipeline p) {
    pipe_destroy(p);
    return 0;
}

extern "C" int tfrpn_pipeline_submit(tfrpn_pipeline p, const float* anchors_dev, int B, int N,
                                     const float* gt_boxes_host, const int32_t* gt_labels_host, int G,
                                     const tfrpn_target_cfg* tcfg, float* deltas_host, float* labels_host,
                                     const float* rpn_reg_host, const float* rpn_cls_host, const tfrpn_proposal_cfg* pcfg,
                                     float* out_boxes_host, float* out_scores_host, int32_t* valid_host,
                                     int32_t* keep_idx_host_or_null, int64_t* ticket_out) {
    if (!p) return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit: null pipeline");
    StepArgs a = {anchors_dev, gt_boxes_host, gt_labels_host, B, N, G, tcfg, deltas_host, labels_host,
                  rpn_reg_host, rpn_cls_host, pcfg, out_boxes_host, out_scores_host, valid_host, keep_idx_host_or_null};
    long long t = -1;
    if (p->acq_live) return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit: a slot is acquired; submit it with tfrpn_pipeline_submit_acquired first");
    if (int rc = pipe_submit(p, a, false, false, nullptr, &t)) return rc;
    if (ticket_out) *ticket_out = t;
    return 0;
}

extern "C" int tfrpn_pipeline_acquire(tfrpn_pipeline p, int B, int N, int G, int post_nms_topn, tfrpn_step_buffers* out) {
    if (!p || !out) return fail(TFRPN_ERR_BAD_ARG, "pipeline_acquire: null pointer");
    if (B <= 0 || N <= 0 || G <= 0 || post_nms_topn <= 0) return fail(TFRPN_ERR_BAD_ARG, "pipeline_acquire: bad shape");
    TFRPN_ENTER(p->h);
    Slot& s = p->slots[p->next_ticket % p->depth];
    if (int rc = slot_finish(p, s)) return rc;
    const Layout L = make_layout(B, N, G, post_nms_topn);
    if (int rc = slot_reserve(p, s, L.total)) return rc;
    p->acq_B = B; p->acq_N = N; p->acq_G = G; p->acq_P = post_nms_topn; p->acq_live = true;
    char* pin = s.pin;
    out->gt_boxes = reinterpret_cast<float*>(pin + L.gt);
    out->gt_labels = reinterpret_cast<int32_t*>(pin + L.gl);
    out->rpn_reg = reinterpret_cast<float*>(pin + L.reg);
    out->rpn_cls = reinterpret_cast<float*>(pin + L.cls);
    out->deltas = reinterpret_cast<float*>(pin + L.d);
    out->labels = reinterpret_cast<float*>(pin + L.l);
    out->out_boxes = reinterpret_cast<float*>(pin + L.ob);
    out->out_scores = reinterpret_cast<float*>(pin + L.os);
    out->valid = reinterpret_cast<int32_t*>(pin + L.v);
    out->keep_idx = reinterpret_cast<int32_t*>(pin + L.k);
    return 0;
}

extern "C" int tfrpn_pipeline_submit_acquired(tfrpn_pipeline p, const float* anchors_dev, const tfrpn_target_cfg* tcfg_or_null,
                                              const tfrpn_proposal_cfg* pcfg_or_null, int64_t* ticket_out) {
    if (!p) return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit_acquired: null pipeline");
    if (!p->acq_live) return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit_acquired: no slot acquired");
    if (pcfg_or_null && pcfg_or_null->post_nms_topn != p->acq_P)
        return fail(TFRPN_ERR_BAD_ARG, "pipeline_submit_acquired: post_nms_topn %d differs from the acquired %d",
                    pcfg_or_null->post_nms_topn, p->acq_P);
    Slot& s = p->slots[p->next_ticket % p->depth];
    const Layout L = make_layout(p->acq_B, p->acq_N, p->acq_G, p->acq_P);
    char* pin = s.pin;
    StepArgs a = {};
    a.anchors_dev = anchors_dev; a.B = p->acq_B; a.N = p->acq_N; a.G = p->acq_G;
    if (tcfg_or_null) {
        a.gt_boxes = reinterpret_cast<float*>(pin + L.gt); a.gt_labels = reinterpret_cast<int32_t*>(pin + L.gl);
        a.tcfg = tcfg_or_null; a.deltas = reinterpret_cast<float*>(pin + L.d); a.labels = reinterpret_cast<float*>(pin + L.l);
    }
    if (pcfg_or_null) {
        a.rpn_reg = reinterpret_cast<float*>(pin + L.reg); a.rpn_cls = reinterpret_cast<float*>(pin + L.cls);
        a.pcfg = pcfg_or_null; a.out_boxes = reinterpret_cast<float*>(pin + L.ob);
        a.out_scores = reinterpret_cast<float*>(pin + L.os); a.valid = reinterpret_cast<int32_t*>(pin + L.v);
        a.keep_idx = reinterpret_cast<int32_t*>(pin + L.k);
    }
    long long t = -1;
    if (int rc = pipe_submit(p, a, true, false, nullptr, &t)) return rc;
    p->acq_live = false;
    if (ticket_out) *ticket_out = t;
    return 0;
}

extern "C" int tfrpn_pipeline_last_copy_bytes(tfrpn_pipeline p, int64_t* h2d_bytes, int64_t* d2h_bytes) {
    if (!p || !h2d_bytes || !d2h_bytes) return fail(TFRPN_ERR_BAD_ARG, "pipeline_last_copy_bytes: null pointer");
    *h2d_bytes = p->last_h2d + p->last_pulled;   // copy + the 16-byte rows the kernels loaded from the pinned block
    *d2h_bytes = p->last_d2h;
    return 0;
}

extern "C" int tfrpn_pipeline_trace(tfrpn_pipeline p, int64_t ticket, float* ms10) {
    float* ms8 = ms10;
    if (!p || !ms8) return fail(TFRPN_ERR_BAD_ARG, "pipeline_trace: null pointer");
    if (!p->trace) return fail(TFRPN_ERR_UNSUPPORTED, "pipeline_trace: the handle was created without TFRPN_PIPE_TRACE=1");
    const Slot& s = p->slots[(ticket < 0 ? 0 : ticket) % p->depth];
    if (s.tr_ticket != ticket) return fail(TFRPN_ERR_BAD_ARG, "pipeline_trace: step %lld is not the last one retired from its slot", (long long)ticket);
    for (int i = 0; i < 8; ++i) ms8[i] = s.tr_ms[i];
    ms10[8] = s.gather_ms;
    ms10[9] = s.expand_ms;
    return 0;
}

extern "C" int tfrpn_pipeline_set_option(tfrpn_pipeline p, int option, int value) {
    if (!p) return fail(TFRPN_ERR_BAD_ARG, "pipeline_set_option: null pipeline");
    if (option == TFRPN_PIPE_OPT_STABLE_OUTPUTS) {
        TFRPN_ENTER(p->h);
        for (int i = 0; i < p->depth; ++i) if (int rc = slot_finish(p, p->slots[i])) return rc;   // nothing in flight while it changes
        p->stable_outputs = value != 0;
        if (!p->stable_outputs) p->caller_dense.clear();
        return 0;
    }
    return fail(TFRPN_ERR_BAD_ARG, "pipeline_set_option: unknown option %d", option);
}

extern "C" int tfrpn_pipeline_wait(tfrpn_pipeline p, int64_t ticket) {
    if (!p) return fail(TFRPN_ERR_BAD_ARG, "pipeline_wait: null pipeline");
    TFRPN_ENTER(p->h);
    return pipe_wait(p, ticket);
}

extern "C" int tfrpn_pipeline_drain(tfrpn_pipeline p) {
    if (!p) return fail(TFRPN_ERR_BAD_ARG, "pipeline_drain: null pipeline");
    TFRPN_ENTER(p->h);
    for (int i = 0; i < p->depth; ++i) if (int rc = slot_finish(p, p->slots[i])) return rc;
    return 0;
}

// One step from host buffers, synchronous: submit + wait on a depth-1 pipeline owned by the handle.
extern "C" int tfrpn_rpn_step_host(tfrpn_handle h, const float* anchors_dev, const float* gt_boxes_host,
                                   const int32_t* gt_labels_host, int B, int N, int G,
                                   const tfrpn_target_cfg* tcfg, float* deltas_host, float* labels_host,
                                   const float* rpn_reg_host, const float* rpn_cls_host,
                                   const tfrpn_proposal_cfg* pcfg, float* out_boxes_host, float* out_scores_host,
                                   int32_t* valid_host, int32_t* keep_idx_host_or_null, tfrpn_stream s) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "rpn_step_host: null handle");
    if (!gt_boxes_host || !gt_labels_host || !deltas_host || !labels_host || !tcfg || !rpn_reg_host || !rpn_cls_host ||
        !pcfg || !out_boxes_host || !out_scores_host || !valid_host)
        return fail(TFRPN_ERR_BAD_ARG, "rpn_step_host: null pointer");
    if (B <= 0 || N <= 0 || G <= 0 || pcfg->post_nms_topn <= 0) return fail(TFRPN_ERR_BAD_ARG, "rpn_step_host: bad shape");
    TFRPN_ENTER(h);
    if (!h->step_pipe) if (int rc = pipe_create(h, 1, &h->step_pipe)) return rc;
    StepArgs a = {anchors_dev, gt_boxes_host, gt_labels_host, B, N, G, tcfg, deltas_host, labels_host,
                  rpn_reg_host, rpn_cls_host, pcfg, out_boxes_host, out_scores_host, valid_host, keep_idx_host_or_null};
    long long t = -1;
    if (int rc = pipe_submit(h->step_pipe, a, false, true, as_stream(s), &t)) return rc;
    return pipe_wait(h->step_pipe, t);
}
