// api.cu -- handle, error reporting, workspace, and the host-buffer entry points of libtfrpn_cuda.so.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "common.cuh"

namespace tfrpn {

static thread_local char g_err[512] = "";
static thread_local uint64_t g_launches = 0;

int fail(int status, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return status;
}

int cuda_fail(cudaError_t e, const char* what) {
    return fail(TFRPN_ERR_CUDA, "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
}

void count_launch() { ++g_launches; }

size_t targets_workspace_bytes(int B, int N, int G);  // targets.cu
size_t prefilter_workspace_bytes(int B, int N, int k);  // proposals.cu (0 when the prefilter does not apply)

int sm_count_of(tfrpn_handle h) { return h ? h->sm_count : 148; }

int device_of_pointer(const void* p) {
    if (!p) return -1;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return -1; }
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) return -1;
    return attr.device;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE property of a kernel: set it once for every
// device a call touches (not once per thread), with that device current.
int ensure_kernel_attributes(int device) {
    constexpr int MAX_DEV = 64;
    static bool done[MAX_DEV] = {};
    static std::mutex mu;
    if (device < 0 || device >= MAX_DEV) return fail(TFRPN_ERR_BAD_ARG, "device %d out of range", device);
    std::lock_guard<std::mutex> lock(mu);
    if (done[device]) return 0;
    if (int rc = set_attributes_targets()) return rc;
    if (int rc = set_attributes_proposals()) return rc;
    if (int rc = set_attributes_boxmath()) return rc;
    if (int rc = set_attributes_evaluate()) return rc;
    done[device] = true;
    return 0;
}

static int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return (e && *e) ? atoi(e) : dflt;   // (an empty value means "not set")
}

int grow_buffer(char** buf, size_t* have, size_t want, cudaStream_t s, bool pinned) {
    if (want <= *have) return 0;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone)
        return fail(TFRPN_ERR_WORKSPACE, "workspace must grow to %zu B while the stream is capturing; call tfrpn_reserve first", want);
    if (*buf) {
        TFRPN_CHECK_CUDA(cudaStreamSynchronize(s));
        TFRPN_CHECK_CUDA(cudaDeviceSynchronize());
        if (pinned) TFRPN_CHECK_CUDA(cudaFreeHost(*buf)); else TFRPN_CHECK_CUDA(cudaFree(*buf));
        *buf = nullptr;
        *have = 0;
    }
    want = (want + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
    void* p = nullptr;
    if (pinned) TFRPN_CHECK_CUDA(cudaHostAlloc(&p, want, cudaHostAllocDefault)); else TFRPN_CHECK_CUDA(cudaMalloc(&p, want));
    *buf = static_cast<char*>(p);
    *have = want;
    return 0;
}

int ensure_workspace(tfrpn_handle h, size_t bytes, cudaStream_t s, char** out) {
    if (int rc = grow_buffer(&h->ws, &h->ws_bytes, bytes, s, false)) return rc;
    *out = h->ws;
    return 0;
}

int ensure_workspace_prop(tfrpn_handle h, size_t bytes, cudaStream_t s, char** out) {
    if (int rc = grow_buffer(&h->ws_prop, &h->ws_prop_bytes, bytes, s, false)) return rc;
    *out = h->ws_prop;
    return 0;
}

void prof_begin(tfrpn_handle h, int kernel_id, cudaStream_t s) {
    if (!h || !h->prof_on) return;
    tfrpn_ctx::Rec r;
    r.id = kernel_id;
    cudaEventCreate(&r.a);
    cudaEventCreate(&r.b);
    cudaEventRecord(r.a, s);
    h->recs.push_back(r);
}
void prof_end(tfrpn_handle h, cudaStream_t s) {
    if (!h || !h->prof_on || h->recs.empty()) return;
    cudaEventRecord(h->recs.back().b, s);
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace tfrpn

using namespace tfrpn;

extern "C" int tfrpn_version(void) { return TFRPN_VERSION; }
extern "C" const char* tfrpn_last_error(void) { return g_err; }
extern "C" uint64_t tfrpn_launch_count(void) { return g_launches; }

extern "C" int tfrpn_profile_enable(tfrpn_handle h, int on) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "profile_enable: null handle");
    TFRPN_ENTER(h);
    h->prof_on = on != 0;
    return 0;
}

extern "C" int tfrpn_profile_read(tfrpn_handle h, int kernel_id, double* total_ms, int* launches) {
    if (!h || !total_ms || !launches) return fail(TFRPN_ERR_BAD_ARG, "profile_read: null pointer");
    TFRPN_ENTER(h);
    TFRPN_CHECK_CUDA(cudaDeviceSynchronize());
    double ms = 0;
    int n = 0;
    std::vector<tfrpn_ctx::Rec> rest;
    for (auto& r : h->recs) {
        if (r.id != kernel_id) { rest.push_back(r); continue; }
        float t = 0.f;
        if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { ms += t; ++n; }
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    cudaGetLastError();
    h->recs.swap(rest);
    *total_ms = ms;
    *launches = n;
    return 0;
}

extern "C" const char* tfrpn_kernel_name(int id) {
    switch (id) {
        case TFRPN_K_IOU_ARGMAX: return "rpn_iou_argmax_kernel";
        case TFRPN_K_LABEL_ENCODE: return "rpn_label_encode_kernel";
        case TFRPN_K_SELECT_MASK: return "select_mask_kernel";
        case TFRPN_K_PROPOSAL: return "proposal_kernel";
        case TFRPN_K_PROPOSAL_CLUSTER: return "proposal_cluster_kernel";
        case TFRPN_K_NMS_MASK: return "nms_mask_kernel";
        case TFRPN_K_NMS_SWEEP: return "nms_sweep_kernel";
        case TFRPN_K_LOSS: return "rpn_loss_partial_kernel";
        case TFRPN_K_RECALL: return "recall_kernel";
        case TFRPN_K_NMS_MC_STAGE: return "nms_mc_stage_kernel";
        case TFRPN_K_NMS_MC_MERGE: return "nms_mc_merge_kernel";
        case TFRPN_K_MAP_MATCH: return "map_match_kernel";
        case TFRPN_K_MAP_AP: return "map_ap_kernel";
        default: return "?";
    }
}

extern "C" int tfrpn_create(tfrpn_handle* out, int device) {
    if (!out) return fail(TFRPN_ERR_BAD_ARG, "create: out is null");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(TFRPN_ERR_CUDA, "no CUDA device available (%s); libtfrpn_cuda has no CPU fallback",
                    e == cudaSuccess ? "0 devices" : cudaGetErrorString(e));
    if (device < 0) TFRPN_CHECK_CUDA(cudaGetDevice(&device));
    if (device >= count) return fail(TFRPN_ERR_BAD_ARG, "create: device %d of %d", device, count);
    DeviceGuard guard(device);   // the caller's current device is restored on return
    if (guard.err != cudaSuccess) return cuda_fail(guard.err, "cudaSetDevice");
    if (int rc = ensure_kernel_attributes(device)) return rc;
    tfrpn_ctx* h = new tfrpn_ctx();
    h->device = device;
    // A/B switches: read here, once per handle, never on the launch path
    h->opts.k2_apt = env_int("TFRPN_K2_APT", 0);
    h->opts.k2_scalar = getenv("TFRPN_K2_SCALAR") != nullptr;
    h->opts.pipe_dense = getenv("TFRPN_PIPE_DENSE") != nullptr;
    h->opts.pipe_chunks = env_int("TFRPN_PIPE_CHUNKS", 0);
    h->opts.prop_cluster = env_int("TFRPN_PROP_CLUSTER", -1);
    h->opts.prop_threads = env_int("TFRPN_PROP_THREADS", 0);
    h->opts.pipe_dense_in = getenv("TFRPN_PIPE_DENSE_IN") != nullptr;
    h->opts.pipe_trace = getenv("TFRPN_PIPE_TRACE") != nullptr;
    h->opts.pipe_gather_rows = env_int("TFRPN_PIPE_GATHER_ROWS", 0);
    h->opts.host_threads = env_int("TFRPN_HOST_THREADS", 0);
    h->opts.svc_threads = env_int("TFRPN_SVC_THREADS", 0);
    h->opts.pipe_sparse_labels = env_int("TFRPN_PIPE_SPARSE_LABELS", -1);
    if (const char* g = getenv("TFRPN_PIPE_EXPAND")) h->opts.pipe_expand = !strcmp(g, "host") ? 1 : (!strcmp(g, "device") ? 2 : 0);
    if (const char* g = getenv("TFRPN_NMS_PATH")) h->opts.nms_lazy = strcmp(g, "matrix") != 0;
    h->opts.nms_rows = env_int("TFRPN_NMS_ROWS", 0);
    if (const char* g = getenv("TFRPN_NMS_MC_STAGE")) h->opts.nms_mc_stage = !strcmp(g, "column") ? 1 : (!strcmp(g, "rows") ? 2 : 0);
    if (const char* g = getenv("TFRPN_PIPE_GATHER")) h->opts.pipe_gather = !strcmp(g, "host") ? 1 : (!strcmp(g, "device") ? 2 : 0);
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    // device counter of the loss reduction (losses.cu): zero between calls, the kernel resets it
    if (cudaMalloc(&h->ticket, 256) != cudaSuccess || cudaMemset(h->ticket, 0, 256) != cudaSuccess) {
        cudaError_t e2 = cudaGetLastError();
        delete h;
        return cuda_fail(e2, "create: device counter");
    }
    *out = h;
    return 0;
}

extern "C" int tfrpn_destroy(tfrpn_handle h) {
    if (!h) return 0;
    DeviceGuard guard(h->device);
    if (h->ws) cudaFree(h->ws);
    if (h->ws_prop) cudaFree(h->ws_prop);
    if (h->dev) cudaFree(h->dev);
    if (h->pinned) cudaFreeHost(h->pinned);
    if (h->dev2) cudaFree(h->dev2);
    if (h->pinned2) cudaFreeHost(h->pinned2);
    if (h->step_pipe) pipe_destroy(h->step_pipe);
    if (h->ticket) cudaFree(h->ticket);
    if (h->anchor_gen) cudaFree(h->anchor_gen);
    delete h;
    return 0;
}

extern "C" size_t tfrpn_workspace_bytes(int B, int N, int G, int k) {
    // targets scratch + the candidate arrays of the large-N top-k prefilter (small N: top-k / NMS work
    // entirely in shared memory)
    if (B <= 0 || N <= 0) return 0;
    return targets_workspace_bytes(B, N, G > 0 ? G : 1) + prefilter_workspace_bytes(B, N, k);
}

extern "C" int tfrpn_reserve(tfrpn_handle h, int B, int N, int G, int k) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "reserve: null handle");
    TFRPN_ENTER(h);
    char* ws;
    if (B <= 0 || N <= 0) return 0;
    if (int rc = ensure_workspace(h, targets_workspace_bytes(B, N, G > 0 ? G : 1), nullptr, &ws)) return rc;
    const size_t pb = prefilter_workspace_bytes(B, N, k);
    return pb ? ensure_workspace_prop(h, pb, nullptr, &ws) : 0;
}

extern "C" int tfrpn_host_alloc(void** out, size_t bytes) {
    if (!out) return fail(TFRPN_ERR_BAD_ARG, "host_alloc: out is null");
    TFRPN_CHECK_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return 0;
}
extern "C" int tfrpn_host_free(void* p) {
    if (p) TFRPN_CHECK_CUDA(cudaFreeHost(p));
    return 0;
}

// ---- host-buffer entry points ---------------------------------------------------------------------
// Each half has its own device + pinned staging region so that the fused step can run both at once.
struct Staging {
    char** dev; size_t* dev_bytes; char** pin; size_t* pin_bytes;
};
struct HostJob {   // copies out of pinned staging, to run after the stream has been synchronised
    struct Copy { void* dst; const void* src; size_t bytes; } copies[24];
    int n = 0;
    void add(void* d, const void* s, size_t b) { copies[n].dst = d; copies[n].src = s; copies[n].bytes = b; ++n; }
    void finish() { for (int i = 0; i < n; ++i) memcpy(copies[i].dst, copies[i].src, copies[i].bytes); n = 0; }
};

static bool is_pinned(const void* p) {
    cudaPointerAttributes attr;
    bool r = cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    return r;
}

// copy from a caller's host buffer: directly when it is page-locked, else through pinned staging
static int h2d(void* dst, const void* src, size_t bytes, char* pin_slot, cudaStream_t s) {
    if (!is_pinned(src)) {
        memcpy(pin_slot, src, bytes);
        src = pin_slot;
    }
    TFRPN_CHECK_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s));
    return 0;
}
// copy to a caller's host buffer: directly when it is page-locked, else staging + deferred memcpy
static int d2h(void* dst, const void* src_dev, size_t bytes, char* pin_slot, cudaStream_t s, HostJob& job) {
    if (is_pinned(dst)) {
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(dst, src_dev, bytes, cudaMemcpyDeviceToHost, s));
    } else {
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(pin_slot, src_dev, bytes, cudaMemcpyDeviceToHost, s));
        job.add(dst, pin_slot, bytes);
    }
    return 0;
}

static int targets_host_enqueue(tfrpn_handle h, const float* anchors_dev, const float* gt_boxes_host,
                                const int32_t* gt_labels_host, int B, int N, int G, const tfrpn_target_cfg* cfg,
                                float* deltas_host, float* labels_host, cudaStream_t st, HostJob& job) {
    if (!gt_boxes_host || !gt_labels_host || !deltas_host || !labels_host)
        return fail(TFRPN_ERR_BAD_ARG, "rpn_targets_host: null pointer");
    if (B <= 0 || N <= 0 || G <= 0) return fail(TFRPN_ERR_BAD_ARG, "rpn_targets_host: bad shape");
    const size_t b_gt = align256((size_t)B * G * 16), b_gl = align256((size_t)B * G * 4);
    const size_t b_d = align256((size_t)B * N * 16), b_l = align256((size_t)B * N * 4);
    if (int rc = grow_buffer(&h->dev, &h->dev_bytes, b_gt + b_gl + b_d + b_l, st, false)) return rc;
    if (int rc = grow_buffer(&h->pinned, &h->pinned_bytes, b_gt + b_gl + b_d + b_l, st, true)) return rc;
    char* d = h->dev;
    char* pin = h->pinned;
    float* d_gt = reinterpret_cast<float*>(d);
    int32_t* d_gl = reinterpret_cast<int32_t*>(d + b_gt);
    float* d_d = reinterpret_cast<float*>(d + b_gt + b_gl);
    float* d_l = reinterpret_cast<float*>(d + b_gt + b_gl + b_d);
    if (int rc = h2d(d_gt, gt_boxes_host, (size_t)B * G * 16, pin, st)) return rc;
    if (int rc = h2d(d_gl, gt_labels_host, (size_t)B * G * 4, pin + b_gt, st)) return rc;
    if (int rc = tfrpn_rpn_targets(h, anchors_dev, d_gt, d_gl, B, N, G, cfg, d_d, d_l, nullptr, st)) return rc;
    if (int rc = d2h(deltas_host, d_d, (size_t)B * N * 16, pin + b_gt + b_gl, st, job)) return rc;
    if (int rc = d2h(labels_host, d_l, (size_t)B * N * 4, pin + b_gt + b_gl + b_d, st, job)) return rc;
    return 0;
}

static int proposals_host_enqueue(tfrpn_handle h, const float* rpn_reg_host, const float* rpn_cls_host,
                                  const float* anchors_dev, int B, int N, const tfrpn_proposal_cfg* cfg,
                                  float* out_boxes_host, float* out_scores_host, int32_t* valid_host,
                                  int32_t* keep_idx_host_or_null, cudaStream_t st, HostJob& job) {
    if (!rpn_reg_host || !rpn_cls_host || !cfg || !out_boxes_host || !out_scores_host || !valid_host)
        return fail(TFRPN_ERR_BAD_ARG, "proposals_host: null pointer");
    if (B <= 0 || N <= 0 || cfg->post_nms_topn <= 0) return fail(TFRPN_ERR_BAD_ARG, "proposals_host: bad shape");
    if (int rc = check_iou_threshold("proposals_host", cfg->nms_iou_threshold)) return rc;
    const int P = cfg->post_nms_topn;
    const size_t b_reg = align256((size_t)B * N * 16), b_cls = align256((size_t)B * N * 4);
    const size_t b_ob = align256((size_t)B * P * 16), b_os = align256((size_t)B * P * 4);
    const size_t b_v = align256((size_t)B * 4), b_k = align256((size_t)B * P * 4);
    const size_t total = b_reg + b_cls + b_ob + b_os + b_v + b_k;
    if (int rc = grow_buffer(&h->dev2, &h->dev2_bytes, total, st, false)) return rc;
    if (int rc = grow_buffer(&h->pinned2, &h->pinned2_bytes, total, st, true)) return rc;
    char* d = h->dev2;
    char* pin = h->pinned2;
    float* d_reg = reinterpret_cast<float*>(d);
    float* d_cls = reinterpret_cast<float*>(d + b_reg);
    char* d_out = d + b_reg + b_cls;  // boxes | scores | valid | keep, contiguous
    float* d_ob = reinterpret_cast<float*>(d_out);
    float* d_os = reinterpret_cast<float*>(d_out + b_ob);
    int32_t* d_v = reinterpret_cast<int32_t*>(d_out + b_ob + b_os);
    int32_t* d_k = reinterpret_cast<int32_t*>(d_out + b_ob + b_os + b_v);
    if (int rc = h2d(d_reg, rpn_reg_host, (size_t)B * N * 16, pin, st)) return rc;
    if (int rc = h2d(d_cls, rpn_cls_host, (size_t)B * N * 4, pin + b_reg, st)) return rc;
    if (int rc = tfrpn_proposals(h, d_reg, d_cls, anchors_dev, B, N, cfg, d_ob, d_os, d_v, d_k, st)) return rc;
    // the four small results come back in ONE D2H copy through pinned staging
    char* p_out = pin + b_reg + b_cls;
    TFRPN_CHECK_CUDA(cudaMemcpyAsync(p_out, d_out, b_ob + b_os + b_v + b_k, cudaMemcpyDeviceToHost, st));
    job.add(out_boxes_host, p_out, (size_t)B * P * 16);
    job.add(out_scores_host, p_out + b_ob, (size_t)B * P * 4);
    job.add(valid_host, p_out + b_ob + b_os, (size_t)B * 4);
    if (keep_idx_host_or_null) job.add(keep_idx_host_or_null, p_out + b_ob + b_os + b_v, (size_t)B * P * 4);
    return 0;
}

extern "C" int tfrpn_rpn_targets_host(tfrpn_handle h, const float* anchors_dev, const float* gt_boxes_host,
                                      const int32_t* gt_labels_host, int B, int N, int G, const tfrpn_target_cfg* cfg,
                                      float* deltas_host, float* labels_host, tfrpn_stream s) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "rpn_targets_host: null handle");
    TFRPN_ENTER(h);
    HostJob job;
    if (int rc = targets_host_enqueue(h, anchors_dev, gt_boxes_host, gt_labels_host, B, N, G, cfg, deltas_host,
                                      labels_host, as_stream(s), job)) return rc;
    TFRPN_CHECK_CUDA(cudaStreamSynchronize(as_stream(s)));
    job.finish();
    return 0;
}

extern "C" int tfrpn_proposals_host(tfrpn_handle h, const float* rpn_reg_host, const float* rpn_cls_host,
                                    const float* anchors_dev, int B, int N, const tfrpn_proposal_cfg* cfg,
                                    float* out_boxes_host, float* out_scores_host, int32_t* valid_host,
                                    int32_t* keep_idx_host_or_null, tfrpn_stream s) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "proposals_host: null handle");
    TFRPN_ENTER(h);
    HostJob job;
    if (int rc = proposals_host_enqueue(h, rpn_reg_host, rpn_cls_host, anchors_dev, B, N, cfg, out_boxes_host,
                                        out_scores_host, valid_host, keep_idx_host_or_null, as_stream(s), job)) return rc;
    TFRPN_CHECK_CUDA(cudaStreamSynchronize(as_stream(s)));
    job.finish();
    return 0;
}
