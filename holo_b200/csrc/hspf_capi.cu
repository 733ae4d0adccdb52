// hspf_capi.cu — C ABI of the batched SPF engine (include/holo_spf.h).
//
// Host side: CSR validation, transposition, device residency, batch launch.
// There is no CPU compute path in this file: every result plane is produced by
// spf_batch_kernel on the device.
#include <algorithm>
#include <cstring>
#include <functional>
#include <new>
#include <string>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>

#include "holo_spf.h"
#include "quad_layout.h"
#include "spf_kernel.cuh"
#include "spf_quad.cuh"

using namespace hspf;

struct hspf_graph {
    DevGraph d{};
    void *blob = nullptr;      // single device allocation holding every array
    uint32_t max_indeg = 0;
    bool has_leaf = false;     // any HSPF_VF_LEAF / LEAF_UNLESS_ROOT vertex
    bool has_quads = false;    // quad-space image present (see quad_layout.h)
    bool fast = false;         // spf_quad_kernel serves this graph (decided once, at upload)
    QuadDev q{};
    QuadLayout qlay{};         // its shared-memory layout
    std::string why_not_fast;
    // host copies hspf_graph_update_costs validates against
    std::vector<uint32_t> h_row;
    std::vector<uint8_t> h_vflags;
};

struct hspf_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // D2H of finished jobs (host-pointer mode)
    cudaEvent_t chunk_done = nullptr;
    int sm_count = 0;
    size_t smem_optin = 0;
    std::string err;
    uint64_t launches = 0;
    uint32_t *d_counter = nullptr;
    // grow-only scratch
    void *ws = nullptr;      size_t ws_bytes = 0;       // global state workspace
    void *stage = nullptr;   size_t stage_bytes = 0;    // device staging of results (host-pointer mode)
    void *h_pin = nullptr;   size_t h_pin_bytes = 0;    // pinned bounce buffer
    void *scratch = nullptr; size_t scratch_bytes = 0;  // planes the caller did not ask for
    unsigned long long *d_prof = nullptr; int prof_rows = 0;  // optional phase counters (debug)
    bool prof_enabled = false;
    int path = HSPF_PATH_AUTO;                // hspf_debug_set_path
    // progress counters of the pipelined host-pointer call (see run_host)
    uint32_t *d_done = nullptr;               // [kMaxDoneChunks]
    uint32_t *prog_done = nullptr;            // set around one enqueue: the launch publishes per-chunk completion
    uint32_t prog_chunk = 0;
    CUresult (*wait_value)(CUstream, CUdeviceptr, cuuint32_t, unsigned int) = nullptr;
    cudaEvent_t prog_reset = nullptr;
    // fused exchange: peer slots the next 16-bit launches also write (hspf_ctx_set_peer_slots)
    uint32_t n_peer_slots = 0;
    long long peer_delta[7] = {0, 0, 0, 0, 0, 0, 0};
    int reserved_sms = 0;     // SMs left free for concurrent kernels (e.g. NCCL), see hspf_ctx_reserve_sms
};

namespace {

int fail(hspf_ctx *ctx, int code, const std::string &msg) {
    if (ctx) ctx->err = msg;
    return code;
}

int cuda_fail(hspf_ctx *ctx, cudaError_t e, const char *what) {
    return fail(ctx, HSPF_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define CK(call)                                              \
    do {                                                      \
        cudaError_t e_ = (call);                              \
        if (e_ != cudaSuccess) return cuda_fail(ctx, e_, #call); \
    } while (0)

int grow(hspf_ctx *ctx, void **p, size_t *have, size_t need, bool pinned = false) {
    if (*have >= need) return HSPF_OK;
    if (*p) {
        if (pinned) cudaFreeHost(*p); else cudaFree(*p);
        *p = nullptr; *have = 0;
    }
    size_t want = need + need / 4;
    cudaError_t e = pinned ? cudaMallocHost(p, want) : cudaMalloc(p, want);
    if (e != cudaSuccess) { *p = nullptr; return cuda_fail(ctx, e, pinned ? "cudaMallocHost" : "cudaMalloc"); }
    *have = want;
    return HSPF_OK;
}

// Result planes of either width: hspf_result (dist u32, first_parent u32, nh_mask u64 x nh_words)
// or hspf_result16 (all planes u16, one next-hop word of 16 atoms).
enum Plane { kDist, kHops, kFp, kNpar, kNh, kStatus, kPlanes };   // vertex planes, then the job status

struct AnyResult {
    void *p[kPlanes] = {};
    size_t bytes[kPlanes] = {};   // per vertex of a job; kStatus: per job
    uint32_t nh_words = 1;
    bool narrow = false;
};

AnyResult any_of(const hspf_result *r) {
    return {{r->dist, r->hops, r->first_parent, r->n_parents, r->nh_mask, r->job_status},
            {4, 2, 4, 2, 8 * (size_t)r->nh_words, 4}, r->nh_words, false};
}

AnyResult any_of(const hspf_result16 *r) {
    return {{r->dist, r->hops, r->first_parent, r->n_parents, r->nh_mask, r->job_status}, {2, 2, 2, 2, 2, 4}, 1, true};
}

// Points every null plane of `r` at its own 256-byte aligned region of a buffer at `base`, for n_jobs
// jobs of V vertices, and returns the bytes those regions take (base == nullptr: only counts).
size_t place_planes(AnyResult &r, uint32_t n_jobs, uint32_t V, uint8_t *base) {
    size_t used = 0;
    for (int k = 0; k < kPlanes; ++k) {
        if (r.p[k]) continue;
        if (base) r.p[k] = base + used;
        used += align_up((k == kStatus ? 1 : (size_t)V) * n_jobs * r.bytes[k], 256);
    }
    return used;
}

// Does spf_quad_kernel run this batch?  Decides enqueue's kernel and run_host's pipelined copy.
bool quad_runs(const hspf_ctx *ctx, const hspf_graph *g, const AnyResult &out) {
    return g->fast && out.nh_words == 1 && ctx->path == HSPF_PATH_AUTO;
}

// CTAs of `kernel` one SM holds with `smem` bytes of dynamic shared memory (0 when the query fails).
template <typename Args>
int ctas_per_sm(void (*kernel)(Args), int threads, size_t smem) {
    int n = 0;
    if (smem > 0) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess) n = 0;
    return n;
}

// Grid of a persistent launch, whose CTAs fetch jobs from ctx->d_counter: per_sm CTAs on every SM the
// ctx does not reserve, at most one per job.  Enqueues the reset of the job counter and, when
// profiling, of the phase counters (*prof) the launch adds to.
int begin_launch(hspf_ctx *ctx, int per_sm, uint32_t n_jobs, int &grid, unsigned long long *&prof) {
    grid = (ctx->sm_count - ctx->reserved_sms) * per_sm;
    if ((uint32_t)grid > n_jobs) grid = (int)n_jobs;
    if (grid < 1) grid = 1;
    prof = nullptr;
    if (ctx->prof_enabled) {
        if (ctx->prof_rows < grid) {
            if (ctx->d_prof) cudaFree(ctx->d_prof);
            ctx->d_prof = nullptr; ctx->prof_rows = 0;
            CK(cudaMalloc(&ctx->d_prof, (size_t)grid * 16 * sizeof(unsigned long long)));
            ctx->prof_rows = grid;
        }
        CK(cudaMemsetAsync(ctx->d_prof, 0, (size_t)ctx->prof_rows * 16 * sizeof(unsigned long long), ctx->stream));
        prof = ctx->d_prof;
    }
    CK(cudaMemsetAsync(ctx->d_counter, 0, sizeof(uint32_t), ctx->stream));
    return HSPF_OK;
}

template <typename Args>
int start(hspf_ctx *ctx, void (*kernel)(Args), int grid, int threads, size_t smem, const Args &a) {
    if (smem > 0) CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, threads, smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return HSPF_OK;
}

// The arguments both kernels share: graph, jobs, result planes, job counter.
template <typename Args>
Args kernel_args(const hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const AnyResult &out) {
    Args a{};
    a.g = g->d;
    a.n_jobs = jobs->n_jobs;
    a.roots = jobs->roots;
    a.ov_off = jobs->ov_off;
    a.ov_edge = jobs->ov_edge;
    a.ov_cost = jobs->ov_cost;
    a.out_dist = static_cast<uint32_t *>(out.p[kDist]);
    a.out_hops = static_cast<uint16_t *>(out.p[kHops]);
    a.out_fp = static_cast<uint32_t *>(out.p[kFp]);
    a.out_npar = static_cast<uint16_t *>(out.p[kNpar]);
    a.out_nh = static_cast<uint64_t *>(out.p[kNh]);
    a.out_status = static_cast<uint32_t *>(out.p[kStatus]);
    a.job_counter = ctx->d_counter;
    return a;
}

// Enqueue one batch.  All pointers in `jobs`/`out` are device pointers here.
int enqueue(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const AnyResult &out) {
    int grid = 0, rc;
    if (quad_runs(ctx, g, out)) {   // the fast path, spf_quad.cuh
        QuadArgs a = kernel_args<QuadArgs>(ctx, g, jobs, out);
        a.q = g->q;
        a.lay = g->qlay;
        a.narrow = out.narrow ? 1u : 0u;
        a.n_peers = out.narrow ? ctx->n_peer_slots : 0u;
        for (uint32_t k = 0; k < 7; ++k) a.peer_delta[k] = ctx->peer_delta[k];
        a.done = ctx->prog_done;
        a.done_chunk = ctx->prog_chunk ? ctx->prog_chunk : 1u;
        const auto kernel = jobs->ov_off ? spf_quad_kernel<true> : spf_quad_kernel<false>;
        CK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        const int per_sm = ctas_per_sm(kernel, kQuadThreads, a.lay.total);
        if (per_sm < 1) return fail(ctx, HSPF_E_CUDA, "spf_quad_kernel does not fit an SM");
        if ((rc = begin_launch(ctx, per_sm, jobs->n_jobs, grid, a.prof))) return rc;
        return start(ctx, kernel, grid, kQuadThreads, a.lay.total, a);
    }
    if (out.narrow)
        return fail(ctx, HSPF_E_UNSUPPORTED, "16-bit result planes need the packed fast path (" +
                    (g->fast ? std::string("general kernel selected by hspf_debug_set_path") : g->why_not_fast) + ")");
    const uint32_t V = g->d.V;
    const bool q16 = V <= 0xFFFFu;
    BatchArgs a = kernel_args<BatchArgs>(ctx, g, jobs, out);
    a.lay = make_layout(V, g->d.E, q16 ? 2 : 4);
    a.nhw = out.nh_words;
    const size_t sb = a.lay.total;
    // static smem of the kernel (Small) is ~4.5 KB; leave headroom
    const size_t smem_cap = ctx->smem_optin > 6144 ? ctx->smem_optin - 6144 : 0;
    const bool in_smem = sb <= smem_cap;
    // pointer-jumping next-hop phase: needs the aliased layout (dagbit in qa, words over dist)
    a.jump_ok = (ctx->path != HSPF_PATH_GENERAL_KAHN && in_smem && q16 && g->d.iedge16 && g->d.edge16 && g->d.iquad &&
                 a.lay.dagbit == a.lay.qa && a.lay.kq0 == a.lay.dist) ? 1u : 0u;
    // the grid is sized for the variant without the no-override specialisation
    using Kernel = void (*)(BatchArgs);
    const Kernel general = in_smem ? (q16 ? spf_batch_kernel<uint16_t, true, false> : spf_batch_kernel<uint32_t, true, false>)
                                   : (q16 ? spf_batch_kernel<uint16_t, false, false> : spf_batch_kernel<uint32_t, false, false>);
    const bool fast = in_smem && !jobs->ov_off && !(g->d.flags & HSPF_GF_HOPCOUNT) && !g->has_leaf && out.nh_words == 1;
    const Kernel kernel = !fast ? general : q16 ? spf_batch_kernel<uint16_t, true, true> : spf_batch_kernel<uint32_t, true, true>;
    const size_t smem = in_smem ? sb : 0;
    if ((rc = begin_launch(ctx, std::max(1, ctas_per_sm(general, kThreads, smem)), jobs->n_jobs, grid, a.prof))) return rc;
    if (!in_smem) {
        if ((rc = grow(ctx, &ctx->ws, &ctx->ws_bytes, sb * (size_t)grid))) return rc;
        a.ws = static_cast<uint8_t *>(ctx->ws);
        a.ws_stride = sb;
    }
    return start(ctx, kernel, grid, kThreads, smem, a);
}

// Device-pointer call.
int run_device(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const AnyResult &out) {
    // planes the caller skipped still have to exist on the device
    AnyResult r = out;
    if (const size_t need = place_planes(r, jobs->n_jobs, g->d.V, nullptr)) {
        if (const int rc = grow(ctx, &ctx->scratch, &ctx->scratch_bytes, need)) return rc;
        place_planes(r, jobs->n_jobs, g->d.V, static_cast<uint8_t *>(ctx->scratch));
    }
    return enqueue(ctx, g, jobs, r);
}

// D2H on the copy stream: jobs [j0, j0 + nj) of every vertex plane the caller asked for.
int copy_out(hspf_ctx *ctx, const AnyResult &host, const AnyResult &dev, uint32_t V, uint32_t j0, uint32_t nj) {
    for (int k = 0; k < kStatus; ++k) {
        if (!host.p[k]) continue;
        const size_t o = (size_t)j0 * V * host.bytes[k];
        CK(cudaMemcpyAsync(static_cast<uint8_t *>(host.p[k]) + o, static_cast<uint8_t *>(dev.p[k]) + o,
                           (size_t)nj * V * host.bytes[k], cudaMemcpyDeviceToHost, ctx->copy_stream));
    }
    return HSPF_OK;
}

// Host image of a device buffer (a graph's blob, a batch's job arrays): sections back to back, each
// 256-byte aligned, and the pointer fields to aim at them once the buffer has its device address.
struct BlobImage {
    std::vector<uint8_t> bytes;
    std::vector<std::function<void(const uint8_t *)>> bind;
    // n elements of src (null: the section stays zero); `field` is null unless `used`
    template <typename F, typename S>
    void add(const F *&field, const S *src, size_t n, bool used = true) {
        const size_t o = bytes.size();
        bytes.resize(o + align_up(n * sizeof(S), 256), 0);
        if (src && n) std::memcpy(bytes.data() + o, src, n * sizeof(S));
        field = nullptr;
        if (used) bind.push_back([&field, o](const uint8_t *b) { field = reinterpret_cast<const F *>(b + o); });
    }
    template <typename F, typename S>
    void add(const F *&field, const std::vector<S> &v, bool used = true) { add(field, v.data(), v.size(), used); }
};

// Host-pointer call: validate the jobs, stage them in, run, stage the planes out.
int run_host(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const AnyResult &out) {
    const uint32_t n = jobs->n_jobs, V = g->d.V;
    int rc;
    uint32_t n_ov = 0;
    for (uint32_t j = 0; j < n; ++j)
        if (jobs->roots[j] >= V) return fail(ctx, HSPF_E_INVAL, "root out of range");
    if (jobs->ov_off) {
        if (!jobs->ov_edge || !jobs->ov_cost) {
            if (jobs->ov_off[n] != 0) return fail(ctx, HSPF_E_INVAL, "null override arrays");
        }
        for (uint32_t j = 0; j < n; ++j) {
            if (jobs->ov_off[j + 1] < jobs->ov_off[j]) return fail(ctx, HSPF_E_INVAL, "ov_off not monotone");
            if (jobs->ov_off[j + 1] - jobs->ov_off[j] > HSPF_MAX_OVERRIDES)
                return fail(ctx, HSPF_E_UNSUPPORTED, "more than HSPF_MAX_OVERRIDES overrides in a job");
        }
        n_ov = jobs->ov_off[n];
        for (uint32_t i = 0; i < n_ov; ++i)
            if (jobs->ov_edge[i] >= g->d.E) return fail(ctx, HSPF_E_INVAL, "override edge out of range");
    }
    hspf_jobs dj{};
    dj.n_jobs = n;
    BlobImage in;
    in.add(dj.roots, jobs->roots, n);
    in.add(dj.ov_off, jobs->ov_off, jobs->ov_off ? n + 1 : 0, jobs->ov_off != nullptr);
    in.add(dj.ov_edge, jobs->ov_edge, n_ov);
    in.add(dj.ov_cost, jobs->ov_cost, n_ov);
    const size_t in_total = in.bytes.size();
    AnyResult dr = out;
    for (void *&p : dr.p) p = nullptr;
    const size_t dev_total = in_total + place_planes(dr, n, V, nullptr);
    rc = grow(ctx, &ctx->stage, &ctx->stage_bytes, dev_total);
    if (rc) return rc;
    rc = grow(ctx, &ctx->h_pin, &ctx->h_pin_bytes, in_total, true);
    if (rc) return rc;
    uint8_t *dp = static_cast<uint8_t *>(ctx->stage);
    std::memcpy(ctx->h_pin, in.bytes.data(), in_total);
    CK(cudaMemcpyAsync(dp, ctx->h_pin, in_total, cudaMemcpyHostToDevice, ctx->stream));
    for (auto &b : in.bind) b(dp);
    place_planes(dr, n, V, dp + in_total);
    // Fast path: ONE launch for the whole batch; the kernel counts finished jobs per piece
    // (release ordered behind their planes) and the copy stream waits on those counters with
    // stream memory operations, so a piece's planes travel to the host while the rest of the
    // batch still computes.  (Launching the batch in pieces instead costs more than it hides:
    // a launch cannot finish faster than one job's latency.  Measured on B200, C2, 6 B/vertex:
    // 1 piece 631 k SPF/s, 4 pieces 532 k, 16 pieces 264 k.)  Four pieces: few, large copies,
    // every cudaMemcpyAsync costs ~10 us here.
    const bool pipelined = quad_runs(ctx, g, out) && ctx->wait_value && n >= 256;
    const uint32_t piece = (n + 3) / 4;
    if (pipelined) {
        CK(cudaMemsetAsync(ctx->d_done, 0, 64 * sizeof(uint32_t), ctx->stream));
        CK(cudaEventRecord(ctx->prog_reset, ctx->stream));
        ctx->prog_done = ctx->d_done; ctx->prog_chunk = piece;
    }
    rc = enqueue(ctx, g, &dj, dr);
    ctx->prog_done = nullptr; ctx->prog_chunk = 0;
    if (rc) return rc;
    CK(cudaEventRecord(ctx->chunk_done, ctx->stream));
    cudaStream_t cs = ctx->copy_stream;
    if (pipelined) {
        CK(cudaStreamWaitEvent(cs, ctx->prog_reset, 0));       // the counters of this call, not of the last one
        for (uint32_t c = 0, c0 = 0; c0 < n; ++c, c0 += piece) {
            const uint32_t cn = std::min(piece, n - c0);
            if (ctx->wait_value(reinterpret_cast<CUstream>(cs), reinterpret_cast<CUdeviceptr>(ctx->d_done + c), cn,
                                CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
                return fail(ctx, HSPF_E_CUDA, "cuStreamWaitValue32 failed");
            if ((rc = copy_out(ctx, out, dr, V, c0, cn))) return rc;
        }
    }
    CK(cudaStreamWaitEvent(cs, ctx->chunk_done, 0));
    if (!pipelined && (rc = copy_out(ctx, out, dr, V, 0, n))) return rc;
    std::vector<uint32_t> st(n);
    CK(cudaMemcpyAsync(st.data(), dr.p[kStatus], (size_t)n * 4, cudaMemcpyDeviceToHost, cs));
    CK(cudaStreamSynchronize(cs));
    CK(cudaStreamSynchronize(ctx->stream));
    bool any = false;
    for (uint32_t j = 0; j < n; ++j) any |= (st[j] != 0);
    if (out.p[kStatus]) std::memcpy(out.p[kStatus], st.data(), (size_t)n * 4);
    if (any) return fail(ctx, HSPF_E_JOB_STATUS, "one or more jobs need the CPU path (see job_status)");
    return HSPF_OK;
}

// The four run calls: shared checks, then the device-pointer call (synchronised unless async) or the
// host-pointer call.
template <typename R>
int run_checked(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const R *out, bool async, uint32_t flags) {
    if (!ctx || !g || !jobs) return HSPF_E_INVAL;
    if (!out) return fail(ctx, HSPF_E_INVAL, "null result");
    const AnyResult r = any_of(out);
    if (r.nh_words < 1 || r.nh_words > 4) return fail(ctx, HSPF_E_INVAL, "nh_words must be 1..4");
    if (jobs->n_jobs == 0) return HSPF_OK;
    if (!jobs->roots) return fail(ctx, HSPF_E_INVAL, "null roots");
    try {
        CK(cudaSetDevice(ctx->device));
        if (!async && !(flags & HSPF_RUN_DEVICE_PTRS)) return run_host(ctx, g, jobs, r);
        const int rc = run_device(ctx, g, jobs, r);
        if (rc || async) return rc;
        CK(cudaStreamSynchronize(ctx->stream));
        return HSPF_OK;   // job_status stays on the device in this mode
    } catch (const std::bad_alloc &) {
        return fail(ctx, HSPF_E_NOMEM, "host allocation failed");
    } catch (...) {
        return fail(ctx, HSPF_E_INVAL, "unexpected exception");
    }
}

// Transposed CSR: the in-edges of v are src/cost/fwd[irow[v] .. irow[v + 1]), ordered by (source,
// forward edge index).  col[] must be in range.
struct Transposed {
    std::vector<uint32_t> irow, src, cost, fwd;
};

Transposed transpose(const hspf_csr *g) {
    const uint32_t V = g->n_vertices, E = g->n_edges;
    Transposed t;
    t.irow.assign(V + 1, 0);
    t.src.resize(E); t.cost.resize(E); t.fwd.resize(E);
    for (uint32_t e = 0; e < E; ++e) t.irow[g->col[e] + 1]++;
    for (uint32_t v = 0; v < V; ++v) t.irow[v + 1] += t.irow[v];
    std::vector<uint32_t> fill(t.irow.begin(), t.irow.end() - 1);
    for (uint32_t u = 0; u < V; ++u)
        for (uint32_t e = g->row_ptr[u]; e < g->row_ptr[u + 1]; ++e) {
            const uint32_t k = fill[g->col[e]]++;
            t.src[k] = u; t.cost[k] = g->cost[e]; t.fwd[k] = e;
        }
    return t;
}

QuadHost quads_of(const hspf_csr *g, const Transposed &t) {
    return build_quads(g->n_vertices, g->n_edges, g->row_ptr, g->col, g->cost, g->vflags, t.irow.data(), t.src.data(),
                       t.cost.data(), t.fwd.data(), g->delta);
}

}  // namespace

extern "C" {

const char *hspf_version(void) { return "holo_spf 0.1 sm_100a"; }

int hspf_ctx_create(int device, hspf_ctx **out) {
    if (!out) return HSPF_E_INVAL;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0 || device < 0 || device >= n) return HSPF_E_CUDA;
    hspf_ctx *ctx = new (std::nothrow) hspf_ctx();
    if (!ctx) return HSPF_E_NOMEM;
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return HSPF_E_CUDA; }
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return HSPF_E_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return HSPF_E_CUDA; }
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->chunk_done, cudaEventDisableTiming) != cudaSuccess ||
        cudaMalloc(&ctx->d_counter, sizeof(uint32_t)) != cudaSuccess) {
        if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
        if (ctx->chunk_done) cudaEventDestroy(ctx->chunk_done);
        cudaStreamDestroy(ctx->stream); delete ctx; return HSPF_E_CUDA;
    }
    // optional: stream memory operations for the pipelined host-pointer call
    {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &q) == cudaSuccess && fn &&
            q == cudaDriverEntryPointSuccess &&
            cudaMalloc(&ctx->d_done, 64 * sizeof(uint32_t)) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->prog_reset, cudaEventDisableTiming) == cudaSuccess)
            ctx->wait_value = reinterpret_cast<decltype(ctx->wait_value)>(fn);
    }
    *out = ctx;
    return HSPF_OK;
}

void hspf_ctx_destroy(hspf_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    if (ctx->chunk_done) cudaEventDestroy(ctx->chunk_done);
    if (ctx->d_counter) cudaFree(ctx->d_counter);
    if (ctx->d_done) cudaFree(ctx->d_done);
    if (ctx->prog_reset) cudaEventDestroy(ctx->prog_reset);
    if (ctx->d_prof) cudaFree(ctx->d_prof);
    if (ctx->ws) cudaFree(ctx->ws);
    if (ctx->stage) cudaFree(ctx->stage);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    delete ctx;
}

const char *hspf_last_error(const hspf_ctx *ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

void *hspf_stream(hspf_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

uint64_t hspf_launch_count(const hspf_ctx *ctx) { return ctx ? ctx->launches : 0; }
/* kernels other translation units of the library enqueue on the ctx stream (route_cells.h) */
void hspf_note_launches(hspf_ctx *ctx, uint32_t n) { if (ctx) ctx->launches += n; }
int hspf_ctx_device(const hspf_ctx *ctx) { return ctx ? ctx->device : -1; }

int hspf_ctx_set_peer_slots(hspf_ctx *ctx, uint32_t n_peers, const int64_t *deltas) {
    if (!ctx || n_peers > 7 || (n_peers && !deltas)) return HSPF_E_INVAL;
    ctx->n_peer_slots = n_peers;
    for (uint32_t k = 0; k < n_peers; ++k) ctx->peer_delta[k] = (long long)deltas[k];
    return HSPF_OK;
}

int hspf_ctx_reserve_sms(hspf_ctx *ctx, int n_sms) {
    if (!ctx || n_sms < 0 || n_sms >= ctx->sm_count) return HSPF_E_INVAL;
    ctx->reserved_sms = n_sms;
    return HSPF_OK;
}

int hspf_debug_phase_profile(hspf_ctx *ctx, int enable, uint64_t out[16]) {
    if (!ctx) return HSPF_E_INVAL;
    if (out) {
        for (int k = 0; k < 16; ++k) out[k] = 0;
        if (ctx->d_prof && ctx->prof_rows > 0) {
            CK(cudaStreamSynchronize(ctx->stream));
            std::vector<unsigned long long> h((size_t)ctx->prof_rows * 16);
            CK(cudaMemcpy(h.data(), ctx->d_prof, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            for (int r = 0; r < ctx->prof_rows; ++r)
                for (int k = 0; k < 16; ++k) out[k] += h[(size_t)r * 16 + k];
        }
    }
    ctx->prof_enabled = enable != 0;
    return HSPF_OK;
}

int hspf_debug_set_path(hspf_ctx *ctx, int path) {
    if (!ctx || path < HSPF_PATH_AUTO || path > HSPF_PATH_GENERAL_KAHN) return HSPF_E_INVAL;
    ctx->path = path;
    return HSPF_OK;
}

int hspf_graph_upload(hspf_ctx *ctx, const hspf_csr *g, hspf_graph **out) {
    if (!ctx || !g || !out) return HSPF_E_INVAL;
    *out = nullptr;
    try {
        const uint32_t V = g->n_vertices, E = g->n_edges;
        if (V == 0 || V >= 0xFFFFFFF0u) return fail(ctx, HSPF_E_INVAL, "n_vertices out of range");
        if (!g->row_ptr || !g->vflags || (E && (!g->col || !g->cost))) return fail(ctx, HSPF_E_INVAL, "null CSR array");
        if (g->row_ptr[0] != 0 || g->row_ptr[V] != E) return fail(ctx, HSPF_E_INVAL, "row_ptr[0]!=0 or row_ptr[V]!=E");
        bool zero_cost_hop_tail = false;
        uint64_t cost_sum = 0;
        for (uint32_t u = 0; u < V; ++u) {
            if (g->row_ptr[u + 1] < g->row_ptr[u]) return fail(ctx, HSPF_E_INVAL, "row_ptr not monotone");
            const bool uh = g->vflags[u] & HSPF_VF_HOP;
            for (uint32_t e = g->row_ptr[u]; e < g->row_ptr[u + 1]; ++e) {
                const uint32_t v = g->col[e];
                if (v >= V) return fail(ctx, HSPF_E_INVAL, "col out of range");
                if (v == u) return fail(ctx, HSPF_E_INVAL, "self loop");
                if (g->cost[e] == HSPF_COST_DISABLED) return fail(ctx, HSPF_E_INVAL, "cost 0xFFFFFFFF is reserved");
                if (!uh && !(g->vflags[v] & HSPF_VF_HOP)) return fail(ctx, HSPF_E_INVAL, "edge joins two non-HOP vertices");
                if (uh && g->cost[e] == 0) zero_cost_hop_tail = true;
                cost_sum += g->cost[e];
            }
        }
        if (g->flags & HSPF_GF_HOPCOUNT) {
            for (uint32_t u = 0; u < V; ++u)
                for (uint32_t e = g->row_ptr[u]; e < g->row_ptr[u + 1]; ++e) {
                    const bool zero = (g->vflags[u] & HSPF_VF_HOP) && !(g->vflags[g->col[e]] & HSPF_VF_HOP);
                    if (g->cost[e] != (zero ? 0u : 1u))
                        return fail(ctx, HSPF_E_INVAL, "HSPF_GF_HOPCOUNT: costs must be 0 (HOP->non-HOP) or 1");
                }
        } else if (zero_cost_hop_tail)
            return fail(ctx, HSPF_E_NEEDS_ORACLE,
                        "zero-cost link out of a hop-counting vertex: ECMP DAG depends on pop order");
        const Transposed t = transpose(g);
        uint32_t max_indeg = 0;
        for (uint32_t v = 0; v < V; ++v) max_indeg = std::max(max_indeg, t.irow[v + 1] - t.irow[v]);
        if (max_indeg >= 0xFFFFu) return fail(ctx, HSPF_E_UNSUPPORTED, "in-degree >= 65535");

        std::vector<uint4> iedge(E);
        std::vector<uint2> fedge(E);
        for (uint32_t k = 0; k < E; ++k) iedge[k] = make_uint4(t.src[k], t.cost[k], t.fwd[k], 0u);
        for (uint32_t e = 0; e < E; ++e) fedge[e] = make_uint2(g->col[e], g->cost[e]);

        // compact twins used by the jump phase when ids and costs fit 16 bits: row offsets
        // (kept in shared memory during the SSSP) and in-edges as (source | cost << 16)
        uint32_t max_cost = 0;
        for (uint32_t e = 0; e < E; ++e) max_cost = std::max(max_cost, g->cost[e]);
        const bool pack_rows = V <= 0xFFFFu && E <= 0xFFFFu;
        const bool pack_in = V <= 0xFFFFu && max_cost <= 0xFFFFu;
        std::vector<uint16_t> row16(pack_rows ? V : 0);
        for (uint32_t v = 0; v < (uint32_t)row16.size(); ++v) row16[v] = (uint16_t)g->row_ptr[v];
        std::vector<uint32_t> iedge16(pack_in ? E : 0);
        for (uint32_t k = 0; k < (uint32_t)iedge16.size(); ++k) iedge16[k] = t.src[k] | (t.cost[k] << 16);
        // ... and the same in-edge records padded per vertex to whole 16-byte quads (pad record:
        // the vertex itself with cost 0xFFFF, which can never be a parent), so the parents pass reads the usual
        // four in-edges of a vertex with one 128-bit load
        std::vector<uint32_t> iquad_row(pack_in ? V + 1 : 0);
        std::vector<uint32_t> iquad;
        if (pack_in) {
            for (uint32_t v = 0; v < V; ++v) {
                iquad_row[v] = (uint32_t)(iquad.size() / 4);
                for (uint32_t k = t.irow[v]; k < t.irow[v + 1]; ++k) iquad.push_back(iedge16[k]);
                while (iquad.size() % 4) iquad.push_back(v | 0xFFFF0000u);   // pad: self-loop, never a parent
            }
            iquad_row[V] = (uint32_t)(iquad.size() / 4);
        }
        std::vector<uint32_t> edge16(pack_in ? E : 0);     // forward edges as (head | cost << 16)
        for (uint32_t e = 0; e < (uint32_t)edge16.size(); ++e) edge16[e] = fedge[e].x | (fedge[e].y << 16);

        // quad-space image for spf_quad_kernel (quad_layout.h), when ids and costs pack
        const QuadHost QH = quads_of(g, t);

        hspf_graph *G = new hspf_graph();
        G->has_quads = QH.eligible && !iedge16.empty();
        BlobImage img;
        img.add(G->d.row, g->row_ptr, V + 1);
        img.add(G->d.edge, fedge);
        img.add(G->d.irow, t.irow);
        img.add(G->d.iedge, iedge);
        img.add(G->d.vflags, g->vflags, V);
        img.add(G->d.row16, row16, !row16.empty());
        img.add(G->d.iedge16, iedge16, !iedge16.empty());
        img.add(G->d.edge16, edge16, !edge16.empty());
        img.add(G->d.iquad_row, iquad_row, !iquad_row.empty());
        img.add(G->d.iquad, iquad, !iquad.empty());
        // (a graph that fails late in build_quads keeps the room of the arrays built so far, zeroed)
        auto add_quads = [&](auto &field, const auto &v) { img.add(field, QH.eligible ? v.data() : nullptr, v.size(), G->has_quads); };
        add_quads(G->q.fq, QH.fq);
        add_quads(G->q.fcont, QH.fcont);
        add_quads(G->q.slot_of, QH.slot_of);
        add_quads(G->q.vert_of, QH.vert_of);
        add_quads(G->q.iq, QH.iq);
        add_quads(G->q.imeta, QH.imeta);
        add_quads(G->q.fpos, QH.fpos);
        add_quads(G->q.ipos, QH.ipos);
        cudaError_t e = cudaSetDevice(ctx->device);
        if (e == cudaSuccess) e = cudaMalloc(&G->blob, img.bytes.size());
        if (e != cudaSuccess) { delete G; return cuda_fail(ctx, e, "cudaMalloc(graph)"); }
        e = cudaMemcpyAsync(G->blob, img.bytes.data(), img.bytes.size(), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { cudaFree(G->blob); delete G; return cuda_fail(ctx, e, "graph H2D"); }
        for (auto &b : img.bind) b(static_cast<const uint8_t *>(G->blob));

        G->d.V = V; G->d.E = E;
        if (G->has_quads) {
            G->q.NQ = QH.NQ; G->q.NIQ = QH.NIQ; G->q.shift = QH.shift;
            uint32_t st = 0;
            while ((1u << st) < QH.max_ichain) ++st;
            G->q.isteps = st;
        }
        G->d.reject_above = g->reject_above;
        G->d.saturate_at = g->saturate_at;
        G->d.flags = g->flags;
        uint32_t delta = g->delta;
        if (delta == 0) {
            // near/far bucket width: ~4x the mean link cost keeps the SSSP at a few buckets
            // (fewer barrier rounds) with ~1.3x re-expansion on the BASELINE shapes
            uint64_t mean = E ? cost_sum / E : 1;
            delta = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(4 * mean, 1), 0x7FFFFFFFu);
        }
        G->d.delta = delta;
        G->max_indeg = max_indeg;
        G->h_row.assign(g->row_ptr, g->row_ptr + V + 1);
        G->h_vflags.assign(g->vflags, g->vflags + V);
        for (uint32_t v = 0; v < V; ++v)
            if (g->vflags[v] & (HSPF_VF_LEAF | HSPF_VF_LEAF_UNLESS_ROOT)) G->has_leaf = true;
        // the fast path, decided once: its per-job state must fit this device's shared memory (2 KB
        // headroom for the kernel's static shared memory)
        if (!G->has_quads) {
            G->why_not_fast = QH.why;
        } else if (G->has_leaf || (g->flags & HSPF_GF_HOPCOUNT)) {
            G->why_not_fast = "LEAF flags / hop-count mode";
        } else {
            G->qlay = make_quad_layout(V, QH.NQ);
            G->fast = (size_t)G->qlay.total + 2048 <= ctx->smem_optin;
            if (!G->fast) G->why_not_fast = "per-job state exceeds shared memory";
        }
        *out = G;
        return HSPF_OK;
    } catch (const std::bad_alloc &) {
        return fail(ctx, HSPF_E_NOMEM, "host allocation failed");
    } catch (...) {
        return fail(ctx, HSPF_E_INVAL, "unexpected exception");
    }
}

int hspf_graph_update_costs(hspf_ctx *ctx, hspf_graph *g, uint32_t n, const uint32_t *edges, const uint32_t *costs) {
    if (!ctx || !g || (n && (!edges || !costs))) return HSPF_E_INVAL;
    if (n == 0) return HSPF_OK;
    try {
        if (g->d.flags & HSPF_GF_HOPCOUNT) return fail(ctx, HSPF_E_UNSUPPORTED, "hop-count graphs have fixed costs");
        for (uint32_t i = 0; i < n; ++i) {
            const uint32_t e = edges[i], c = costs[i];
            if (e >= g->d.E) return fail(ctx, HSPF_E_INVAL, "edge out of range");
            if (c == HSPF_COST_DISABLED) return fail(ctx, HSPF_E_INVAL, "cost 0xFFFFFFFF is reserved");
            const uint32_t tail = (uint32_t)(std::upper_bound(g->h_row.begin(), g->h_row.end(), e) - g->h_row.begin()) - 1;
            if (c == 0 && (g->h_vflags[tail] & HSPF_VF_HOP))
                return fail(ctx, HSPF_E_NEEDS_ORACLE, "zero-cost link out of a hop-counting vertex");
            if (g->d.iedge16 && c > 0xFFFFu) return fail(ctx, HSPF_E_UNSUPPORTED, "cost does not fit the packed image");
            if (g->has_quads && (c > 65534u || (unsigned long long)c > (3ull << g->q.shift)))
                return fail(ctx, HSPF_E_UNSUPPORTED, "cost outside the bucket ring of the uploaded image");
        }
        cudaError_t er = cudaSetDevice(ctx->device);
        uint32_t *d = nullptr;
        if (er == cudaSuccess) er = cudaMalloc(&d, (size_t)n * 8);
        if (er != cudaSuccess) return cuda_fail(ctx, er, "cudaMalloc(cost patch)");
        er = cudaMemcpyAsync(d, edges, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
        if (er == cudaSuccess) er = cudaMemcpyAsync(d + n, costs, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
        if (er == cudaSuccess) {
            hspf::patch_costs_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(g->d, g->q, g->has_quads, n, d, d + n);
            er = cudaGetLastError();
            ctx->launches++;
        }
        if (er == cudaSuccess) er = cudaStreamSynchronize(ctx->stream);
        cudaFree(d);
        if (er != cudaSuccess) return cuda_fail(ctx, er, "cost patch");
        return HSPF_OK;
    } catch (const std::bad_alloc &) {
        return fail(ctx, HSPF_E_NOMEM, "host allocation failed");
    }
}

void hspf_graph_free(hspf_ctx *ctx, hspf_graph *g) {
    if (!g) return;
    if (ctx) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); }
    if (g->blob) cudaFree(g->blob);
    delete g;
}

int hspf_sync(hspf_ctx *ctx) {
    if (!ctx) return HSPF_E_INVAL;
    CK(cudaStreamSynchronize(ctx->stream));
    return HSPF_OK;
}

int hspf_run_batch_async(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const hspf_result *out) {
    return run_checked(ctx, g, jobs, out, true, 0);
}

int hspf_run_batch(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const hspf_result *out, uint32_t flags) {
    return run_checked(ctx, g, jobs, out, false, flags);
}

int hspf_run_batch16_async(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const hspf_result16 *out) {
    return run_checked(ctx, g, jobs, out, true, 0);
}

int hspf_run_batch16(hspf_ctx *ctx, const hspf_graph *g, const hspf_jobs *jobs, const hspf_result16 *out, uint32_t flags) {
    return run_checked(ctx, g, jobs, out, false, flags);
}

int hspf_graph_info(const hspf_graph *g, uint32_t info[8]) {
    if (!g || !info) return HSPF_E_INVAL;
    info[0] = g->fast ? 1u : 0u;   // fast path / 16-bit planes available
    info[1] = g->q.NQ; info[2] = g->q.NIQ; info[3] = g->q.shift;   // zero without a quad image
    info[4] = g->d.V; info[5] = g->d.E; info[6] = g->max_indeg; info[7] = 0;
    return HSPF_OK;
}

int hspf_debug_quad_image(const hspf_csr *g, uint32_t hdr[8], uint32_t *fq, uint32_t *fcont, uint16_t *slot_of,
                          uint16_t *vert_of, uint32_t *iq, uint32_t *imeta, uint32_t *fpos, uint32_t *ipos) {
    if (!g || !hdr) return HSPF_E_INVAL;
    try {
        for (uint32_t e = 0; e < g->n_edges; ++e)
            if (g->col[e] >= g->n_vertices) return HSPF_E_INVAL;
        const QuadHost Q = quads_of(g, transpose(g));
        hdr[0] = Q.eligible ? 1u : 0u; hdr[1] = Q.NQ; hdr[2] = Q.NIQ; hdr[3] = Q.shift;
        hdr[4] = Q.max_ichain; hdr[5] = Q.max_atoms; hdr[6] = 0; hdr[7] = 0;
        if (!Q.eligible) return HSPF_OK;
        auto cp = [](auto *dst, const auto &v) { if (dst && !v.empty()) std::memcpy(dst, v.data(), v.size() * sizeof(v[0])); };
        cp(fq, Q.fq); cp(fcont, Q.fcont); cp(slot_of, Q.slot_of); cp(vert_of, Q.vert_of);
        cp(iq, Q.iq); cp(imeta, Q.imeta); cp(fpos, Q.fpos); cp(ipos, Q.ipos);
        return HSPF_OK;
    } catch (...) {
        return HSPF_E_NOMEM;
    }
}

int hspf_atom_count(const hspf_csr *g, uint32_t root, uint32_t *n_atoms) {
    if (!g || !n_atoms || root >= g->n_vertices) return HSPF_E_INVAL;
    uint32_t rb = g->row_ptr[root], re = g->row_ptr[root + 1];
    uint32_t n = re - rb;
    for (uint32_t e = rb; e < re; ++e) {
        uint32_t h = g->col[e];
        if (!(g->vflags[h] & HSPF_VF_HOP)) n += g->row_ptr[h + 1] - g->row_ptr[h];
    }
    *n_atoms = n;
    return HSPF_OK;
}

int hspf_atom_decode(const hspf_csr *g, uint32_t root, uint32_t atom, uint32_t *tail, uint32_t *edge) {
    if (!g || !tail || !edge || root >= g->n_vertices) return HSPF_E_INVAL;
    uint32_t rb = g->row_ptr[root], re = g->row_ptr[root + 1];
    uint32_t deg = re - rb;
    if (atom < deg) { *tail = root; *edge = rb + atom; return HSPF_OK; }
    uint32_t base = deg;
    for (uint32_t e = rb; e < re; ++e) {
        uint32_t h = g->col[e];
        if (g->vflags[h] & HSPF_VF_HOP) continue;
        uint32_t d = g->row_ptr[h + 1] - g->row_ptr[h];
        if (atom < base + d) { *tail = h; *edge = g->row_ptr[h] + (atom - base); return HSPF_OK; }
        base += d;
    }
    return HSPF_E_INVAL;
}

}  // extern "C"
