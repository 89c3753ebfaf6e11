// C ABI of libfluidaudio_b200.so (declared in include/fluidaudio_b200.h and include/FastClusterWrapper.h).
// No exception and no CUDA type crosses this boundary; there is no CPU fallback behind it.
#include "../../include/FastClusterWrapper.h"
#include "../../include/fluidaudio_b200.h"

#include "ahc_plan.h"
#include "assign_host.h"
#include "mel_plan.h"
#include "vbx_plan.h"
#include "kmeans_plan.h"
#include "reconstruct_host.h"

#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <set>
#include <string>
#include <thread>
#include <vector>

#define FA_API extern "C" __attribute__((visibility("default")))

namespace fa {

static thread_local char g_error[512] = "";
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}
const char *last_error() { return g_error; }

static std::atomic<long long> g_launches{0};

#define FA_CUDA_TRY(expr)                                                                               \
    do {                                                                                                \
        cudaError_t e__ = (expr);                                                                       \
        if (e__ != cudaSuccess) {                                                                       \
            fa::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return e__ == cudaErrorMemoryAllocation ? FA_ALLOCATION_FAILURE : FA_CUDA_ERROR;            \
        }                                                                                               \
    } while (0)

static int usable_device_count() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int i = 0; i < n; ++i) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
    }
    return ok;
}

static int require_device() {
    static std::atomic<int> cached{-1};
    int c = cached.load();
    if (c < 0) {
        c = usable_device_count();
        cached.store(c);
    }
    if (c <= 0) {
        set_error("no sm_100a (B200) device visible; fluidaudio_b200 has no CPU fallback");
        return FA_NO_DEVICE;
    }
    return FA_OK;
}

// ---- clustering context: one per concurrent caller, leased from a pool (the reference boundary is
// synchronous, stateless and re-entrant: FastClusterWrapper.cpp keeps no state, SURVEY §8b) -------------
struct ClusterContext {
    int device = 0;
    cudaStream_t stream = nullptr;
    ahc::Solver solver;
    vbx::Workspace vbx_ws, cent_ws;
    // pipeline buffers
    void *d_buf = nullptr;
    size_t d_bytes = 0;
    void *h_buf = nullptr;
    size_t h_bytes = 0;
    cudaEvent_t ev[8] = {};
    bool ready = false;
    int worker_limit = 0;

    int init(int worker_lim) {
        FA_CUDA_TRY(cudaGetDevice(&device));
        FA_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        for (auto &e : ev) FA_CUDA_TRY(cudaEventCreate(&e));
        worker_limit = worker_lim;
        const int st = solver.init(stream, worker_lim);
        if (st != FA_OK) return st;
        ready = true;
        return FA_OK;
    }
    ~ClusterContext() {
        if (d_buf) cudaFree(d_buf);
        if (h_buf) cudaFreeHost(h_buf);
        for (auto &e : ev)
            if (e) cudaEventDestroy(e);
        if (stream) cudaStreamDestroy(stream);
    }
    int reserve(size_t dbytes, size_t hbytes) {
        if (dbytes > d_bytes) {
            if (d_buf) cudaFree(d_buf);
            d_buf = nullptr;
            d_bytes = 0;
            FA_CUDA_TRY(cudaMalloc(&d_buf, dbytes));
            d_bytes = dbytes;
        }
        if (hbytes > h_bytes) {
            if (h_buf) cudaFreeHost(h_buf);
            h_buf = nullptr;
            h_bytes = 0;
            FA_CUDA_TRY(cudaMallocHost(&h_buf, hbytes));
            h_bytes = hbytes;
        }
        return FA_OK;
    }
};

static std::mutex g_pool_mutex;
static std::vector<std::unique_ptr<ClusterContext>> g_pool;   // idle contexts

struct Lease {
    std::unique_ptr<ClusterContext> ctx;
    int status = FA_OK;
    explicit Lease(int worker_limit = 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) {
            set_error("cudaGetDevice failed");
            status = FA_CUDA_ERROR;
            return;
        }
        {
            std::lock_guard<std::mutex> lock(g_pool_mutex);
            for (size_t i = 0; i < g_pool.size(); ++i)
                if (g_pool[i]->device == dev && g_pool[i]->worker_limit == worker_limit) {
                    ctx = std::move(g_pool[i]);
                    g_pool.erase(g_pool.begin() + i);
                    break;
                }
        }
        if (!ctx) {
            ctx.reset(new ClusterContext());
            status = ctx->init(worker_limit);
        }
    }
    ~Lease() {
        if (ctx && ctx->ready && status != FA_CUDA_ERROR) {
            std::lock_guard<std::mutex> lock(g_pool_mutex);
            g_pool.push_back(std::move(ctx));
        }
    }
};

struct Carver {
    char *base;
    size_t off = 0;
    template <typename T> T *take(size_t count) {
        off = (off + 255) & ~size_t(255);
        T *p = reinterpret_cast<T *>(base + off);
        off += count * sizeof(T);
        return p;
    }
};

static float ms_between(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

// OfflineDiarizerManager.cluster(_:) :286-375 on one context.  All inputs are host pointers.
static int cluster_pipeline(ClusterContext &C, const float *emb, const double *rho, size_t N, size_t E, size_t R,
                            const double *psi, const fa_cluster_config &cfg, int32_t *labels, int32_t *initial_out,
                            double *centroids_out, int32_t max_centroids, fa_cluster_info *info,
                            const int32_t *chunk_index = nullptr) {
    const auto wall0 = std::chrono::steady_clock::now();
    cudaStream_t s = C.stream;
    const int n = (int)N, e = (int)E, r = (int)R;
    // ---- device arena -----------------------------------------------------------------------------------
    size_t bytes = 0;
    {
        Carver c{nullptr};
        c.take<float>(N * E);
        c.take<double>(N * E);       // embd
        c.take<double>(N * R);       // rho
        c.take<unsigned char>(N);
        c.take<int>(N);              // train idx
        c.take<double>(N * E);       // train
        c.take<double>(N * R);       // train rho
        c.take<double>(N * E);       // normalised train
        c.take<int>(N);              // init labels
        c.take<int>(N);              // hard
        c.take<int>(N);              // labels
        c.take<int>(64);
        bytes = c.off + 4096;
    }
    int st = C.reserve(bytes, N * (sizeof(int) * 4 + 8) + (N > 1 ? (N - 1) * 4 * sizeof(double) : 0) + 4096);
    if (st != FA_OK) return st;
    Carver c{static_cast<char *>(C.d_buf)};
    float *d_emb32 = c.take<float>(N * E);
    double *d_emb = c.take<double>(N * E);
    double *d_rho = c.take<double>(N * R);
    unsigned char *d_ok = c.take<unsigned char>(N);
    int *d_idx = c.take<int>(N);
    double *d_train = c.take<double>(N * E);
    double *d_train_rho = c.take<double>(N * R);
    double *d_norm = c.take<double>(N * E);
    int *d_init = c.take<int>(N);
    int *d_hard = c.take<int>(N);
    int *d_labels = c.take<int>(N);
    int *d_count = c.take<int>(64);
    Carver hc{static_cast<char *>(C.h_buf)};
    unsigned char *h_ok = hc.take<unsigned char>(N);
    int *h_idx = hc.take<int>(N);
    int32_t *h_init = hc.take<int32_t>(N);
    int *h_count = hc.take<int>(16);
    double *h_Z = hc.take<double>(N > 1 ? (N - 1) * 4 : 4);

    FA_CUDA_TRY(cudaEventRecord(C.ev[0], s));
    FA_CUDA_TRY(cudaMemcpyAsync(d_emb32, emb, N * E * sizeof(float), cudaMemcpyHostToDevice, s));
    FA_CUDA_TRY(cudaMemcpyAsync(d_rho, rho, N * R * sizeof(double), cudaMemcpyHostToDevice, s));
    st = ahc::launch_widen_rows(d_emb32, d_emb, (long long)N * E, s);   // :286  Float -> Double
    if (st != FA_OK) return st;
    st = vbx::finite_rows_device(d_emb32, n, e, d_ok, s);               // :591-611
    if (st != FA_OK) return st;
    g_launches += 2;
    FA_CUDA_TRY(cudaMemcpyAsync(h_ok, d_ok, N, cudaMemcpyDeviceToHost, s));
    FA_CUDA_TRY(cudaStreamSynchronize(s));
    int Tn = 0;
    for (int i = 0; i < n; ++i)
        if (h_ok[i]) h_idx[Tn++] = i;
    if (Tn == 0) {
        for (int i = 0; i < n; ++i) h_idx[i] = i;
        Tn = n;
    }
    const double *d_tr = d_emb, *d_tr_rho = d_rho;
    if (Tn != n) {
        FA_CUDA_TRY(cudaMemcpyAsync(d_idx, h_idx, Tn * sizeof(int), cudaMemcpyHostToDevice, s));
        st = vbx::gather_rows_device(d_emb, d_idx, Tn, e, d_train, s);
        if (st != FA_OK) return st;
        st = vbx::gather_rows_device(d_rho, d_idx, Tn, r, d_train_rho, s);
        if (st != FA_OK) return st;
        g_launches += 2;
        d_tr = d_train;
        d_tr_rho = d_train_rho;
    }
    // ---- AHC (:301-309) ---------------------------------------------------------------------------------
    FA_CUDA_TRY(cudaEventRecord(C.ev[1], s));
    float ms_norm = 0, ms_ahc = 0, ms_cut = 0;
    if (Tn >= 2) {
        st = ahc::launch_normalize_rows(d_tr, d_norm, Tn, e, s);
        if (st != FA_OK) return st;
        g_launches += 1;
        FA_CUDA_TRY(cudaEventRecord(C.ev[2], s));
        const long long before = C.solver.launches;
        st = C.solver.linkage_device(d_norm, Tn, e, h_Z);
        g_launches += C.solver.launches - before;
        FA_CUDA_TRY(cudaEventRecord(C.ev[3], s));
        FA_CUDA_TRY(cudaEventSynchronize(C.ev[3]));
        ms_norm = ms_between(C.ev[1], C.ev[2]);
        ms_ahc = ms_between(C.ev[2], C.ev[3]);
        const auto t0 = std::chrono::steady_clock::now();
        if (st == FA_OK) {
            ahc::dendrogram_cut(h_Z, Tn, cfg.threshold, h_init);
        } else if (st == FA_RUNTIME_ERROR || st == FA_UNSUPPORTED) {
            for (int i = 0; i < Tn; ++i) h_init[i] = i;   // AHCClustering.swift:52-55: FFI failure -> identity labels
        } else {
            return st;
        }
        ms_cut = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    } else {
        for (int i = 0; i < Tn; ++i) h_init[i] = 0;
    }
    int S = 0;
    for (int i = 0; i < Tn; ++i) S = std::max(S, h_init[i] + 1);   // labels are canonical 0..S-1
    S = std::max(S, 1);
    if (initial_out) {
        for (int i = 0; i < n; ++i) initial_out[i] = -1;
        for (int i = 0; i < Tn; ++i) initial_out[h_idx[i]] = h_init[i];
    }
    // ---- VBx (:311-343) -----------------------------------------------------------------------------------
    FA_CUDA_TRY(cudaEventRecord(C.ev[4], s));
    FA_CUDA_TRY(cudaMemcpyAsync(d_init, h_init, Tn * sizeof(int), cudaMemcpyHostToDevice, s));
    // arena for gamma / pi / elbos / centroids (depends on S, known only now)
    vbx::Config vc;
    vc.Fa = cfg.vbx.Fa;
    vc.Fb = cfg.vbx.Fb;
    vc.max_iterations = cfg.vbx.max_iterations;
    vc.epsilon = cfg.vbx.epsilon;
    vc.init_smoothing = cfg.vbx.init_smoothing;
    const size_t gbytes = ((size_t)Tn * S + 2 * (size_t)S + std::max(vc.max_iterations, 1) + 2 * ((size_t)S * E + E)) *
                              sizeof(double) + 8192;
    st = C.cent_ws.reserve(std::max(gbytes, (size_t)1 << 20));
    if (st != FA_OK) return st;
    Carver gc{static_cast<char *>(C.cent_ws.pool)};
    double *d_gamma = gc.take<double>((size_t)Tn * S);
    double *d_pi = gc.take<double>(S);
    double *d_elbos = gc.take<double>(std::max(vc.max_iterations, 1));
    double *d_cent = gc.take<double>((size_t)S * E + E);
    double *d_cent_n = gc.take<double>((size_t)S * E + E);
    int iterations = 0;
    std::vector<double> psi_eff(R, 1.0);   // VBxClustering.swift:71-76: identity when psi does not match
    if (psi) std::memcpy(psi_eff.data(), psi, R * sizeof(double));
    bool used_vbx = false;
    long long lc = 0;
    if (Tn > 0) {
        st = vbx::refine_device(C.vbx_ws, d_tr_rho, Tn, r, psi_eff.data(), d_init, S, vc, d_gamma, d_pi, d_elbos, d_hard,
                                &iterations, s, &lc);
        if (st != FA_OK) return st;
        used_vbx = true;
    }
    // ---- speaker-count constraints (:311-336, VBxClustering.swift:685-733) ----------------------------------
    bool adjusted = false;
    int detected = S, K = 0;
    if (used_vbx && (cfg.num_speakers != FA_NO_VALUE || cfg.min_speakers != FA_NO_VALUE || cfg.max_speakers != FA_NO_VALUE)) {
        std::vector<int> hard(Tn);
        FA_CUDA_TRY(cudaMemcpyAsync(hard.data(), d_hard, sizeof(int) * Tn, cudaMemcpyDeviceToHost, s));
        FA_CUDA_TRY(cudaStreamSynchronize(s));
        std::vector<char> seen(S, 0);
        detected = 0;                                       // VBxOutput.assignedClusterCount: row-argmax winners
        for (int i = 0; i < Tn; ++i)
            if (hard[i] >= 0 && hard[i] < S && !seen[hard[i]]) {
                seen[hard[i]] = 1;
                ++detected;
            }
        long long lo = 1, hi = Tn;
        kmeans::resolve_constraints(Tn, cfg.num_speakers, cfg.min_speakers, cfg.max_speakers, &lo, &hi);
        if (detected < lo || detected > hi) {
            const int target = (int)(detected < lo ? lo : hi);
            st = C.cent_ws.reserve(std::max(C.cent_ws.pool_bytes, gbytes + 2 * (size_t)target * E * sizeof(double)));
            if (st != FA_OK) return st;
            // the arena may have moved: re-carve (gamma / pi are not needed any more on this path)
            Carver kc{static_cast<char *>(C.cent_ws.pool)};
            d_cent = kc.take<double>((size_t)target * E + E);
            d_cent_n = kc.take<double>((size_t)target * E + E);
            int rows = 0;
            st = kmeans::cluster_ninit_device(C.vbx_ws, d_tr, Tn, e, target, 100, 10, 0ull, d_hard, d_cent, &rows, nullptr,
                                              s, &lc);
            if (st != FA_OK) return st;
            st = ahc::launch_normalize_rows_keep(d_cent, d_cent_n, rows, e, s);   // normalize (:824-860) for the cosine
            if (st != FA_OK) return st;
            lc += 1;
            K = rows;
            adjusted = true;
        }
    }
    FA_CUDA_TRY(cudaEventRecord(C.ev[5], s));
    // ---- centroids (:345-353) + assignment (:371-374) -----------------------------------------------------
    if (!adjusted) {
        st = vbx::centroids_device(C.vbx_ws, d_tr, Tn, e, d_gamma, d_pi, S, d_cent, d_cent_n, d_count, s, &lc);
        if (st != FA_OK) return st;
        FA_CUDA_TRY(cudaMemcpyAsync(h_count, d_count, sizeof(int), cudaMemcpyDeviceToHost, s));
        FA_CUDA_TRY(cudaStreamSynchronize(s));
        K = *h_count;
        if (K == 0 && used_vbx) {
            // no speaker with pi > 1e-7: computeCentroidsFromClusters(initialClusters) (:687-690)
            st = vbx::onehot_device(d_init, Tn, S, d_gamma, d_pi, s);
            if (st != FA_OK) return st;
            st = vbx::centroids_device(C.vbx_ws, d_tr, Tn, e, d_gamma, d_pi, S, d_cent, d_cent_n, d_count, s, &lc);
            if (st != FA_OK) return st;
            lc += 1;
            FA_CUDA_TRY(cudaMemcpyAsync(h_count, d_count, sizeof(int), cudaMemcpyDeviceToHost, s));
            FA_CUDA_TRY(cudaStreamSynchronize(s));
            K = *h_count;
        }
    }
    if (K == 0) {
        // computeFallbackCentroids: mean of all embeddings (:748-786)
        st = vbx::mean_rows_device(d_emb, n, e, d_cent, s);
        if (st != FA_OK) return st;
        st = vbx::onehot_device(d_init, 0, 1, d_gamma, d_pi, s);   // pi[0] = 1
        if (st != FA_OK) return st;
        // OfflineDiarizerManager.normalize on the one centroid (:824-860: a zero row is kept)
        st = ahc::launch_normalize_rows_keep(d_cent, d_cent_n, 1, e, s);
        if (st != FA_OK) return st;
        ++lc;
        K = 1;
        lc += 2;
    }
    // constrained assignment (:357-369) needs the full N x K score matrix on the host; plain argmax (:371-374) does not
    const bool constrained = chunk_index != nullptr && K > 1 && !adjusted;   // :357-360
    double *d_scores = nullptr;
    if (constrained) {
        st = C.vbx_ws.reserve(std::max(C.vbx_ws.pool_bytes, N * (size_t)K * sizeof(double) + 1024));
        if (st != FA_OK) return st;
        d_scores = static_cast<double *>(C.vbx_ws.pool);
    }
    st = vbx::assign_device(d_emb, n, e, d_cent_n, nullptr, K, d_labels, d_scores, s, &lc);
    if (st != FA_OK) return st;
    g_launches += lc;
    if (constrained) {
        std::vector<double> h_scores(N * (size_t)K);
        FA_CUDA_TRY(cudaMemcpyAsync(h_scores.data(), d_scores, h_scores.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
        FA_CUDA_TRY(cudaStreamSynchronize(s));
        assign::constrained_assign(h_scores.data(), (long long)N, K, chunk_index, labels);
    } else {
        FA_CUDA_TRY(cudaMemcpyAsync(labels, d_labels, N * sizeof(int), cudaMemcpyDeviceToHost, s));
    }
    if (centroids_out && max_centroids > 0) {
        const int kc = std::min(K, max_centroids);
        FA_CUDA_TRY(cudaMemcpyAsync(centroids_out, d_cent, (size_t)kc * E * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    FA_CUDA_TRY(cudaEventRecord(C.ev[6], s));
    // VBxOutput.assignedClusterCount for the caller's info when no speaker-count constraint asked for it above: the
    // row-argmax winners travel with the final synchronisation
    std::vector<int> hard_info;
    const bool count_winners = info && used_vbx && !adjusted && detected == S && Tn > 0 &&
                               cfg.num_speakers == FA_NO_VALUE && cfg.min_speakers == FA_NO_VALUE && cfg.max_speakers == FA_NO_VALUE;
    if (count_winners) {
        hard_info.resize(Tn);
        FA_CUDA_TRY(cudaMemcpyAsync(hard_info.data(), d_hard, sizeof(int) * Tn, cudaMemcpyDeviceToHost, s));
    }
    FA_CUDA_TRY(cudaStreamSynchronize(s));
    if (count_winners) {
        std::vector<char> seen(S, 0);
        detected = 0;
        for (int i = 0; i < Tn; ++i)
            if (hard_info[i] >= 0 && hard_info[i] < S && !seen[hard_info[i]]) {
                seen[hard_info[i]] = 1;
                ++detected;
            }
    }
    if (info) {
        info->training_count = Tn;
        info->initial_clusters = S;
        info->vbx_iterations = iterations;
        info->centroid_count = K;
        info->ms_normalize = ms_norm;
        info->ms_ahc = ms_ahc;
        info->ms_cut = ms_cut;
        info->ms_vbx = ms_between(C.ev[4], C.ev[5]);
        info->ms_assign = ms_between(C.ev[5], C.ev[6]);
        info->ms_total =
            std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - wall0).count();
        info->was_adjusted = adjusted ? 1 : 0;
        info->detected_clusters = detected;
    }
    return FA_OK;
}

// timer state for fa_timer_*
static thread_local cudaEvent_t t_ev0 = nullptr, t_ev1 = nullptr;

struct MelHandle {
    mel::MelPlan plan;
    int device = 0;
};

} // namespace fa

using namespace fa;

#define FA_GUARD_BEGIN try {
#define FA_GUARD_END                                              \
    }                                                             \
    catch (const std::bad_alloc &) {                              \
        fa::set_error("host allocation failed");                  \
        return (fa_status)FA_ALLOCATION_FAILURE;                  \
    }                                                             \
    catch (const std::exception &ex) {                            \
        fa::set_error("exception: %s", ex.what());                \
        return (fa_status)FA_RUNTIME_ERROR;                       \
    }                                                             \
    catch (...) {                                                 \
        fa::set_error("unknown exception");                       \
        return (fa_status)FA_UNKNOWN_ERROR;                       \
    }

// ------------------------------------------------------------------------------------------------ runtime
FA_API const char *fa_version(void) { return "fluidaudio_b200 0.1.0 (sm_100a)"; }
FA_API const char *fa_last_error(void) { return fa::last_error(); }
FA_API int32_t fa_device_count(void) { return usable_device_count(); }

#define API_CUDA_TRY(expr)                                                                              \
    do {                                                                                                \
        cudaError_t e__ = (expr);                                                                       \
        if (e__ != cudaSuccess) {                                                                       \
            fa::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return e__ == cudaErrorMemoryAllocation ? FA_STATUS_ALLOCATION_FAILURE : FA_STATUS_CUDA_ERROR; \
        }                                                                                               \
    } while (0)
#define API_REQUIRE_DEVICE()                                       \
    do {                                                           \
        if (require_device() != FA_OK) return FA_STATUS_NO_DEVICE; \
    } while (0)

FA_API fa_status fa_set_device(int32_t ordinal) {
    API_REQUIRE_DEVICE();
    API_CUDA_TRY(cudaSetDevice(ordinal));
    return FA_STATUS_OK;
}

FA_API fa_status fa_device_synchronize(void) {
    API_REQUIRE_DEVICE();
    API_CUDA_TRY(cudaDeviceSynchronize());
    return FA_STATUS_OK;
}

FA_API int64_t fa_kernel_launch_count(void) { return g_launches.load(); }

FA_API fa_status fa_host_alloc(size_t bytes, void **out) {
    if (!out) return FA_STATUS_INVALID_ARGUMENT;
    API_REQUIRE_DEVICE();
    API_CUDA_TRY(cudaMallocHost(out, bytes ? bytes : 1));
    return FA_STATUS_OK;
}
FA_API fa_status fa_host_free(void *p) {
    if (p) API_CUDA_TRY(cudaFreeHost(p));
    return FA_STATUS_OK;
}
FA_API fa_status fa_device_alloc(size_t bytes, void **out) {
    if (!out) return FA_STATUS_INVALID_ARGUMENT;
    API_REQUIRE_DEVICE();
    API_CUDA_TRY(cudaMalloc(out, bytes ? bytes : 1));
    return FA_STATUS_OK;
}
FA_API fa_status fa_device_free(void *p) {
    if (p) API_CUDA_TRY(cudaFree(p));
    return FA_STATUS_OK;
}
FA_API fa_status fa_memcpy_h2d(void *dst, const void *src, size_t bytes) {
    API_REQUIRE_DEVICE();
    API_CUDA_TRY(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    return FA_STATUS_OK;
}
FA_API fa_status fa_memcpy_d2h(void *dst, const void *src, size_t bytes) {
    API_REQUIRE_DEVICE();
    API_CUDA_TRY(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return FA_STATUS_OK;
}

// Bare copy-engine probe: `reps` rounds of an H2D copy of h2d_bytes and a D2H copy of d2h_bytes issued together on two
// streams (device scratch allocated here), wall-clock per round.  bench.py uses it to name the floor under every
// host-buffer (end-to-end) number: what the PCIe / host-memory path delivers with no kernel in the way.
FA_API fa_status fa_memcpy_probe(const void *host_src, size_t h2d_bytes, void *host_dst, size_t d2h_bytes, int32_t reps,
                                 float *ms_per_round) {
    if (!ms_per_round || reps < 1 || (!host_src && h2d_bytes) || (!host_dst && d2h_bytes)) return FA_STATUS_INVALID_ARGUMENT;
    API_REQUIRE_DEVICE();
    struct R {
        void *a = nullptr, *b = nullptr;
        cudaStream_t s[2] = {nullptr, nullptr};
        ~R() {
            if (a) cudaFree(a);
            if (b) cudaFree(b);
            for (auto x : s)
                if (x) cudaStreamDestroy(x);
        }
    } r;
    API_CUDA_TRY(cudaMalloc(&r.a, h2d_bytes + 16));
    API_CUDA_TRY(cudaMalloc(&r.b, d2h_bytes + 16));
    API_CUDA_TRY(cudaMemset(r.b, 0, d2h_bytes + 16));
    for (auto &x : r.s) API_CUDA_TRY(cudaStreamCreateWithFlags(&x, cudaStreamNonBlocking));
    API_CUDA_TRY(cudaDeviceSynchronize());
    const auto t0 = std::chrono::steady_clock::now();
    for (int i = 0; i < reps; ++i) {
        if (h2d_bytes) API_CUDA_TRY(cudaMemcpyAsync(r.a, host_src, h2d_bytes, cudaMemcpyHostToDevice, r.s[0]));
        if (d2h_bytes) API_CUDA_TRY(cudaMemcpyAsync(host_dst, r.b, d2h_bytes, cudaMemcpyDeviceToHost, r.s[1]));
        API_CUDA_TRY(cudaStreamSynchronize(r.s[0]));
        API_CUDA_TRY(cudaStreamSynchronize(r.s[1]));
    }
    const auto t1 = std::chrono::steady_clock::now();
    *ms_per_round = (float)(std::chrono::duration<double, std::milli>(t1 - t0).count() / reps);
    return FA_STATUS_OK;
}

// Events on the legacy default stream order against every blocking stream AND, because the library's own streams
// are non-blocking, the timed entry points synchronise their streams before returning (device-side async calls
// are timed by the caller bracketing fa_device_synchronize()).
FA_API fa_status fa_timer_start(void) {
    API_REQUIRE_DEVICE();
    if (!t_ev0) {
        API_CUDA_TRY(cudaEventCreate(&t_ev0));
        API_CUDA_TRY(cudaEventCreate(&t_ev1));
    }
    API_CUDA_TRY(cudaDeviceSynchronize());
    API_CUDA_TRY(cudaEventRecord(t_ev0, 0));
    return FA_STATUS_OK;
}
FA_API fa_status fa_timer_stop_ms(float *elapsed_ms) {
    if (!elapsed_ms || !t_ev0) return FA_STATUS_INVALID_ARGUMENT;
    API_CUDA_TRY(cudaDeviceSynchronize());
    API_CUDA_TRY(cudaEventRecord(t_ev1, 0));
    API_CUDA_TRY(cudaEventSynchronize(t_ev1));
    API_CUDA_TRY(cudaEventElapsedTime(elapsed_ms, t_ev0, t_ev1));
    return FA_STATUS_OK;
}

// ------------------------------------------------------------------------------------------------ mel
FA_API void fa_mel_default_config(fa_mel_config *cfg) {
    if (!cfg) return;
    cfg->sample_rate = 16000;
    cfg->n_mels = 128;
    cfg->n_fft = 512;
    cfg->hop_length = 160;
    cfg->win_length = 400;
    cfg->preemph = 0.97f;
    cfg->pad_to = 0;
    cfg->log_floor = ldexpf(1.0f, -24);
    cfg->log_floor_mode = 0;
    cfg->window_periodic = 0;
}

FA_API fa_status fa_mel_create(const fa_mel_config *cfg, fa_mel **out) {
    if (!cfg || !out) return FA_STATUS_INVALID_ARGUMENT;
    *out = nullptr;
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    std::unique_ptr<MelHandle> h(new MelHandle());
    mel::MelConfig c{cfg->sample_rate, cfg->n_mels, cfg->n_fft, cfg->hop_length, cfg->win_length, cfg->preemph,
                     cfg->pad_to, cfg->log_floor, cfg->log_floor_mode, cfg->window_periodic};
    API_CUDA_TRY(cudaGetDevice(&h->device));
    const int st = h->plan.init(c);
    if (st != FA_OK) return (fa_status)st;
    *out = reinterpret_cast<fa_mel *>(h.release());
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API void fa_mel_destroy(fa_mel *mel) { delete reinterpret_cast<MelHandle *>(mel); }

FA_API fa_status fa_mel_get_window(const fa_mel *mel, float *out, size_t len) {
    if (!mel || !out) return FA_STATUS_INVALID_ARGUMENT;
    const auto &w = reinterpret_cast<const MelHandle *>(mel)->plan.window;
    if (len < w.size()) return FA_STATUS_OUTPUT_TOO_SMALL;
    std::memcpy(out, w.data(), w.size() * sizeof(float));
    return FA_STATUS_OK;
}

FA_API fa_status fa_mel_get_filterbank(const fa_mel *mel, float *out, size_t len) {
    if (!mel || !out) return FA_STATUS_INVALID_ARGUMENT;
    const auto &f = reinterpret_cast<const MelHandle *>(mel)->plan.filterbank;
    if (len < f.size()) return FA_STATUS_OUTPUT_TOO_SMALL;
    std::memcpy(out, f.data(), f.size() * sizeof(float));
    return FA_STATUS_OK;
}

FA_API int64_t fa_mel_frame_count(const fa_mel *mel, int64_t n, int32_t padding_mode, int64_t expected) {
    if (!mel) return -1;
    return reinterpret_cast<const MelHandle *>(mel)->plan.frame_count(n, padding_mode, expected);
}

FA_API fa_status fa_mel_set_precision(fa_mel *mel, int32_t precision) {
    if (!mel || (precision != FA_MEL_PRECISION_F64 && precision != FA_MEL_PRECISION_F32)) {
        fa::set_error("precision must be FA_MEL_PRECISION_F64 (0) or FA_MEL_PRECISION_F32 (1)");
        return FA_STATUS_INVALID_ARGUMENT;
    }
    reinterpret_cast<MelHandle *>(mel)->plan.precision = precision;
    return FA_STATUS_OK;
}
FA_API fa_status fa_mel_set_pipeline_chunks(fa_mel *mel, int32_t chunks) {
    if (!mel || chunks < 1 || chunks > 1024) return FA_STATUS_INVALID_ARGUMENT;
    reinterpret_cast<MelHandle *>(mel)->plan.pipeline_chunks = chunks;
    return FA_STATUS_OK;
}
FA_API fa_status fa_mel_set_zero_copy_output(fa_mel *mel, int32_t enabled) {
    if (!mel) return FA_STATUS_INVALID_ARGUMENT;
    reinterpret_cast<MelHandle *>(mel)->plan.zero_copy_out = enabled != 0;
    return FA_STATUS_OK;
}
FA_API int32_t fa_mel_get_precision(const fa_mel *mel) {
    return mel ? reinterpret_cast<const MelHandle *>(mel)->plan.precision : -1;
}

static bool mel_args_ok(int32_t mode, int32_t layout) {
    if (mode < 0 || mode > 2 || layout < 0 || layout > 1) {
        fa::set_error("padding_mode must be 0..2 and layout 0..1");
        return false;
    }
    return true;
}

FA_API fa_status fa_mel_compute(fa_mel *mel, const float *audio, size_t n, float last, int32_t mode, int64_t expected,
                                int32_t layout, float *out, size_t out_len, int64_t *mel_length, int64_t *num_frames) {
    if (!mel || !out || (!audio && n) || !mel_args_ok(mode, layout)) return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    auto *h = reinterpret_cast<MelHandle *>(mel);
    long long ml = 0, nf = 0;
    const long long before = h->plan.launches;
    const int st = h->plan.compute_host(audio, (long long)n, last, mode, expected, layout, out, (long long)out_len, &ml, &nf);
    g_launches += h->plan.launches - before;
    if (mel_length) *mel_length = ml;
    if (num_frames) *num_frames = nf;
    return (fa_status)st;
    FA_GUARD_END
}

FA_API fa_status fa_mel_compute_device(fa_mel *mel, const float *d_audio, size_t n, float last, int32_t mode,
                                       int64_t expected, int32_t layout, float *d_out, size_t out_len,
                                       int64_t *mel_length, int64_t *num_frames) {
    if (!mel || !d_out || (!d_audio && n) || !mel_args_ok(mode, layout)) return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    auto *h = reinterpret_cast<MelHandle *>(mel);
    long long ml = 0, nf = 0;
    const long long before = h->plan.launches;
    const int st = h->plan.compute_device(d_audio, (long long)n, last, mode, expected, layout, d_out, (long long)out_len,
                                          &ml, &nf, h->plan.streams[1]);
    g_launches += h->plan.launches - before;
    if (mel_length) *mel_length = ml;
    if (num_frames) *num_frames = nf;
    return (fa_status)st;
    FA_GUARD_END
}

FA_API fa_status fa_mel_compute_batch(fa_mel *mel, const float *audio, const int64_t *offsets, int32_t count,
                                      const float *last, int32_t mode, int32_t layout, float *out,
                                      const int64_t *out_offsets, int64_t *mel_lengths, int64_t *num_frames) {
    if (!mel || !audio || !offsets || !out || !out_offsets || count < 0 || !mel_args_ok(mode, layout))
        return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    auto *h = reinterpret_cast<MelHandle *>(mel);
    const long long before = h->plan.launches;
    static_assert(sizeof(long long) == sizeof(int64_t), "int64 layout");
    const int st = h->plan.compute_batch_host(audio, reinterpret_cast<const long long *>(offsets), count, last, mode, layout,
                                              out, reinterpret_cast<const long long *>(out_offsets),
                                              reinterpret_cast<long long *>(mel_lengths),
                                              reinterpret_cast<long long *>(num_frames));
    g_launches += h->plan.launches - before;
    return (fa_status)st;
    FA_GUARD_END
}

FA_API fa_status fa_mel_compute_batch_device(fa_mel *mel, const float *d_audio, const int64_t *offsets, int32_t count,
                                             const float *last, int32_t mode, int32_t layout, float *d_out,
                                             const int64_t *out_offsets, int64_t *mel_lengths, int64_t *num_frames) {
    if (!mel || !d_audio || !offsets || !d_out || !out_offsets || count < 0 || !mel_args_ok(mode, layout))
        return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    auto *h = reinterpret_cast<MelHandle *>(mel);
    const long long before = h->plan.launches;
    const int st = h->plan.compute_batch_device(d_audio, reinterpret_cast<const long long *>(offsets), count, last, mode,
                                                layout, d_out, reinterpret_cast<const long long *>(out_offsets),
                                                reinterpret_cast<long long *>(mel_lengths),
                                                reinterpret_cast<long long *>(num_frames), h->plan.streams[1]);
    g_launches += h->plan.launches - before;
    return (fa_status)st;
    FA_GUARD_END
}

// CUDA-event timing on the stream the mel kernels are launched on (device-resident entry points are asynchronous).
FA_API fa_status fa_mel_timer_start(fa_mel *mel) {
    if (!mel) return FA_STATUS_INVALID_ARGUMENT;
    auto *h = reinterpret_cast<MelHandle *>(mel);
    if (!h->plan.timer[0]) {
        API_CUDA_TRY(cudaEventCreate(&h->plan.timer[0]));
        API_CUDA_TRY(cudaEventCreate(&h->plan.timer[1]));
    }
    API_CUDA_TRY(cudaStreamSynchronize(h->plan.streams[1]));
    API_CUDA_TRY(cudaEventRecord(h->plan.timer[0], h->plan.streams[1]));
    return FA_STATUS_OK;
}
FA_API fa_status fa_mel_timer_stop_ms(fa_mel *mel, float *elapsed_ms) {
    if (!mel || !elapsed_ms) return FA_STATUS_INVALID_ARGUMENT;
    auto *h = reinterpret_cast<MelHandle *>(mel);
    if (!h->plan.timer[0]) return FA_STATUS_INVALID_ARGUMENT;
    API_CUDA_TRY(cudaEventRecord(h->plan.timer[1], h->plan.streams[1]));
    API_CUDA_TRY(cudaEventSynchronize(h->plan.timer[1]));
    API_CUDA_TRY(cudaEventElapsedTime(elapsed_ms, h->plan.timer[0], h->plan.timer[1]));
    return FA_STATUS_OK;
}

// UnifiedMelExtractor.features(window:validCount:) (UnifiedMelExtractor.swift:52-86): log-mel + per-feature
// normalisation + [1, nMels, T] packing, normalisation and packing as a device epilogue of the mel kernel.
FA_API fa_status fa_mel_unified_features(fa_mel *mel, const float *window, size_t window_samples, size_t valid_count,
                                         float *out, size_t out_len, int64_t *total_frames, int32_t *valid_frames) {
    if (!mel || !out || (!window && window_samples)) return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    auto *h = reinterpret_cast<MelHandle *>(mel);
    const long long before = h->plan.launches;
    long long T = 0;
    int valid = 0;
    const int st = fa::mel::unified_features(h->plan, window, (long long)window_samples, (long long)valid_count, out,
                                             (long long)out_len, &T, &valid);
    g_launches += h->plan.launches - before;
    if (total_frames) *total_frames = T;
    if (valid_frames) *valid_frames = valid;
    return (fa_status)st;
    FA_GUARD_END
}

// LSEENDPreprocessor.processAudioQueue (LSEENDPreprocessor.swift:249-283): .prePadded log-mel of one audio chunk,
// log10 scaling and cumulative mean normalisation; (cmn_mean, cmn_count) is the preprocessor's running state.
FA_API fa_status fa_mel_lseend_features(fa_mel *mel, const float *chunk, size_t n, float *cmn_mean, int64_t *cmn_count,
                                        float *out, size_t out_len, int64_t *frames) {
    if (!mel || !cmn_mean || !cmn_count || *cmn_count < 0 || (!chunk && n) || (!out && out_len))
        return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    auto *h = reinterpret_cast<MelHandle *>(mel);
    const long long before = h->plan.launches;
    long long T = 0, count = *cmn_count;
    const int st = fa::mel::lseend_features(h->plan, chunk, (long long)n, cmn_mean, &count, out, (long long)out_len, &T);
    g_launches += h->plan.launches - before;
    *cmn_count = count;
    if (frames) *frames = T;
    return (fa_status)st;
    FA_GUARD_END
}

// UnifiedMelExtractor.normalizePerFeature (UnifiedMelExtractor.swift:88-113).  O(T*M) on a caller-owned host
// buffer that is about to be handed to the encoder; not a GPU hot path.
FA_API fa_status fa_mel_normalize_per_feature(float *x, int64_t frames, int32_t n_mels, int64_t valid) {
    if (!x || frames < 0 || n_mels <= 0) return FA_STATUS_INVALID_ARGUMENT;
    if (valid > frames) valid = frames;   // UnifiedMelExtractor.swift:66: validFrames = min(validCount / hop, totalFrames)
    if (frames == 0) return FA_STATUS_OK;
    if (valid <= 0) {                     // no valid frame: everything is padding
        std::memset(x, 0, sizeof(float) * (size_t)frames * n_mels);
        return FA_STATUS_OK;
    }
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    const int st = mel::normalize_per_feature_host(x, (long long)frames, n_mels, (long long)valid);
    if (st == FA_OK) ++g_launches;
    return (fa_status)st;
    FA_GUARD_END
}

// ------------------------------------------------------------------------------------------------ AudioConverter stage
static bool audio_format_ok(const fa_audio_format *f) {
    if (!f || !(f->in_rate > 0) || !(f->out_rate > 0) || f->channels < 1 || f->channels > 64 ||
        (f->format != FA_PCM_F32 && f->format != FA_PCM_I16) || f->algorithm < 0 || f->algorithm > 2) {
        fa::set_error("audio format: rates must be positive, 1..64 channels, format F32/I16, algorithm 0..2");
        return false;
    }
    return true;
}
static resample::AudioFormat to_format(const fa_audio_format *f) {
    return resample::AudioFormat{f->in_rate, f->out_rate, f->channels, f->format, f->interleaved ? 1 : 0, f->algorithm};
}

FA_API int64_t fa_resample_output_count(const fa_audio_format *fmt, int64_t frames) {
    if (!fmt || frames < 0 || !(fmt->in_rate > 0) || !(fmt->out_rate > 0)) return -1;
    return resample::output_count(frames, fmt->in_rate, fmt->out_rate);
}

FA_API fa_status fa_audio_resample(const void *pcm, int64_t frames, const fa_audio_format *fmt, float *out,
                                   int64_t out_cap, int64_t *out_count) {
    if (!audio_format_ok(fmt) || frames < 0 || !out_count) return FA_STATUS_INVALID_ARGUMENT;
    const long long n = resample::output_count(frames, fmt->in_rate, fmt->out_rate);
    *out_count = n;
    if (!out) return FA_STATUS_OK;            // sizing call: pcm may be NULL
    if (!pcm && frames) {
        fa::set_error("fa_audio_resample: pcm is NULL");
        return FA_STATUS_INVALID_ARGUMENT;
    }
    if (out_cap < n) return FA_STATUS_OUTPUT_TOO_SMALL;
    if (n == 0) return FA_STATUS_OK;
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    const resample::AudioFormat f = to_format(fmt);
    resample::Design d;
    if (f.in_rate != f.out_rate) {
        const int st = resample::make_design(f.in_rate, f.out_rate, d);
        if (st != FA_OK) return (fa_status)st;
    }
    const size_t bytes = (size_t)frames * f.channels * (f.format == resample::kPcmI16 ? 2 : 4);
    struct Bufs {
        void *pcm = nullptr;
        float *tab = nullptr, *out = nullptr;
        cudaStream_t s = nullptr;
        ~Bufs() {
            if (pcm) cudaFree(pcm);
            if (tab) cudaFree(tab);
            if (out) cudaFree(out);
            if (s) cudaStreamDestroy(s);
        }
    } b;
    API_CUDA_TRY(cudaStreamCreateWithFlags(&b.s, cudaStreamNonBlocking));
    API_CUDA_TRY(cudaMalloc(&b.pcm, bytes + 16));
    API_CUDA_TRY(cudaMalloc(&b.out, (size_t)n * sizeof(float)));
    if (!d.table.empty()) {
        API_CUDA_TRY(cudaMalloc(&b.tab, d.table.size() * sizeof(float)));
        API_CUDA_TRY(cudaMemcpyAsync(b.tab, d.table.data(), d.table.size() * sizeof(float), cudaMemcpyHostToDevice, b.s));
    }
    API_CUDA_TRY(cudaMemcpyAsync(b.pcm, pcm, bytes, cudaMemcpyHostToDevice, b.s));
    long long launches = 0;
    const int st = resample::launch_convert(b.pcm, frames, f, d, b.tab, b.out, 0, n, b.s, &launches);
    g_launches += launches;
    if (st != FA_OK) return (fa_status)st;
    API_CUDA_TRY(cudaMemcpyAsync(out, b.out, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, b.s));
    API_CUDA_TRY(cudaStreamSynchronize(b.s));
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_audio_to_mel(fa_mel *mel, const void *pcm, int64_t frames, const fa_audio_format *fmt, float last,
                                 int32_t mode, int32_t layout, float *out, size_t out_len, int64_t *mel_length,
                                 int64_t *num_frames, int64_t *resampled_count) {
    if (!mel || !out || frames < 0 || (!pcm && frames) || !audio_format_ok(fmt) || !mel_args_ok(mode, layout))
        return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    auto *h = reinterpret_cast<MelHandle *>(mel);
    if (fmt->out_rate != (double)h->plan.cfg.sample_rate) {
        fa::set_error("fa_audio_to_mel: out_rate %.3f differs from the handle's sample_rate %d", fmt->out_rate,
                      h->plan.cfg.sample_rate);
        return FA_STATUS_INVALID_ARGUMENT;
    }
    long long ml = 0, nf = 0, rs = 0;
    const long long before = h->plan.launches;
    const resample::AudioFormat f = to_format(fmt);
    int st;
    if (resample::is_identity(f)) {   // mono float32 at the model rate: AudioConverter returns the samples as they are (:66-68)
        rs = frames;
        st = h->plan.compute_host(static_cast<const float *>(pcm), (long long)frames, last, mode, -1, layout, out,
                                  (long long)out_len, &ml, &nf);
    } else {
        st = h->plan.compute_host_pcm(pcm, (long long)frames, f, last, mode, layout, out, (long long)out_len, &ml, &nf, &rs);
    }
    g_launches += h->plan.launches - before;
    if (mel_length) *mel_length = ml;
    if (num_frames) *num_frames = nf;
    if (resampled_count) *resampled_count = rs;
    return (fa_status)st;
    FA_GUARD_END
}

// AudioConverter.linearResample (AudioConverter.swift:388-442): boundary glue for >2-channel input.
FA_API fa_status fa_linear_resample(const float *in, int64_t frames, int32_t channels, double in_rate, double out_rate,
                                    float *out, int64_t out_cap, int64_t *out_count) {
    if (frames < 0 || channels <= 0 || !(in_rate > 0) || !(out_rate > 0) || !out_count || (out && !in && frames))
        return FA_STATUS_INVALID_ARGUMENT;
    // planar float32, the two-tap float32 interpolation whatever the channel count: the converter stage's linear kernel
    fa_audio_format fmt{};
    fmt.in_rate = in_rate;
    fmt.out_rate = out_rate;
    fmt.channels = channels;
    fmt.format = FA_PCM_F32;
    fmt.interleaved = 0;
    fmt.algorithm = FA_RESAMPLE_LINEAR;
    return fa_audio_resample(in, frames, &fmt, out, out_cap, out_count);
}

// ------------------------------------------------------------------------------------------------ clustering
static fastcluster_wrapper_status to_fc(int st) {
    switch (st) {
    case FA_OK: return FASTCLUSTER_WRAPPER_SUCCESS;
    case FA_INVALID_ARGUMENT: return FASTCLUSTER_WRAPPER_INVALID_ARGUMENT;
    case FA_INDEX_OVERFLOW: return FASTCLUSTER_WRAPPER_INDEX_OVERFLOW;
    case FA_OUTPUT_TOO_SMALL: return FASTCLUSTER_WRAPPER_OUTPUT_TOO_SMALL;
    case FA_ALLOCATION_FAILURE: return FASTCLUSTER_WRAPPER_ALLOCATION_FAILURE;
    case FA_UNKNOWN_ERROR: return FASTCLUSTER_WRAPPER_UNKNOWN_ERROR;
    default: return FASTCLUSTER_WRAPPER_RUNTIME_ERROR;   // NaN, CUDA failure, no device, unsupported size
    }
}

FA_API fastcluster_wrapper_status fastcluster_compute_centroid_linkage(const double *data, size_t pointCount,
                                                                       size_t dimension, double *dendrogramOut,
                                                                       size_t dendrogramLength) {
    // argument contract first, exactly as FastClusterWrapper.cpp:203-223 (no device needed for these)
    if (data == nullptr || dendrogramOut == nullptr) return FASTCLUSTER_WRAPPER_INVALID_ARGUMENT;
    if (pointCount == 0) return FASTCLUSTER_WRAPPER_SUCCESS;
    if (dimension == 0) return FASTCLUSTER_WRAPPER_INVALID_ARGUMENT;
    if (pointCount > 0x7fffffffull || dimension > 0x7fffffffull) return FASTCLUSTER_WRAPPER_INDEX_OVERFLOW;
    const size_t need = pointCount > 1 ? (pointCount - 1) * 4 : 0;
    if (dendrogramLength < need) return FASTCLUSTER_WRAPPER_OUTPUT_TOO_SMALL;
    if (pointCount == 1) return FASTCLUSTER_WRAPPER_SUCCESS;
    try {
        if (require_device() != FA_OK) return FASTCLUSTER_WRAPPER_RUNTIME_ERROR;
        Lease lease;
        if (lease.status != FA_OK) return to_fc(lease.status);
        const long long before = lease.ctx->solver.launches;
        const int st = lease.ctx->solver.linkage_host(data, pointCount, dimension, dendrogramOut, dendrogramLength);
        g_launches += lease.ctx->solver.launches - before;
        lease.status = st == FA_CUDA_ERROR ? FA_CUDA_ERROR : FA_OK;
        return to_fc(st);
    } catch (const std::bad_alloc &) {
        return FASTCLUSTER_WRAPPER_ALLOCATION_FAILURE;
    } catch (const std::exception &) {
        return FASTCLUSTER_WRAPPER_RUNTIME_ERROR;
    } catch (...) {
        return FASTCLUSTER_WRAPPER_UNKNOWN_ERROR;
    }
}

FA_API void fa_ahc_last_stage_ms(float *out4) {
    if (!out4) return;
    const float *m = ahc::last_stage_ms();
    for (int q = 0; q < 4; ++q) out4[q] = m[q];
}

FA_API void fa_ahc_last_placement(int32_t *out6) {
    if (!out6) return;
    const int *p = ahc::last_placement();
    for (int q = 0; q < 6; ++q) out6[q] = p[q];
}

FA_API fa_status fa_l2_normalize_rows(const double *x, size_t rows, size_t dim, double *out) {
    if (!x || !out) return FA_STATUS_INVALID_ARGUMENT;
    if (rows == 0 || dim == 0) return FA_STATUS_OK;
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    Lease lease;
    if (lease.status != FA_OK) return (fa_status)lease.status;
    ClusterContext &C = *lease.ctx;
    int st = C.reserve(2 * rows * dim * sizeof(double) + 512, 64);
    if (st != FA_OK) return (fa_status)st;
    double *d_in = static_cast<double *>(C.d_buf);
    double *d_out = d_in + rows * dim;
    API_CUDA_TRY(cudaMemcpyAsync(d_in, x, rows * dim * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    st = ahc::launch_normalize_rows(d_in, d_out, (int)rows, (int)dim, C.stream);
    if (st != FA_OK) return (fa_status)st;
    g_launches += 1;
    API_CUDA_TRY(cudaMemcpyAsync(out, d_out, rows * dim * sizeof(double), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaStreamSynchronize(C.stream));
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_dendrogram_cut(const double *Z, size_t count, double threshold, int32_t *labels) {
    if ((!Z && count > 1) || (!labels && count > 0)) return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    ahc::dendrogram_cut(Z, (long long)count, threshold, labels);
    return FA_STATUS_OK;
    FA_GUARD_END
}

// AHCClustering.cluster (AHCClustering.swift:20-67)
FA_API fa_status fa_ahc_cluster(const double *features, size_t count, size_t dim, double threshold, int32_t *labels) {
    if (count == 0) return FA_STATUS_OK;                       // guard count > 0 else []
    if (!labels) return FA_STATUS_INVALID_ARGUMENT;
    if (dim == 0) {                                            // zero-dimension vectors: all cluster 0 (:26-28)
        for (size_t i = 0; i < count; ++i) labels[i] = 0;
        return FA_STATUS_OK;
    }
    if (!features) return FA_STATUS_INVALID_ARGUMENT;
    if (count == 1) {
        labels[0] = 0;
        return FA_STATUS_OK;
    }
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    Lease lease;
    if (lease.status != FA_OK) return (fa_status)lease.status;
    ClusterContext &C = *lease.ctx;
    int st = C.reserve(2 * count * dim * sizeof(double) + 512, (count - 1) * 4 * sizeof(double) + 512);
    if (st != FA_OK) return (fa_status)st;
    double *d_in = static_cast<double *>(C.d_buf);
    double *d_norm = d_in + count * dim;
    double *h_Z = static_cast<double *>(C.h_buf);
    API_CUDA_TRY(cudaMemcpyAsync(d_in, features, count * dim * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    st = ahc::launch_normalize_rows(d_in, d_norm, (int)count, (int)dim, C.stream);
    if (st != FA_OK) return (fa_status)st;
    const long long before = C.solver.launches;
    st = C.solver.linkage_device(d_norm, (int)count, (int)dim, h_Z);
    g_launches += 1 + C.solver.launches - before;
    if (st == FA_RUNTIME_ERROR || st == FA_UNSUPPORTED) {      // FFI failure -> Array(0..<count) (:52-55)
        for (size_t i = 0; i < count; ++i) labels[i] = (int32_t)i;
        return FA_STATUS_OK;
    }
    if (st != FA_OK) return (fa_status)st;
    ahc::dendrogram_cut(h_Z, (long long)count, threshold, labels);
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API void fa_vbx_default_config(fa_vbx_config *cfg) {
    if (!cfg) return;
    cfg->Fa = 0.07;
    cfg->Fb = 0.8;
    cfg->max_iterations = 20;
    cfg->epsilon = 1e-4;
    cfg->init_smoothing = 7.0;
}

FA_API void fa_cluster_default_config(fa_cluster_config *cfg) {
    if (!cfg) return;
    cfg->threshold = 0.6;
    fa_vbx_default_config(&cfg->vbx);
    cfg->num_speakers = cfg->min_speakers = cfg->max_speakers = FA_NO_VALUE;
    cfg->reserved = 0;
}

FA_API void fa_reconstruct_default_config(fa_reconstruct_config *cfg) {
    if (!cfg) return;
    const reconstruct::Config d;
    cfg->frame_duration = d.frame_duration;
    cfg->window_duration = d.window_duration;
    cfg->min_gap_duration = d.min_gap_duration;
    cfg->seg_min_duration_off = d.seg_min_duration_off;
    cfg->seg_min_duration_on = d.seg_min_duration_on;
    cfg->min_segment_duration = d.min_segment_duration;
    cfg->exclusive_segments = d.exclusive_segments ? 1 : 0;
    cfg->reserved = 0;
}

FA_API fa_status fa_build_segments(const float *weights, int32_t num_chunks, int32_t num_frames, int32_t num_speakers,
                                   const double *chunk_offsets, int32_t offsets_count, const int32_t *hard_clusters,
                                   int32_t hard_rows, int32_t centroid_count, const fa_reconstruct_config *cfg,
                                   int32_t *seg_cluster, float *seg_start, float *seg_end, float *seg_quality,
                                   int32_t segment_cap, int32_t *segment_count) {
    if (!cfg || !segment_count || num_speakers < 0 || offsets_count < 0 || hard_rows < 0 || segment_cap < 0 ||
        (num_chunks > 0 && num_frames > 0 && num_speakers > 0 && !weights) || (offsets_count > 0 && !chunk_offsets) ||
        (hard_rows > 0 && !hard_clusters))
        return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    reconstruct::Config c;
    c.frame_duration = cfg->frame_duration;
    c.window_duration = cfg->window_duration;
    c.min_gap_duration = cfg->min_gap_duration;
    c.seg_min_duration_off = cfg->seg_min_duration_off;
    c.seg_min_duration_on = cfg->seg_min_duration_on;
    c.min_segment_duration = cfg->min_segment_duration;
    c.exclusive_segments = cfg->exclusive_segments != 0;
    std::vector<reconstruct::Segment> segs;
    reconstruct::build_segments(weights, num_chunks, num_frames, num_speakers, chunk_offsets, offsets_count, hard_clusters,
                                hard_rows, centroid_count, c, segs);
    *segment_count = (int32_t)segs.size();
    const int32_t n = std::min<int32_t>((int32_t)segs.size(), segment_cap);
    for (int32_t i = 0; i < n; ++i) {
        if (seg_cluster) seg_cluster[i] = segs[i].cluster;
        if (seg_start) seg_start[i] = segs[i].start;
        if (seg_end) seg_end[i] = segs[i].end;
        if (seg_quality) seg_quality[i] = segs[i].quality;
    }
    return (int32_t)segs.size() > segment_cap ? FA_STATUS_OUTPUT_TOO_SMALL : FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_build_speaker_database(const int32_t *seg_cluster, int32_t segment_count, const double *centroids,
                                           int32_t K, int32_t dim, float *database, int32_t *segment_counts) {
    if (segment_count < 0 || K < 0 || dim < 0 || (segment_count > 0 && !seg_cluster) ||
        (K > 0 && (!segment_counts || (dim > 0 && (!centroids || !database)))))
        return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    reconstruct::build_speaker_database(seg_cluster, segment_count, centroids, K, dim, database, segment_counts);
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_speaker_constraints_resolve(int64_t num_embeddings, int64_t num_speakers, int64_t min_speakers,
                                                int64_t max_speakers, int64_t *resolved_min, int64_t *resolved_max) {
    if (!resolved_min || !resolved_max) return FA_STATUS_INVALID_ARGUMENT;
    long long lo = 0, hi = 0;
    kmeans::resolve_constraints(num_embeddings, num_speakers, min_speakers, max_speakers, &lo, &hi);
    *resolved_min = lo;
    *resolved_max = hi;
    return FA_STATUS_OK;
}

FA_API fa_status fa_kmeans_cluster(const double *emb, size_t N, size_t D, int32_t num_clusters, int32_t max_iterations,
                                   int32_t n_init, uint64_t base_seed, int32_t *labels, double *centroids,
                                   int32_t centroid_cap, int32_t *centroid_rows, int32_t *best_init) {
    if (centroid_rows) *centroid_rows = 0;
    if (best_init) *best_init = 0;
    if (N == 0) return FA_STATUS_OK;                                  // :50-52
    if (!emb || !labels || max_iterations < 0) return FA_STATUS_INVALID_ARGUMENT;
    const long long rows_needed = D == 0 || num_clusters <= 0 ? 0 : std::min<long long>(num_clusters, (long long)N);
    if (rows_needed > 0 && (!centroids || centroid_cap < rows_needed)) return FA_STATUS_OUTPUT_TOO_SMALL;
    if (rows_needed == 0) {                                           // :53-58: dimension 0 or k <= 0 -> all zeros
        for (size_t i = 0; i < N; ++i) labels[i] = 0;
        return FA_STATUS_OK;
    }
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    Lease lease;
    if (lease.status != FA_OK) return (fa_status)lease.status;
    ClusterContext &C = *lease.ctx;
    Carver sz{nullptr};
    sz.take<double>(N * D);
    sz.take<double>((size_t)rows_needed * D);
    sz.take<int>(N);
    int st = C.reserve(sz.off + 1024, 64);
    if (st != FA_OK) return (fa_status)st;
    Carver c{static_cast<char *>(C.d_buf)};
    double *d_emb = c.take<double>(N * D);
    double *d_cent = c.take<double>((size_t)rows_needed * D);
    int *d_labels = c.take<int>(N);
    API_CUDA_TRY(cudaMemcpyAsync(d_emb, emb, N * D * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    long long lc = 0;
    int rows = 0, best = 0;
    st = kmeans::cluster_ninit_device(C.vbx_ws, d_emb, (int)N, (int)D, num_clusters, max_iterations, n_init, base_seed,
                                      d_labels, d_cent, &rows, &best, C.stream, &lc);
    g_launches += lc;
    if (st != FA_OK) return (fa_status)st;
    API_CUDA_TRY(cudaMemcpyAsync(labels, d_labels, N * sizeof(int), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaMemcpyAsync(centroids, d_cent, (size_t)rows * D * sizeof(double), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaStreamSynchronize(C.stream));
    if (centroid_rows) *centroid_rows = rows;
    if (best_init) *best_init = best;
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_vbx_refine(const double *rho, size_t T, size_t D, const double *psi, size_t psi_len,
                               const int32_t *initial, int32_t S, const fa_vbx_config *cfg, double *gamma, double *pi,
                               double *elbos, int32_t *hard, int32_t *iterations) {
    if (!rho || !cfg || !gamma || !pi || !elbos || !hard || T == 0 || D == 0 || S <= 0) return FA_STATUS_INVALID_ARGUMENT;
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    Lease lease;
    if (lease.status != FA_OK) return (fa_status)lease.status;
    ClusterContext &C = *lease.ctx;
    const int cap = std::max(cfg->max_iterations, 1);
    Carver sz{nullptr};
    sz.take<double>(T * D);
    sz.take<int>(T);
    sz.take<double>(T * (size_t)S);
    sz.take<double>(S);
    sz.take<double>(cap);
    sz.take<int>(T);
    int st = C.reserve(sz.off + 1024, 64);
    if (st != FA_OK) return (fa_status)st;
    Carver c{static_cast<char *>(C.d_buf)};
    double *d_x = c.take<double>(T * D);
    int *d_init = c.take<int>(T);
    double *d_gamma = c.take<double>(T * (size_t)S);
    double *d_pi = c.take<double>(S);
    double *d_elbos = c.take<double>(cap);
    int *d_hard = c.take<int>(T);
    std::vector<double> psi_eff(D, 1.0);
    if (psi && psi_len == D) std::memcpy(psi_eff.data(), psi, D * sizeof(double));
    API_CUDA_TRY(cudaMemcpyAsync(d_x, rho, T * D * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    if (initial) API_CUDA_TRY(cudaMemcpyAsync(d_init, initial, T * sizeof(int), cudaMemcpyHostToDevice, C.stream));
    vbx::Config vc;
    vc.Fa = cfg->Fa;
    vc.Fb = cfg->Fb;
    vc.max_iterations = cfg->max_iterations;
    vc.epsilon = cfg->epsilon;
    vc.init_smoothing = cfg->init_smoothing;
    int its = 0;
    long long lc = 0;
    st = vbx::refine_device(C.vbx_ws, d_x, (int)T, (int)D, psi_eff.data(), initial ? d_init : nullptr, S, vc, d_gamma,
                            d_pi, d_elbos, d_hard, &its, C.stream, &lc);
    g_launches += lc;
    if (st != FA_OK) return (fa_status)st;
    API_CUDA_TRY(cudaMemcpyAsync(gamma, d_gamma, T * (size_t)S * sizeof(double), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaMemcpyAsync(pi, d_pi, S * sizeof(double), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaMemcpyAsync(elbos, d_elbos, cap * sizeof(double), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaMemcpyAsync(hard, d_hard, T * sizeof(int), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaStreamSynchronize(C.stream));
    if (iterations) *iterations = its;
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_compute_centroids(const double *emb, size_t T, size_t dim, const double *gamma, const double *pi,
                                      int32_t S, double *centroids, int32_t *centroid_count) {
    if (!emb || !gamma || !pi || !centroids || !centroid_count || T == 0 || dim == 0 || S <= 0)
        return FA_STATUS_INVALID_ARGUMENT;
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    Lease lease;
    if (lease.status != FA_OK) return (fa_status)lease.status;
    ClusterContext &C = *lease.ctx;
    Carver sz{nullptr};
    sz.take<double>(T * dim);
    sz.take<double>(T * (size_t)S);
    sz.take<double>(S);
    sz.take<double>((size_t)S * dim);
    sz.take<double>((size_t)S * dim);
    sz.take<int>(64);
    int st = C.reserve(sz.off + 1024, 64);
    if (st != FA_OK) return (fa_status)st;
    Carver c{static_cast<char *>(C.d_buf)};
    double *d_emb = c.take<double>(T * dim);
    double *d_gamma = c.take<double>(T * (size_t)S);
    double *d_pi = c.take<double>(S);
    double *d_cent = c.take<double>((size_t)S * dim);
    double *d_cent_n = c.take<double>((size_t)S * dim);
    int *d_count = c.take<int>(64);
    API_CUDA_TRY(cudaMemcpyAsync(d_emb, emb, T * dim * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    API_CUDA_TRY(cudaMemcpyAsync(d_gamma, gamma, T * (size_t)S * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    API_CUDA_TRY(cudaMemcpyAsync(d_pi, pi, S * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    long long lc = 0;
    st = vbx::centroids_device(C.vbx_ws, d_emb, (int)T, (int)dim, d_gamma, d_pi, S, d_cent, d_cent_n, d_count, C.stream, &lc);
    g_launches += lc;
    if (st != FA_OK) return (fa_status)st;
    int K = 0;
    API_CUDA_TRY(cudaMemcpyAsync(&K, d_count, sizeof(int), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaStreamSynchronize(C.stream));
    *centroid_count = K;
    if (K > 0) {
        API_CUDA_TRY(cudaMemcpyAsync(centroids, d_cent, (size_t)K * dim * sizeof(double), cudaMemcpyDeviceToHost, C.stream));
        API_CUDA_TRY(cudaStreamSynchronize(C.stream));
    }
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_assign_embeddings(const double *emb, size_t N, size_t dim, const double *centroids, int32_t K,
                                      int32_t *labels, double *scores) {
    if (N == 0) return FA_STATUS_OK;
    if (!emb || !labels || dim == 0 || (K > 0 && !centroids)) return FA_STATUS_INVALID_ARGUMENT;
    if (K <= 0) {   // guard !centroids.isEmpty else all zeros (:805-807)
        for (size_t i = 0; i < N; ++i) labels[i] = 0;
        return FA_STATUS_OK;
    }
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    Lease lease;
    if (lease.status != FA_OK) return (fa_status)lease.status;
    ClusterContext &C = *lease.ctx;
    Carver sz{nullptr};
    sz.take<double>(N * dim);
    sz.take<double>((size_t)K * dim);
    sz.take<double>((size_t)K * dim);
    sz.take<int>(N);
    sz.take<double>(scores ? N * (size_t)K : 1);
    int st = C.reserve(sz.off + 1024, 64);
    if (st != FA_OK) return (fa_status)st;
    Carver c{static_cast<char *>(C.d_buf)};
    double *d_emb = c.take<double>(N * dim);
    double *d_craw = c.take<double>((size_t)K * dim);
    double *d_cn = c.take<double>((size_t)K * dim);
    int *d_labels = c.take<int>(N);
    double *d_scores = c.take<double>(scores ? N * (size_t)K : 1);
    API_CUDA_TRY(cudaMemcpyAsync(d_emb, emb, N * dim * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    API_CUDA_TRY(cudaMemcpyAsync(d_craw, centroids, (size_t)K * dim * sizeof(double), cudaMemcpyHostToDevice, C.stream));
    // centroid normalisation (:793, :824-860; zero rows kept) with the same kernel the pipeline uses
    st = ahc::launch_normalize_rows_keep(d_craw, d_cn, K, (int)dim, C.stream);
    if (st != FA_OK) return (fa_status)st;
    ++g_launches;
    long long lc = 0;
    st = vbx::assign_device(d_emb, (int)N, (int)dim, d_cn, nullptr, K, d_labels, scores ? d_scores : nullptr, C.stream, &lc);
    g_launches += lc;
    if (st != FA_OK) return (fa_status)st;
    API_CUDA_TRY(cudaMemcpyAsync(labels, d_labels, N * sizeof(int), cudaMemcpyDeviceToHost, C.stream));
    if (scores) API_CUDA_TRY(cudaMemcpyAsync(scores, d_scores, N * (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, C.stream));
    API_CUDA_TRY(cudaStreamSynchronize(C.stream));
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_diarize_cluster(const float *emb256, const double *rho, size_t N, size_t emb_dim, size_t rho_dim,
                                    const double *psi, const fa_cluster_config *cfg, int32_t *labels, int32_t *initial,
                                    double *centroids, int32_t max_centroids, fa_cluster_info *info) {
    if (!emb256 || !rho || !cfg || !labels || N == 0 || emb_dim == 0 || rho_dim == 0) {
        fa::set_error("fa_diarize_cluster: null or empty input (the reference throws noSpeechDetected for N == 0)");
        return FA_STATUS_INVALID_ARGUMENT;
    }
    if (N > 0x7fffffffull / 4) return FA_STATUS_INDEX_OVERFLOW;
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    Lease lease;
    if (lease.status != FA_OK) return (fa_status)lease.status;
    const int st = cluster_pipeline(*lease.ctx, emb256, rho, N, emb_dim, rho_dim, psi, *cfg, labels, initial, centroids,
                                    max_centroids, info);
    lease.status = st == FA_CUDA_ERROR ? FA_CUDA_ERROR : FA_OK;
    return (fa_status)st;
    FA_GUARD_END
}

FA_API fa_status fa_diarize_cluster_chunks(const float *emb256, const double *rho, size_t N, size_t emb_dim,
                                           size_t rho_dim, const double *psi, const fa_cluster_config *cfg,
                                           const int32_t *chunk_index, int32_t *labels, int32_t *initial,
                                           double *centroids, int32_t max_centroids, fa_cluster_info *info) {
    if (!emb256 || !rho || !cfg || !labels || N == 0 || emb_dim == 0 || rho_dim == 0) return FA_STATUS_INVALID_ARGUMENT;
    if (N > 0x7fffffffull / 4) return FA_STATUS_INDEX_OVERFLOW;
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    Lease lease;
    if (lease.status != FA_OK) return (fa_status)lease.status;
    const int st = cluster_pipeline(*lease.ctx, emb256, rho, N, emb_dim, rho_dim, psi, *cfg, labels, initial, centroids,
                                    max_centroids, info, chunk_index);
    lease.status = st == FA_CUDA_ERROR ? FA_CUDA_ERROR : FA_OK;
    return (fa_status)st;
    FA_GUARD_END
}

FA_API fa_status fa_hungarian_solve(const int64_t *cost, int32_t n, int32_t *assignment) {
    if (n < 0 || (n > 0 && (!cost || !assignment))) return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    assign::min_cost_matching(cost, n, assignment);
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_max_score_assignment(const double *scores, int32_t rows, int32_t cols, int32_t *assignment) {
    if (rows < 0 || cols < 0 || (rows > 0 && !assignment) || (rows > 0 && cols > 0 && !scores))
        return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    assign::max_score_matching(scores, rows, cols, assignment);
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_constrained_assign(const double *scores, size_t N, int32_t K, const int32_t *chunk_index,
                                       int32_t *labels) {
    if (N == 0) return FA_STATUS_OK;
    if (!chunk_index || !labels || K < 0 || (K > 0 && !scores)) return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    assign::constrained_assign(scores, (long long)N, K, chunk_index, labels);
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_build_chunk_assignments(const int32_t *chunk_index, const int32_t *speaker_index,
                                            const int32_t *assignments, size_t N, int32_t num_chunks,
                                            int32_t num_speakers, int32_t cluster_count, int32_t *matrix) {
    if (num_chunks < 0 || num_speakers < 0 || (!matrix && (size_t)num_chunks * num_speakers > 0) ||
        (N > 0 && (!chunk_index || !speaker_index || !assignments)))
        return FA_STATUS_INVALID_ARGUMENT;
    FA_GUARD_BEGIN
    assign::build_chunk_assignments(chunk_index, speaker_index, assignments, (long long)N, num_chunks, num_speakers,
                                    cluster_count, matrix);
    return FA_STATUS_OK;
    FA_GUARD_END
}

// Independent sets run on disjoint SM partitions: `lanes` host threads, each leasing a context whose merge kernel
// is capped at (SMs / lanes) - 1 worker CTAs, pull sets from a shared counter.
static fa_status cluster_batch_impl(const float *emb256, const double *rho, const int64_t *set_offsets,
                                    int32_t set_count, size_t emb_dim, size_t rho_dim, const double *psi,
                                    const fa_cluster_config *cfg, const int32_t *chunk_index, int32_t *labels,
                                    fa_cluster_info *infos) {
    if (!emb256 || !rho || !set_offsets || !cfg || !labels || set_count < 0 || emb_dim == 0 || rho_dim == 0)
        return FA_STATUS_INVALID_ARGUMENT;
    if (set_count == 0) return FA_STATUS_OK;
    API_REQUIRE_DEVICE();
    FA_GUARD_BEGIN
    int dev = 0;
    API_CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    API_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    // Concurrency: as many sets at a time as still leaves each of them enough SMs to keep its node vectors in shared
    // memory (the merge loop is ~3x slower when they are streamed from L2): 5 000 x 256 needs 46 workers + 1 master,
    // so three sets run side by side on 148 SMs; small sets run four at a time.
    long long n_max = 0;
    for (int m = 0; m < set_count; ++m) n_max = std::max<long long>(n_max, set_offsets[m + 1] - set_offsets[m]);
    int lanes = std::max(1, std::min(set_count, 4));
    const int need = ahc::resident_workers_needed((int)std::min<long long>(n_max, INT32_MAX), (int)emb_dim);
    if (need > 0 && need + 1 <= prop.multiProcessorCount)
        lanes = std::max(1, std::min(lanes, prop.multiProcessorCount / (need + 1)));
    const int worker_limit = lanes == 1 ? 0 : std::max(1, prop.multiProcessorCount / lanes - 1);
    std::atomic<int> next{0};
    std::vector<int> status(lanes, FA_OK);
    std::vector<std::string> messages(lanes);
    // Each lane is a plain std::thread: nothing may escape it (an exception leaving a thread function is std::terminate,
    // and FA_GUARD_* only covers the calling thread), so the body is wrapped and failures are reported through status[].
    auto run_lane = [&](int lane) {
        if (cudaSetDevice(dev) != cudaSuccess) {
            status[lane] = FA_CUDA_ERROR;
            return;
        }
        Lease lease(worker_limit);
        if (lease.status != FA_OK) {
            status[lane] = lease.status;
            messages[lane] = fa::last_error();
            return;
        }
        for (;;) {
            const int m = next.fetch_add(1);
            if (m >= set_count) break;
            const int64_t a = set_offsets[m], b = set_offsets[m + 1];
            if (b <= a) continue;
            const int st = cluster_pipeline(*lease.ctx, emb256 + (size_t)a * emb_dim, rho + (size_t)a * rho_dim,
                                            (size_t)(b - a), emb_dim, rho_dim, psi, *cfg, labels + a, nullptr, nullptr,
                                            0, infos ? infos + m : nullptr, chunk_index ? chunk_index + a : nullptr);
            if (st != FA_OK) {
                status[lane] = st;
                messages[lane] = fa::last_error();
                lease.status = st == FA_CUDA_ERROR ? FA_CUDA_ERROR : FA_OK;
                break;
            }
        }
    };
    auto run = [&](int lane) noexcept {
        try {
            run_lane(lane);
        } catch (const std::bad_alloc &) {
            status[lane] = FA_ALLOCATION_FAILURE;
            try { messages[lane] = "host allocation failed"; } catch (...) {}
        } catch (const std::exception &ex) {
            status[lane] = FA_RUNTIME_ERROR;
            try { messages[lane] = std::string("exception: ") + ex.what(); } catch (...) {}
        } catch (...) {
            status[lane] = FA_UNKNOWN_ERROR;
        }
        if (status[lane] != FA_OK) next.store(set_count);   // the other lanes stop taking new sets
    };
    // threads already started are always joined, also when starting a later one fails
    struct Joiner {
        std::vector<std::thread> t;
        ~Joiner() {
            for (auto &x : t)
                if (x.joinable()) x.join();
        }
    } threads;
    threads.t.reserve(lanes);
    int started = 1;
    try {
        for (int l = 1; l < lanes; ++l) {
            threads.t.emplace_back(run, l);
            ++started;
        }
    } catch (...) {   // std::system_error: run with the lanes that did start
    }
    (void)started;
    run(0);
    for (auto &t : threads.t) t.join();
    for (int l = 0; l < lanes; ++l)
        if (status[l] != FA_OK) {
            fa::set_error("%s", messages[l].c_str());
            return (fa_status)status[l];
        }
    return FA_STATUS_OK;
    FA_GUARD_END
}

FA_API fa_status fa_diarize_cluster_batch(const float *emb256, const double *rho, const int64_t *set_offsets,
                                          int32_t set_count, size_t emb_dim, size_t rho_dim, const double *psi,
                                          const fa_cluster_config *cfg, int32_t *labels, fa_cluster_info *infos) {
    return cluster_batch_impl(emb256, rho, set_offsets, set_count, emb_dim, rho_dim, psi, cfg, nullptr, labels, infos);
}

// The reference's default (constrained) assignment per set: chunk_index[row] = TimedEmbedding.chunkIndex of that row,
// numbered inside its own set.
FA_API fa_status fa_diarize_cluster_batch_chunks(const float *emb256, const double *rho, const int64_t *set_offsets,
                                                 int32_t set_count, size_t emb_dim, size_t rho_dim, const double *psi,
                                                 const fa_cluster_config *cfg, const int32_t *chunk_index,
                                                 int32_t *labels, fa_cluster_info *infos) {
    return cluster_batch_impl(emb256, rho, set_offsets, set_count, emb_dim, rho_dim, psi, cfg, chunk_index, labels, infos);
}
