// libhbegp.so — C ABI (include/hbegp.h) over the sm_100a kernels in gemm.cuh / kernels.cuh.
//
// One evaluation of the reference's lml_with_gradient (src/gpr/lml.rs:29-79) is, on the device:
//   scale X -> assemble K (lower tiles) -> recursive Cholesky fused with the triangular inverse
//   (L and W = L^-1 come out together; panel solves, trailing SYRKs and inverse merges are DMMA GEMMs)
//   -> alpha = W^T (W y) -> K^-1 = W^T W (lower tiles, DMMA) -> fused gradient contraction -> finish.
// Evaluations are batched: every kernel carries the batch index in grid.z, and the batch is split over
// a few CUDA streams so that the latency-bound 64x64 leaves of one group overlap the GEMMs of another.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <limits>
#include <condition_variable>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/hbegp.h"
#include "gemm.cuh"
#include "gemm_tf32.cuh"
#include "gemm_i8.cuh"
#include "kernels.cuh"
#include "node_mma.cuh"
#include "lbfgs.h"
#include "adapter.h"
#include "comm.h"

namespace hbegp {

static thread_local std::string g_last_error;

static int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess) {                                                                         \
            int _code = (_e == cudaErrorMemoryAllocation) ? HBEGP_ERR_NOMEM : HBEGP_ERR_CUDA;            \
            return fail(_code, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ +    \
                                   ":" + std::to_string(__LINE__) + ")");                                \
        }                                                                                                \
    } while (0)

static inline double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static const bool g_trace_model = getenv("HBEGP_TRACE_MODEL") != nullptr;  // phase times of model creation on stderr

static inline int round_up(long v, int m) { return (int)(((v + m - 1) / m) * m); }

// dynamic shared memory the d-dependent kernels may use (opt-in limit on sm_100a is 227 KB)
constexpr size_t kMaxFeatureSmem = 200 * 1024;

// Device buffers of dropped models, kept by their context for the next model.  The tuner replaces its model every
// generation; cudaMalloc / cudaFree of the n x n factor and the prediction scratch cost 5-80 ms per model (measured
// at n = 4096..6144), several times the evaluation that fills them.
struct BufPool {
    struct Item {
        void* p;
        size_t bytes;
    };
    std::vector<Item> items;
    size_t held = 0;
    static constexpr size_t kMaxItems = 24;
    static constexpr size_t kMaxHeld = (size_t)16 << 30;
    void* get(size_t need, size_t* got) {
        int best = -1;
        for (int i = 0; i < (int)items.size(); i++)
            if (items[i].bytes >= need && items[i].bytes <= 2 * need + (1 << 20) && (best < 0 || items[i].bytes < items[best].bytes))
                best = i;
        if (best < 0) return nullptr;
        void* p = items[best].p;
        *got = items[best].bytes;
        held -= items[best].bytes;
        items.erase(items.begin() + best);
        return p;
    }
    void put(void* p, size_t bytes) {
        if (items.size() >= kMaxItems || held + bytes > kMaxHeld) {
            cudaFree(p);
            return;
        }
        items.push_back({p, bytes});
        held += bytes;
    }
    void clear() {
        for (auto& it : items) cudaFree(it.p);
        items.clear();
        held = 0;
    }
    ~BufPool() { clear(); }
};

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    BufPool* pool = nullptr;  // optional: where released memory goes and new memory is looked for first
    int ensure(size_t need) {
        if (need <= bytes) return HBEGP_OK;
        release();
        if (pool && (p = pool->get(need, &bytes))) return HBEGP_OK;
        cudaError_t e = cudaMalloc(&p, need);
        if (e != cudaSuccess && pool && !pool->items.empty()) {  // out of memory with memory parked in the pool
            cudaGetLastError();
            pool->clear();
            e = cudaMalloc(&p, need);
        }
        if (e != cudaSuccess) p = nullptr;
        CUDA_TRY(e);
        bytes = need;
        return HBEGP_OK;
    }
    void release() {
        if (p) {
            if (pool) pool->put(p, bytes);
            else cudaFree(p);
        }
        p = nullptr;
        bytes = 0;
    }
};

struct Model;

struct EngineBase {
    int device = 0, dtype = HBEGP_F64;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::vector<cudaStream_t> sub;
    std::vector<cudaEvent_t> sub_done;
    // side stream + two events per group: the inverse-merge product T = L21 W11 of a node runs beside its trailing
    // update (both only read L21); used where the launch sequence is a captured graph (n <= 2048)
    std::vector<cudaStream_t> side;
    std::vector<cudaEvent_t> side_a, side_b;
    cudaStream_t main_side = nullptr;
    cudaEvent_t main_a = nullptr, main_b = nullptr;
    cudaEvent_t fork_ev = nullptr;
    long n = 0;
    int d = 0, np = 0;
    size_t ws_limit = 0;
    long long launches = 0;
    std::vector<Model*> models;  // live models of this context, oldest first (orphaned, not leaked, on ctx_destroy)
    int resident_limit = 4;      // models that keep their factor on the device (<= 0: all); hbegp_ctx_set_resident_models
    long long n_evictions = 0, n_rebuilds = 0;
    void evict_old_models();
    BufPool model_pool;          // buffers of destroyed models (see BufPool)
    virtual ~EngineBase() {}
    virtual int set_data(long n, int d, const void* x, const void* y, bool on_device) = 0;
    virtual int eval_batch(double nu, int B, const double* theta, const double* lo, const double* hi, double* lml,
                           double* grad, int* status) = 0;
    virtual int model_create(double nu, const double* theta, const double* lo, const double* hi, Model** out,
                             double* lml, void* alpha_out, void* kinv_out) = 0;
    virtual int model_extend(Model* prior, Model** out, double* lml, void* alpha_out, void* kinv_out, int* appended) = 0;
    virtual int debug_factor(double nu, const double* theta, void* k, void* w, void* kinv, int* status) = 0;
    virtual int bench_phase(double nu, int B, const double* theta, int phase, int reps, float* ms_out) = 0;
    virtual int debug_poison() = 0;
    virtual int kernel_matrix(double nu, int d, const double* theta, long n1, const void* x1, long n2, const void* x2, void* out) = 0;
    virtual int kernel_theta_grad(double nu, int d, const double* theta, long n, const void* x, void* k_out, void* grad_out) = 0;
    double next_model_noise = 0.0;  // clamped noise of the model being built (fit.rs:164; see Model::noise_clamped)

    // ---- exchange between GPUs (multi-process mode: one context per rank, hbegp_comm_init) -- NCCL on device buffers
    ncclComm_t comm = nullptr;
    int comm_rank = 0, comm_world = 1;
    DevBuf comm_send, comm_recv;
    void* h_comm = nullptr;  // pinned
    size_t h_comm_bytes = 0;
    cudaEvent_t ev_c0 = nullptr, ev_c1 = nullptr;
    double coll_ms_total = 0.0;
    long long n_collectives = 0;
    int last_eval_cnt = -1;  // evaluations whose results the device buffers below hold (-1: spread over several chunks)
    virtual const double* dev_lml() const = 0;
    virtual const double* dev_grad() const = 0;
    virtual const int* dev_status() const = 0;
    virtual Model* new_empty_model(int nu2, const std::vector<double>& prm_h, double noise_clamped) = 0;
    virtual int alloc_data(long n, int d) = 0;  // set_data without the copies (the receiving side of a broadcast)
    virtual void* dev_x() = 0;
    virtual void* dev_y() = 0;
    virtual size_t elem_size() const = 0;
    int ensure_host_comm(size_t bytes) {
        if (bytes <= h_comm_bytes) return HBEGP_OK;
        if (h_comm) cudaFreeHost(h_comm);
        h_comm = nullptr;
        h_comm_bytes = 0;
        CUDA_TRY(cudaMallocHost(&h_comm, bytes));
        h_comm_bytes = bytes;
        return HBEGP_OK;
    }
    void note_collective() {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ev_c0, ev_c1) == cudaSuccess) coll_ms_total += ms;
        n_collectives++;
    }
};

#define NCCL_TRY(expr)                                                                                        \
    do {                                                                                                      \
        ncclResult_t _r = (expr);                                                                             \
        if (_r != ncclSuccess)                                                                                \
            return fail(HBEGP_ERR_CUDA, std::string(#expr) + ": " + Nccl::get().GetErrorString(_r) + " (" + __FILE__ + ":" + \
                                            std::to_string(__LINE__) + ")");                                  \
    } while (0)

struct Model {
    EngineBase* eng = nullptr;
    int dtype = 0;
    long n = 0;
    int d = 0, np = 0, nu2 = 5;
    double c = 1.0;
    DevBuf W, alpha, xsT, ls;  // inverse Cholesky factor (np x np), alpha (np), scaled X^T (d x np), length scales
    DevBuf ldp;                // sum of ln L_ii per 64-row leaf (kept for model_extend)
    std::vector<double> prm_h; // [noise, c, l_1..l_d] as evaluated (after clamping), in the data type's precision
    // noise.with_clamped_value(exp(theta_0) rounded through A) (fit.rs:164, gpr.rs:322): what `extend` evaluates with.
    // prm_h[0] is the unclamped value the fit evaluated (fit.rs:96 does not clamp); they differ only when the optimum
    // sits outside the noise bounds by rounding.
    double noise_clamped = 0.0;
    // How W was computed, which rebuild_nu replays to get the same bits: the recursion over np0 rows of the evaluation
    // that started the chain, then merge_node(r1, np_k - r1) of each append (model_extend) as (r1, np_k).  An append
    // recomputes every row of W from its r1 on, so the entries it supersedes (r1_k >= r1) are dropped.
    int np0 = 0;
    std::vector<std::pair<int, int>> appends;
    // Retained-model policy (SURVEY F10 / H6: the minimizer keeps EVERY generation's model, minimize.rs:331, :407): only
    // the newest few models of a context keep their n x n factor W = L^-1 on the device.  An older one gives W and its
    // prediction scratch back to the pool (O(n d) stays: X^T / l, alpha, the parameters) and refactorises on its next
    // predict_* call.
    bool evicted = false;
    void evict() {
        W.release(); kstar.release(); part.release(); pmean.release(); xs_tmp.release(); mean_tmp.release(); var_tmp.release();
        acq1.release(); acq2.release();
        evicted = true;
    }
    virtual int ensure_resident() = 0;
    // values < -sqrt(1e-5) of the last host prediction (predict.rs:39-46 lists them), in row order
    DevBuf warn_rows, warn_vals;
    std::vector<double> last_warn_vals;
    std::vector<long> last_warn_rows;
    static constexpr int kWarnCap = 4096;
    DevBuf kstar, part, pmean, nbelow, xs_tmp, mean_tmp, var_tmp;
    void release_all() {
        W.release(); alpha.release(); xsT.release(); ls.release(); ldp.release();
        kstar.release(); part.release(); pmean.release(); nbelow.release(); xs_tmp.release(); mean_tmp.release(); var_tmp.release();
        acq1.release(); acq2.release(); argv.release(); argi.release(); warn_rows.release(); warn_vals.release();
    }
    virtual ~Model() {
        release_all();
        if (eng) eng->models.erase(std::remove(eng->models.begin(), eng->models.end(), this), eng->models.end());
    }
    virtual int predict_device(long m, const void* xs, void* mean, void* var, long* n_below_device) = 0;
    virtual int predict_host(long m, const void* xs, void* mean, void* var, long* n_below) = 0;
    virtual int predict_sharded(long m, const void* xs, void* mean, void* var, long* n_below) = 0;
    virtual int predict_acquisition(int mode, const hbegp_ynorm* yn, long m, const void* xs, double param, void* out1,
                                    void* out2, long* best, long* n_below) = 0;
    DevBuf acq1, acq2, argv, argi;
    void use_pool(BufPool* pl) {
        for (DevBuf* b : {&W, &alpha, &xsT, &ls, &ldp, &kstar, &part, &pmean, &nbelow, &xs_tmp, &mean_tmp, &var_tmp, &acq1, &acq2,
                          &argv, &argi, &warn_rows, &warn_vals})
            b->pool = pl;
    }
};

inline void EngineBase::evict_old_models() {
    if (resident_limit <= 0) return;
    int resident = 0;
    for (auto it = models.rbegin(); it != models.rend(); ++it) {
        if ((*it)->evicted) continue;
        if (++resident > resident_limit) {
            (*it)->evict();
            n_evictions++;
        }
    }
}

static int nu_to_nu2(double nu, int* nu2) {
    const double eps = std::numeric_limits<double>::epsilon();
    if (std::fabs(nu - 0.5) <= eps) *nu2 = 1;
    else if (std::fabs(nu - 1.5) <= eps) *nu2 = 3;
    else if (std::fabs(nu - 2.5) <= eps) *nu2 = 5;
    else return fail(HBEGP_ERR_UNSUPPORTED, "Matern kernel with arbitrary values for nu (matern_kernel.rs:79)");
    return HBEGP_OK;
}

template <typename T>
struct ModelT;

template <typename T>
struct Engine : EngineBase {
    DevBuf dX, dY;
    // batched workspaces (capacity `cap` evaluations)
    int cap = 0;
    DevBuf A, W, xsT, prm, u, alpha, ldp, tpart, gpart, d_lml, d_grad, d_status;
    DevBuf oz;  // residue planes of the emulated K^-1 product (gemm_i8.cuh), oz::slot_bytes(np) per evaluation
    // CUDA graphs of whole batched evaluations, keyed by (nu2, count, want_grad, want_kinv, phase): the fit
    // loop replays the same launch sequence hundreds of times, and at small n the host launch rate (hundreds
    // of kernels per evaluation) would otherwise be the bottleneck.
    struct CachedGraph {
        cudaGraphExec_t exec = nullptr;
        long long kernels = 0;
        unsigned epoch = 0;  // graph_epoch it was captured (or last updated) in
    };
    // New training data with the same padded size and feature count leaves the topology of every cached graph intact:
    // only kernel arguments (n, possibly the data pointers) change.  set_data then bumps the epoch instead of dropping
    // the graphs, and a stale graph is re-captured and patched in place with cudaGraphExecUpdate (~1 ms for the 132
    // nodes of a 3-matrix graph at n = 500) instead of being instantiated anew — the reference's loop adds ten rows per
    // generation (src/core/minimize.rs:331-407), so the padded size changes only every sixth generation.
    unsigned graph_epoch = 0;
    std::map<std::tuple<int, int, int, int, int>, CachedGraph> graphs;
    T* h_prm = nullptr;  // pinned staging
    double* h_out = nullptr;
    int* h_status = nullptr;
    size_t h_prm_bytes = 0, h_out_bytes = 0, h_status_bytes = 0;

    void drop_graphs() {
        for (auto& kv : graphs)
            if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
        graphs.clear();
        exact_sizes.clear();
        pad_last_cnt = -1;
        pad_repeat = 0;
    }

    // Batch size a chunk of `cnt` evaluations runs with.  Every distinct size is a graph capture + instantiation
    // (~20 ms at n = 1024), and a fit walks through many sizes as its runs finish, so sizes are rounded up to a
    // multiple of 4 (copies of the last theta, results ignored: 33 distinct graphs -> 9, first fit 0.90 -> 0.27 s).
    // The padding is not free any more now that small batches keep the GPU busy (B = 33 -> 36: +5 % per call), so a
    // size that keeps coming back — a caller's steady loop, the first rounds of a fit — gets its exact graph after
    // four consecutive requests (profiles/r02_pad_ab.log).
    std::vector<int> exact_sizes;
    int pad_last_cnt = -1, pad_repeat = 0;
    int padded_batch(int cnt) {
        if (!(np <= 2048 && cnt > 4)) return cnt;
        const int padded = std::min(cap, (cnt + 3) / 4 * 4);
        if (padded == cnt) return cnt;
        if (std::find(exact_sizes.begin(), exact_sizes.end(), cnt) != exact_sizes.end()) return cnt;
        if (cnt == pad_last_cnt) pad_repeat++;
        else { pad_last_cnt = cnt; pad_repeat = 1; }
        if (pad_repeat >= 4) {
            exact_sizes.push_back(cnt);
            return cnt;
        }
        return padded;
    }

    ~Engine() override {
        drop_graphs();
        for (DevBuf* b : {&dX, &dY, &A, &W, &xsT, &prm, &u, &alpha, &ldp, &tpart, &gpart, &d_lml, &d_grad, &d_status, &oz})
            b->release();
        if (h_prm) cudaFreeHost(h_prm);
        if (h_out) cudaFreeHost(h_out);
        if (h_status) cudaFreeHost(h_status);
    }

    void* dev_x() override { return dX.p; }
    void* dev_y() override { return dY.p; }
    size_t elem_size() const override { return sizeof(T); }
    int alloc_data(long n_, int d_) override { return set_data(n_, d_, nullptr, nullptr, true); }
    const double* dev_lml() const override { return (const double*)d_lml.p; }
    const double* dev_grad() const override { return (const double*)d_grad.p; }
    const int* dev_status() const override { return (const int*)d_status.p; }
    Model* new_empty_model(int nu2, const std::vector<double>& prm_h, double noise_clamped) override;

    int p() const { return d + 2; }
    long mstride() const { return (long)np * np; }
    int ntiles_lower() const { int t = np / TILE; return t * (t + 1) / 2; }
    int nchunks() const { return (np + 255) / 256; }

    int set_data(long n_, int d_, const void* x, const void* y, bool on_device) override {
        const bool alloc_only = on_device && !x && !y;  // alloc_data(): buffers sized and padded, contents arrive by broadcast
        if (n_ <= 0 || d_ <= 0 || (!alloc_only && (!x || !y))) return fail(HBEGP_ERR_INVALID, "set_data: n, d must be positive and x, y non-null");
        if (n_ > 46000) return fail(HBEGP_ERR_INVALID, "set_data: n too large for a single-GPU factorisation");
        if (d_ > 65536) return fail(HBEGP_ERR_UNSUPPORTED, "set_data: more than 65536 features");
        CUDA_TRY(cudaSetDevice(device));
        const void *oldx = dX.p, *oldy = dY.p;
        const bool same_shape = (n == n_ && d == d_);
        const bool same_padded = (np == round_up(n_, TILE) && d == d_ && n > 0);
        n = n_;
        d = d_;
        np = round_up(n, TILE);
        int rc;
        if ((rc = dX.ensure((size_t)np * d * sizeof(T)))) return rc;  // sized by the padded row count: stable while np is
        if ((rc = dY.ensure((size_t)np * sizeof(T)))) return rc;
        if (!same_shape || oldx != dX.p || oldy != dY.p) {
            if (same_padded) {
                graph_epoch++;  // same topology: the cached graphs are patched on their next use (run_chunk)
            } else {
                drop_graphs();
                cap = 0;  // workspaces are re-sized lazily
            }
        }
        cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        CUDA_TRY(cudaMemsetAsync(dY.p, 0, (size_t)np * sizeof(T), stream));
        if (alloc_only) return HBEGP_OK;
        CUDA_TRY(cudaMemcpyAsync(dX.p, x, (size_t)n * d * sizeof(T), kind, stream));
        CUDA_TRY(cudaMemcpyAsync(dY.p, y, (size_t)n * sizeof(T), kind, stream));
        if (!on_device) CUDA_TRY(cudaStreamSynchronize(stream));  // the caller may free x / y
        return HBEGP_OK;
    }

    size_t per_slot_bytes() const {
        size_t s = 2 * (size_t)np * np * sizeof(T);
        s += (size_t)d * np * sizeof(T) + (size_t)p() * sizeof(T) + 2 * (size_t)np * sizeof(T);
        s += (size_t)(np / TILE) * sizeof(T) + (size_t)nchunks() * np * sizeof(T);
        s += (size_t)ntiles_lower() * p() * sizeof(double) + (size_t)(p() + 1) * sizeof(double) + sizeof(int);
        if (kinv_emulated()) s += oz::slot_bytes(np);
        return s;
    }

    int ensure_capacity(int want) {
        if (n <= 0) return fail(HBEGP_ERR_INVALID, "no training data: call hbegp_set_data first");
        if (want <= cap) return HBEGP_OK;
        size_t limit = ws_limit;
        size_t fr = 0, tot = 0;
        CUDA_TRY(cudaMemGetInfo(&fr, &tot));
        // memory already held by the current workspaces (and parked in the model pool) is reusable
        const size_t held = A.bytes + W.bytes + gpart.bytes + tpart.bytes + xsT.bytes + oz.bytes;
        if (limit == 0) limit = (size_t)((double)(fr + held + model_pool.held) * 0.7);
        size_t per = per_slot_bytes();
        int fit = (int)std::min<size_t>(limit / per, 4096);
        if (fit < 1) return fail(HBEGP_ERR_NOMEM, "workspace limit too small for one n x n evaluation");
        int newcap = std::min(want, fit);
        if (newcap <= cap) return HBEGP_OK;
        if ((size_t)newcap * per > fr + held) model_pool.clear();
        drop_graphs();  // buffers may move
        int rc;
        size_t c = (size_t)newcap;
        if ((rc = A.ensure(c * np * np * sizeof(T)))) return rc;
        if ((rc = W.ensure(c * np * np * sizeof(T)))) return rc;
        if ((rc = xsT.ensure(c * d * np * sizeof(T)))) return rc;
        if ((rc = prm.ensure(c * p() * sizeof(T)))) return rc;
        if ((rc = u.ensure(c * np * sizeof(T)))) return rc;
        if ((rc = alpha.ensure(c * np * sizeof(T)))) return rc;
        if ((rc = ldp.ensure(c * (np / TILE) * sizeof(T)))) return rc;
        if ((rc = tpart.ensure(c * nchunks() * np * sizeof(T)))) return rc;
        if ((rc = gpart.ensure(c * ntiles_lower() * p() * sizeof(double)))) return rc;
        if ((rc = d_lml.ensure(c * sizeof(double)))) return rc;
        if ((rc = d_grad.ensure(c * p() * sizeof(double)))) return rc;
        if ((rc = d_status.ensure(((size_t)c + 1) * sizeof(int)))) return rc;  // + the prefix check of model_extend
        if (kinv_emulated() && (rc = oz.ensure(c * oz::slot_bytes(np)))) return rc;
        if (h_prm_bytes < c * p() * sizeof(T)) {
            if (h_prm) cudaFreeHost(h_prm);
            h_prm_bytes = c * p() * sizeof(T);
            CUDA_TRY(cudaMallocHost((void**)&h_prm, h_prm_bytes));
        }
        if (h_out_bytes < c * (p() + 1) * sizeof(double)) {
            if (h_out) cudaFreeHost(h_out);
            h_out_bytes = c * (p() + 1) * sizeof(double);
            CUDA_TRY(cudaMallocHost((void**)&h_out, h_out_bytes));
        }
        if (h_status_bytes < c * sizeof(int)) {
            if (h_status) cudaFreeHost(h_status);
            h_status_bytes = c * sizeof(int);
            CUDA_TRY(cudaMallocHost((void**)&h_status, h_status_bytes));
        }
        cap = newcap;
        return HBEGP_OK;
    }

    // theta (ln space) -> clamped natural parameters rounded to T (fit.rs:94-96, matern_kernel.rs:167-179,
    // constant_kernel.rs:58-62, bounded_value.rs:43-56).  Noise is not clamped.
    void fill_params(const double* theta, const double* lo, const double* hi, T* out) const {
        out[0] = (T)std::exp(theta[0]);
        for (int k = 1; k < p(); k++) {
            double v = std::exp(theta[k]);
            if (lo && v < lo[k]) v = lo[k];
            else if (hi && hi[k] < v) v = hi[k];
            out[k] = (T)v;
        }
    }

    // ---------------------------------------------------------------- recursive Cholesky + inverse
    struct Side {
        cudaStream_t st = nullptr;
        cudaEvent_t a = nullptr, b = nullptr;
    };

    int chol_inv(cudaStream_t st, int s0, int cnt, int r0, int s, Side sd = Side()) {
        T* Ab = (T*)A.p + (size_t)s0 * mstride();
        T* Wb = (T*)W.p + (size_t)s0 * mstride();
        if (s == TILE) {
            CUDA_TRY(launch_prio(k_leaf<T>, dim3(1, 1, cnt), dim3(256), leaf_smem_bytes<T>(), st, Ab, Wb, mstride(), np, r0,
                                 (T*)ldp.p + (size_t)s0 * (np / TILE), np / TILE, (int*)d_status.p + s0));
            launches++;
            return HBEGP_OK;
        }
        if (s == 2 * TILE) {  // the bottom node of the tree in one launch, FP64 arithmetic inside for both precisions
            CUDA_TRY(launch_prio(k_node128_v2<false, T>, dim3(1, 1, cnt), dim3(256), node128_v2_smem_bytes(), st, Ab, Wb, mstride(), np, r0,
                                 (T*)ldp.p + (size_t)s0 * (np / TILE), np / TILE, (int*)d_status.p + s0, (long long*)nullptr));
            launches++;
            return HBEGP_OK;
        }
        // The large blocks are kept multiples of 128 and k_node128_v2 zeroes the (0,1) block of every bottom node, so every
        // 128-wide diagonal tile of W has exact zeros above its diagonal: the invariant the 128-wide tcgen05 tiles (f32)
        // need for their triangular k ranges.
        int q = s / TILE, q1 = (q + 1) / 2;
        if (q >= 4 && (q1 & 1)) q1 += 1;
        if (q1 >= q) q1 = q - 1;
        const int s1 = q1 * TILE, s2 = s - s1;
        int rc;
        if ((rc = chol_inv(st, s0, cnt, r0, s1, sd))) return rc;
        return merge_node(st, s0, cnt, r0, s1, s2, sd);
    }

    // One node of the recursion with the (1,1) block already done: W11 = L11^-1 is in W, the rows below hold A21 and
    // A22.  Also the whole of an append (model_extend): W11 comes from the prior model, s2 covers the new rows.
    int merge_node(cudaStream_t st, int s0, int cnt, int r0, int s1, int s2, Side sd) {
        T* Ab = (T*)A.p + (size_t)s0 * mstride();
        T* Wb = (T*)W.p + (size_t)s0 * mstride();
        int rc;
        T* A21 = Ab + (long)(r0 + s1) * np + r0;
        T* W21 = Wb + (long)(r0 + s1) * np + r0;
        T* W11 = Wb + (long)r0 * np + r0;
        T* A22 = Ab + (long)(r0 + s1) * np + r0 + s1;
        T* W22 = Wb + (long)(r0 + s1) * np + r0 + s1;
        GemmArgs<T> g{};
        g.lda = g.ldb = g.ldc = np;
        g.sA = g.sB = g.sC = mstride();
        g.rowsumsq = nullptr;
        g.small_ctas = np <= SMALL_TILE_NP ? SMALL_TILE_CTAS : 0;
        // 1. panel solve as a product with the inverse: L21 = A21 W11^T  -> W(2,1)
        g.A = A21; g.B = W11; g.C = W21; g.M = s2; g.N = s1; g.K = s1; g.kmode = K_LE_N; g.lower_only = 0;
        g.alpha = T(1); g.beta = T(0);
        CUDA_TRY((launch_gemm_auto<T, true, true>(g, cnt, st))); launches++;
        // 3. T = L21 W11 -> A(2,1); independent of step 2 and of the second half, so it may run on the side stream
        cudaStream_t st3 = st;
        if (sd.st) {
            CUDA_TRY(cudaEventRecord(sd.a, st));
            CUDA_TRY(cudaStreamWaitEvent(sd.st, sd.a, 0));
            st3 = sd.st;
        }
        g.A = W21; g.B = W11; g.C = A21; g.M = s2; g.N = s1; g.K = s1; g.kmode = K_GE_N; g.lower_only = 0;
        g.alpha = T(1); g.beta = T(0);
        CUDA_TRY((launch_gemm_auto<T, true, false>(g, cnt, st3))); launches++;
        if (sd.st) CUDA_TRY(cudaEventRecord(sd.b, sd.st));
        // 2. trailing update: A22 -= L21 L21^T (lower tiles)
        g.A = W21; g.B = W21; g.C = A22; g.M = s2; g.N = s2; g.K = s1; g.kmode = K_FULL; g.lower_only = 1;
        g.alpha = T(-1); g.beta = T(1);
        CUDA_TRY((launch_gemm_auto<T, true, true>(g, cnt, st))); launches++;
        if ((rc = chol_inv(st, s0, cnt, r0 + s1, s2, sd))) return rc;
        // (a nested node may have re-recorded sd.b later on the side stream: waiting for that implies our product)
        if (sd.st) CUDA_TRY(cudaStreamWaitEvent(st, sd.b, 0));
        // 4. W21 = -W22 T
        g.A = W22; g.B = A21; g.C = W21; g.M = s2; g.N = s1; g.K = s2; g.kmode = K_LE_M; g.lower_only = 0;
        g.alpha = T(-1); g.beta = T(0);
        CUDA_TRY((launch_gemm_auto<T, true, false>(g, cnt, st))); launches++;
        return HBEGP_OK;
    }

    // 32x32 GEMM tiles for grids of at most SMALL_TILE_CTAS 64x64 CTAs at n up to SMALL_TILE_NP (gemm.cuh launch_gemm),
    // in the recursion and for K^-1 = W^T W
    static constexpr long SMALL_TILE_CTAS = 296;
    static constexpr int SMALL_TILE_NP = 1024;

    // The f64 K^-1 = W^T W runs on the integer tensor cores (Ozaki scheme II, gemm_i8.cuh) from this padded size on;
    // below it the DMMA kernel is faster.  Measured (B200, 1000 W; probes/kinv_emul_bench.py, hbegp_bench_phase 5, ms
    // DMMA / emulated): B = 65: n = 1536 2.62 / 3.25, 2048 5.90 / 5.77, 3072 18.9 / 14.4, 4096 43.7 / 27.2; B = 1:
    // n = 1536 0.111 / 0.142, 2048 0.178 / 0.210, 4096 0.715 / 0.612.  K^-1 feeds only the gradient contraction and the
    // caller's kinv, so the LML, alpha, W and every prediction keep their bits either way.  Depends on T and np alone,
    // so that a batch, its B = 1 evaluations, graph replays, models and debug_factor agree.
    static constexpr int OZ_MIN_NP = 2048;
    bool kinv_emulated() const { return std::is_same<T, double>::value && np >= OZ_MIN_NP; }

    // K^-1 = W^T W on the lower tiles, written over the (dead) Cholesky factor in A
    int lauum(cudaStream_t st, int s0, int cnt) {
        T* Ab = (T*)A.p + (size_t)s0 * mstride();
        T* Wb = (T*)W.p + (size_t)s0 * mstride();
        if constexpr (std::is_same<T, double>::value) {
            if (kinv_emulated()) {
                CUDA_TRY(oz::launch_kinv(Wb, Ab, mstride(), np, cnt, (unsigned char*)oz.p + (size_t)s0 * oz::slot_bytes(np), st));
                launches += 4;
                return HBEGP_OK;
            }
        }
        GemmArgs<T> g{};
        g.lda = g.ldb = g.ldc = np;
        g.sA = g.sB = g.sC = mstride();
        g.A = Wb; g.B = Wb; g.C = Ab; g.M = np; g.N = np; g.K = np; g.kmode = K_GE_M; g.lower_only = 1;
        g.alpha = T(1); g.beta = T(0);
        g.rowsumsq = nullptr;
        g.small_ctas = np <= SMALL_TILE_NP ? SMALL_TILE_CTAS : 0;
        CUDA_TRY((launch_gemm_auto<T, false, false>(g, cnt, st))); launches++;
        return HBEGP_OK;
    }

    // `phase` truncates the pipeline for the benchmark's per-phase timings (hbegp_bench_phase):
    // 0 = assembly only, 1 = + factor/inverse recursion, 2 = + alpha and K^-1, 3 (default) = everything,
    // 5 = only the K^-1 = W^T W launches (one per stream group) on the W left by the previous evaluation.
    int phase = 3;

    template <int NU2>
    int pipeline_nu(cudaStream_t st, int s0, int cnt, bool want_grad, bool want_kinv, Side sd) {
        T* Ab = (T*)A.p + (size_t)s0 * mstride();
        T* Wb = (T*)W.p + (size_t)s0 * mstride();
        T* xs = (T*)xsT.p + (size_t)s0 * d * np;
        T* pr = (T*)prm.p + (size_t)s0 * p();
        T* ub = (T*)u.p + (size_t)s0 * np;
        T* al = (T*)alpha.p + (size_t)s0 * np;
        T* tp = (T*)tpart.p + (size_t)s0 * nchunks() * np;
        double* gp = (double*)gpart.p + (size_t)s0 * ntiles_lower() * p();
        const size_t xsm = 2 * (size_t)feat_chunk(d) * TILE * sizeof(T);
        if (phase == 5) return lauum(st, s0, cnt);  // benchmark only: the K^-1 product on the W of the last evaluation
        k_scale_x<T><<<dim3((np + 255) / 256, d, cnt), 256, 0, st>>>((const T*)dX.p, (int)n, d, np, pr, p(), xs);
        launches++;
        k_assemble<T, NU2><<<dim3(ntiles_lower(), 1, cnt), 256, xsm, st>>>(xs, (int)n, d, np, pr, p(), Ab, mstride(), 0);
        launches++;
        CUDA_TRY(cudaGetLastError());
        if (phase < 1) return HBEGP_OK;
        int rc;
        if ((rc = chol_inv(st, s0, cnt, 0, np, sd))) return rc;
        if (phase < 2) return HBEGP_OK;
        // alpha = W^T (W y)   (lml.rs:54 solves K alpha = y through the factorisation).  alpha and K^-1 = W^T W both
        // need W only: with a side stream the three latency-bound alpha kernels run beside the K^-1 product.
        const bool split = sd.st && (want_grad || want_kinv);
        cudaStream_t sa = st;
        if (split) {
            CUDA_TRY(cudaEventRecord(sd.a, st));
            CUDA_TRY(cudaStreamWaitEvent(sd.st, sd.a, 0));
            sa = sd.st;
        }
        k_trmv_lower<T><<<dim3(np / 8, 1, cnt), 256, 0, sa>>>(Wb, mstride(), np, (const T*)dY.p, 0, ub, np);
        launches++;
        k_trmv_lower_t_part<T><<<dim3(np / TILE, nchunks(), cnt), 256, 0, sa>>>(Wb, mstride(), np, ub, np, tp, nchunks());
        launches++;
        CUDA_TRY(launch_prio(k_sum_chunks<T>, dim3((np + 255) / 256, 1, cnt), dim3(256), 0, sa, tp, nchunks(), np, al, (long)np));
        launches++;
        if (split) CUDA_TRY(cudaEventRecord(sd.b, sd.st));
        if (want_grad || want_kinv) {
            if ((rc = lauum(st, s0, cnt))) return rc;
        }
        if (split) CUDA_TRY(cudaStreamWaitEvent(st, sd.b, 0));
        if (phase < 3) return HBEGP_OK;
        if (want_grad) {
            const size_t gsm = xsm + 2 * TILE * sizeof(T) + 8 * (size_t)(feat_chunk(d) + 2) * sizeof(double);
            k_grad_contract<T, NU2><<<dim3(ntiles_lower(), 1, cnt), 256, gsm, st>>>(
                Ab, mstride(), (int)n, d, np, xs, al, np, pr, p(), gp, (long)ntiles_lower() * p());
            launches++;
        }
        CUDA_TRY(launch_prio(k_finish<T>, dim3(cnt), dim3(256), 0, st, (const T*)dY.p, al, np, (int)n, np, (T*)ldp.p + (size_t)s0 * (np / TILE),
                             np / TILE, gp, (long)ntiles_lower() * p(), ntiles_lower(), p(), (int*)d_status.p + s0, (double*)d_lml.p + s0,
                             (double*)d_grad.p + (size_t)s0 * p(), want_grad ? 1 : 0));
        launches++;
        return HBEGP_OK;
    }

    int pipeline(int nu2, cudaStream_t st, int s0, int cnt, bool want_grad, bool want_kinv, Side sd = Side()) {
        // large n with many matrices per group: the GEMMs fill the GPU on their own
        constexpr int SIDE_MAX_CNT = 4;  // at n > 2048 the side stream serves groups of at most this many matrices
        if (!((np <= 2048 || cnt <= SIDE_MAX_CNT) && np > TILE)) sd = Side();
        if (nu2 == 5) return pipeline_nu<5>(st, s0, cnt, want_grad, want_kinv, sd);
        if (nu2 == 3) return pipeline_nu<3>(st, s0, cnt, want_grad, want_kinv, sd);
        return pipeline_nu<1>(st, s0, cnt, want_grad, want_kinv, sd);
    }

    int n_groups(int cnt) const {
        int g = (int)sub.size();
        // Re-measured in round 2 (profiles/r02_c3_streams.log, r02_streams_sweep.log; B = 33, ms per step with
        // 1 / 2 / 4 / 8 groups): n = 512: 0.669 / 0.639 / 0.640 / 0.631; n = 1024: 2.47 / 2.32 / 2.26 / 2.20;
        // n = 2048: 12.59 / 12.23 / 12.07 / 11.89 -- the latency-bound bottom nodes of one group (a few dozen CTAs on
        // 148 SMs) overlap another group's GEMMs.  With the faster bottom node (node_mma.cuh) up to 16 groups of as few
        // as 2 matrices (1 from n = 1024 up) pay off (profiles/r02_group_min.log: n = 1024 B = 33 1.786 -> 1.750 ms,
        // n = 2048 B = 9 3.70 -> 3.39, n = 500 B = 3 unchanged).
        const int gm = np >= 1024 ? 1 : 2;  // fewest matrices per stream group
        if (np <= 2048) g = std::min(g, std::max(1, cnt / gm));
        else g = std::min(g, 4);
        return std::max(1, std::min(g, cnt));
    }

    // The launch sequence of one batched evaluation (captured into a CUDA graph or issued directly).
    int issue_chunk(int nu2, int cnt, bool want_grad, bool want_kinv) {
        CUDA_TRY(cudaMemcpyAsync(prm.p, h_prm, (size_t)cnt * p() * sizeof(T), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemsetAsync(d_status.p, 0, (size_t)cnt * sizeof(int), stream));
        const int groups = n_groups(cnt);
        if (groups <= 1) {
            Side sd;
            sd.st = main_side; sd.a = main_a; sd.b = main_b;
            int rc = pipeline(nu2, stream, 0, cnt, want_grad, want_kinv, sd);
            if (rc) return rc;
        } else {
            CUDA_TRY(cudaEventRecord(fork_ev, stream));
            int base = cnt / groups, extra = cnt % groups, s0 = 0;
            for (int g = 0; g < groups; g++) {
                int c = base + (g < extra ? 1 : 0);
                CUDA_TRY(cudaStreamWaitEvent(sub[g], fork_ev, 0));
                Side sd;
                sd.st = side[g]; sd.a = side_a[g]; sd.b = side_b[g];
                int rc = pipeline(nu2, sub[g], s0, c, want_grad, want_kinv, sd);
                if (rc) return rc;
                CUDA_TRY(cudaEventRecord(sub_done[g], sub[g]));
                CUDA_TRY(cudaStreamWaitEvent(stream, sub_done[g], 0));
                s0 += c;
            }
        }
        CUDA_TRY(cudaMemcpyAsync(h_out, d_lml.p, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, stream));
        if (want_grad)
            CUDA_TRY(cudaMemcpyAsync(h_out + cap, d_grad.p, (size_t)cnt * p() * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaMemcpyAsync(h_status, d_status.p, (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, stream));
        return HBEGP_OK;
    }

    // Evaluates `cnt` <= cap parameter sets already staged in h_prm; results land in h_out / h_status.
    int run_chunk(int nu2, int cnt, bool want_grad, bool want_kinv) {
        // Graphs pay off where the launch sequence is latency bound (small n).  At n > 2048 kernels run for
        // hundreds of microseconds, the asynchronous launches are hidden anyway, and re-instantiating a
        // ~1000-node graph for every distinct batch size of a fit costs more than it saves (measured: 10.2 s
        // with graphs vs 9.5 s without for the north-star fit; 0.37 s vs 0.39 s at n = 1024).
        const bool legacy = (stream == nullptr || stream == cudaStreamLegacy);
        if (legacy || np > 2048) {
            int rc = issue_chunk(nu2, cnt, want_grad, want_kinv);
            if (rc) return rc;
            CUDA_TRY(cudaStreamSynchronize(stream));
            return HBEGP_OK;
        }
        auto key = std::make_tuple(nu2, cnt, (int)want_grad, (int)want_kinv, phase);
        auto it = graphs.find(key);
        if (it == graphs.end() || it->second.epoch != graph_epoch) {
            const long long before = launches;
            const double t_cap = now_ms();
            CUDA_TRY(cudaStreamBeginCapture(stream, cudaStreamCaptureModeRelaxed));
            int rc = issue_chunk(nu2, cnt, want_grad, want_kinv);
            cudaGraph_t graph = nullptr;
            cudaError_t ce = cudaStreamEndCapture(stream, &graph);
            const long long kernels = launches - before;
            launches = before;
            if (rc) {
                if (graph) cudaGraphDestroy(graph);
                return rc;
            }
            if (ce != cudaSuccess) return fail(HBEGP_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
            bool updated = false;
            if (it != graphs.end()) {  // stale: same topology, new arguments
                cudaGraphExecUpdateResultInfo info;
                if (cudaGraphExecUpdate(it->second.exec, graph, &info) == cudaSuccess) {
                    updated = true;
                    it->second.epoch = graph_epoch;
                    it->second.kernels = kernels;
                } else {
                    cudaGetLastError();
                    cudaGraphExecDestroy(it->second.exec);
                    graphs.erase(it);
                    it = graphs.end();
                }
            }
            if (!updated) {
                CachedGraph cg;
                // per-node priorities (launch.h) only count in a graph instantiated with this flag
                ce = cudaGraphInstantiate(&cg.exec, graph, LaunchPriority::get().small_ctas > 0 ? cudaGraphInstantiateFlagUseNodePriority : 0);
                if (ce != cudaSuccess) {
                    cudaGraphDestroy(graph);
                    return fail(HBEGP_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce));
                }
                cg.kernels = kernels;
                cg.epoch = graph_epoch;
                if (graphs.size() > 256) drop_graphs();
                it = graphs.emplace(key, cg).first;
            }
            cudaGraphDestroy(graph);
            if (g_trace_model)
                fprintf(stderr, "[hbegp] graph for %d matrices: %lld kernels, capture + %s %.3f ms\n", cnt, kernels,
                        updated ? "update" : "instantiate", now_ms() - t_cap);
        }
        CUDA_TRY(cudaGraphLaunch(it->second.exec, stream));
        launches += it->second.kernels;
        CUDA_TRY(cudaStreamSynchronize(stream));
        return HBEGP_OK;
    }

    int eval_batch(double nu, int B, const double* theta, const double* lo, const double* hi, double* lml, double* grad,
                   int* status) override {
        int nu2, rc;
        if ((rc = nu_to_nu2(nu, &nu2))) return rc;
        if (B < 0 || (B > 0 && (!theta || !lml))) return fail(HBEGP_ERR_INVALID, "lml_grad_batch: bad arguments");
        if (B == 0) return HBEGP_OK;
        CUDA_TRY(cudaSetDevice(device));
        if ((rc = ensure_capacity((np <= 2048 && B > 4) ? (B + 3) / 4 * 4 : B))) return rc;
        last_eval_cnt = (B <= cap) ? B : -1;
        for (int b0 = 0; b0 < B; b0 += cap) {
            int cnt = std::min(cap, B - b0);
            for (int b = 0; b < cnt; b++) fill_params(theta + (size_t)(b0 + b) * p(), lo, hi, h_prm + (size_t)b * p());
            // Where evaluations are replayed as CUDA graphs (small n, latency bound) a few extra matrices in grid.z
            // cost next to nothing, while every distinct batch size costs a capture + instantiation: round the
            // batch up to a multiple of 4 with copies of the last theta (their results are ignored).
            const int run = padded_batch(cnt);
            for (int b = cnt; b < run; b++) std::memcpy(h_prm + (size_t)b * p(), h_prm + (size_t)(cnt - 1) * p(), sizeof(T) * p());
            if ((rc = run_chunk(nu2, run, grad != nullptr, false))) return rc;
            for (int b = 0; b < cnt; b++) {
                bool bad = h_status[b] != 0 || !std::isfinite(h_out[b]);
                lml[b0 + b] = bad ? -std::numeric_limits<double>::infinity() : h_out[b];
                if (status) status[b0 + b] = bad ? HBEGP_NOT_PD : HBEGP_OK;
                if (grad)
                    for (int k = 0; k < p(); k++) grad[(size_t)(b0 + b) * p() + k] = bad ? 0.0 : h_out[cap + (size_t)b * p() + k];
            }
        }
        return HBEGP_OK;
    }

    int model_extend(Model* prior, Model** out, double* lml, void* alpha_out, void* kinv_out, int* appended) override;
    template <int NU2>
    int append_nu(ModelT<T>* prior, int r1, bool want_kinv);
    int finish_model(int nu2, Model** out, double* lml, void* alpha_out, void* kinv_out);
    int model_create(double nu, const double* theta, const double* lo, const double* hi, Model** out, double* lml,
                     void* alpha_out, void* kinv_out) override;

    int bench_phase(double nu, int B, const double* theta, int ph, int reps, float* ms_out) override {
        int nu2, rc;
        if ((rc = nu_to_nu2(nu, &nu2))) return rc;
        if (B <= 0 || !theta || reps <= 0 || !ms_out) return fail(HBEGP_ERR_INVALID, "bench_phase: bad arguments");
        CUDA_TRY(cudaSetDevice(device));
        if ((rc = ensure_capacity(B))) return rc;
        if (B > cap) return fail(HBEGP_ERR_NOMEM, "bench_phase: batch does not fit the workspace");
        for (int b = 0; b < B; b++) fill_params(theta + (size_t)b * p(), nullptr, nullptr, h_prm + (size_t)b * p());
        cudaEvent_t e0, e1;
        CUDA_TRY(cudaEventCreate(&e0));
        CUDA_TRY(cudaEventCreate(&e1));
        phase = ph;
        rc = run_chunk(nu2, B, true, false);  // warm-up
        float total = 0.f;
        for (int r = 0; r < reps && rc == HBEGP_OK; r++) {
            cudaEventRecord(e0, stream);
            rc = run_chunk(nu2, B, true, false);
            cudaEventRecord(e1, stream);
            cudaEventSynchronize(e1);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            total += ms;
        }
        phase = 3;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        if (rc) return rc;
        *ms_out = total / reps;
        return HBEGP_OK;
    }

    // trait Kernel::kernel(x1, x2) for Product<ConstantKernel, Matern> (src/gpr/kernel.rs:10-14, product_kernel.rs:36-38,
    // matern_kernel.rs:37-80) through the PRODUCTION cross-kernel code: x2 is scaled with k_scale_x and K(x1, x2) is
    // the k* tile output of k_kstar_mean (the kernel that feeds the predictive mean and variance).
    template <int NU2>
    int kernel_matrix_nu(int dd, const double* theta, long n1, const void* x1, long n2, const void* x2, void* out) {
        const int np2 = round_up(n2, TILE);
        std::vector<T> prm_h(dd + 2);
        prm_h[0] = T(0);
        for (int k = 1; k < dd + 2; k++) prm_h[k] = (T)std::exp(theta[k - 1]);
        const long chunk = 4096;
        DevBuf dx1, dx2, dprm, dxsT, dal, dmean, dks, dout;
        int rc = HBEGP_OK;
        auto done = [&](int code) {
            for (DevBuf* b : {&dx1, &dx2, &dprm, &dxsT, &dal, &dmean, &dks, &dout}) b->release();
            return code;
        };
        if ((rc = dx1.ensure((size_t)n1 * dd * sizeof(T))) || (rc = dx2.ensure((size_t)n2 * dd * sizeof(T))) ||
            (rc = dprm.ensure((size_t)(dd + 2) * sizeof(T))) || (rc = dxsT.ensure((size_t)dd * np2 * sizeof(T))) ||
            (rc = dal.ensure((size_t)np2 * sizeof(T))) || (rc = dmean.ensure((size_t)chunk * sizeof(T))) ||
            (rc = dks.ensure((size_t)chunk * np2 * sizeof(T))) || (rc = dout.ensure((size_t)chunk * n2 * sizeof(T))))
            return done(rc);
        cudaStream_t st = stream;
        cudaError_t ce = cudaMemcpyAsync(dx1.p, x1, (size_t)n1 * dd * sizeof(T), cudaMemcpyHostToDevice, st);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(dx2.p, x2, (size_t)n2 * dd * sizeof(T), cudaMemcpyHostToDevice, st);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(dprm.p, prm_h.data(), (size_t)(dd + 2) * sizeof(T), cudaMemcpyHostToDevice, st);
        if (ce == cudaSuccess) ce = cudaMemsetAsync(dal.p, 0, (size_t)np2 * sizeof(T), st);
        if (ce != cudaSuccess) return done(fail(HBEGP_ERR_CUDA, std::string("kernel_matrix: ") + cudaGetErrorString(ce)));
        k_scale_x<T><<<dim3((np2 + 255) / 256, dd, 1), 256, 0, st>>>((const T*)dx2.p, (int)n2, dd, np2, (const T*)dprm.p, dd + 2, (T*)dxsT.p);
        launches++;
        const size_t ksm = (2 * (size_t)feat_chunk(dd) * TILE + TILE) * sizeof(T);
        for (long row0 = 0; row0 < n1; row0 += chunk) {
            const long rows = std::min(chunk, n1 - row0);
            const int rows_p = round_up(rows, TILE);
            k_kstar_mean<T, NU2><<<dim3((unsigned)(rows_p / TILE), 1), 256, ksm, st>>>(
                (const T*)dx1.p, n1, row0, dd, (const T*)dxsT.p, (int)n2, np2, (const T*)dprm.p + 2, prm_h[1], (const T*)dal.p,
                (T*)dks.p, (T*)dmean.p - row0, np2 / TILE, nullptr, rows_p);
            k_copy_cols<T><<<dim3((unsigned)((n2 + 255) / 256), (unsigned)rows), 256, 0, st>>>((const T*)dks.p, np2, rows, (int)n2, (T*)dout.p);
            launches += 2;
            ce = cudaGetLastError();
            if (ce == cudaSuccess) ce = cudaMemcpyAsync((T*)out + row0 * n2, dout.p, (size_t)rows * n2 * sizeof(T), cudaMemcpyDeviceToHost, st);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
            if (ce != cudaSuccess) return done(fail(HBEGP_ERR_CUDA, std::string("kernel_matrix: ") + cudaGetErrorString(ce)));
        }
        return done(HBEGP_OK);
    }

    int kernel_matrix(double nu, int dd, const double* theta, long n1, const void* x1, long n2, const void* x2, void* out) override {
        int nu2, rc;
        if ((rc = nu_to_nu2(nu, &nu2))) return rc;
        if (dd <= 0 || !theta || n1 < 0 || n2 < 0 || ((n1 > 0 && n2 > 0) && (!x1 || !x2 || !out))) return fail(HBEGP_ERR_INVALID, "kernel_matrix: bad arguments");
        if (n1 == 0 || n2 == 0) return HBEGP_OK;
        CUDA_TRY(cudaSetDevice(device));
        if (nu2 == 5) return kernel_matrix_nu<5>(dd, theta, n1, x1, n2, x2, out);
        if (nu2 == 3) return kernel_matrix_nu<3>(dd, theta, n1, x1, n2, x2, out);
        return kernel_matrix_nu<1>(dd, theta, n1, x1, n2, x2, out);
    }

    // trait Kernel::theta_grad(x) -> (K (n, n), dK/dtheta (n, n, d + 1)) (kernel.rs:16-21, product_kernel.rs:40-70).
    int kernel_theta_grad(double nu, int dd, const double* theta, long nn, const void* x, void* k_out, void* grad_out) override {
        int nu2, rc;
        if ((rc = nu_to_nu2(nu, &nu2))) return rc;
        if (dd <= 0 || !theta || nn < 0 || (nn > 0 && !x)) return fail(HBEGP_ERR_INVALID, "kernel_theta_grad: bad arguments");
        if (nn == 0 || (!k_out && !grad_out)) return HBEGP_OK;
        if ((double)nn * nn * (dd + 1) * sizeof(T) > 8e9) return fail(HBEGP_ERR_NOMEM, "kernel_theta_grad: the (n, n, d + 1) tensor exceeds 8 GB");
        CUDA_TRY(cudaSetDevice(device));
        std::vector<T> ls_h(dd);
        for (int k = 0; k < dd; k++) ls_h[k] = (T)std::exp(theta[1 + k]);
        const T c = (T)std::exp(theta[0]);
        DevBuf dx, dls, dk, dg;
        auto done = [&](int code) {
            for (DevBuf* b : {&dx, &dls, &dk, &dg}) b->release();
            return code;
        };
        if ((rc = dx.ensure((size_t)nn * dd * sizeof(T))) || (rc = dls.ensure((size_t)dd * sizeof(T))) ||
            (k_out && (rc = dk.ensure((size_t)nn * nn * sizeof(T)))) ||
            (grad_out && (rc = dg.ensure((size_t)nn * nn * (dd + 1) * sizeof(T)))))
            return done(rc);
        cudaStream_t st = stream;
        cudaError_t ce = cudaMemcpyAsync(dx.p, x, (size_t)nn * dd * sizeof(T), cudaMemcpyHostToDevice, st);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(dls.p, ls_h.data(), (size_t)dd * sizeof(T), cudaMemcpyHostToDevice, st);
        if (ce != cudaSuccess) return done(fail(HBEGP_ERR_CUDA, std::string("kernel_theta_grad: ") + cudaGetErrorString(ce)));
        dim3 grid((unsigned)((nn + 127) / 128), (unsigned)nn);
        if (nu2 == 5) k_kernel_theta_grad<T, 5><<<grid, 128, 0, st>>>((const T*)dx.p, (int)nn, dd, (const T*)dls.p, c, (T*)dk.p, (T*)dg.p);
        else if (nu2 == 3) k_kernel_theta_grad<T, 3><<<grid, 128, 0, st>>>((const T*)dx.p, (int)nn, dd, (const T*)dls.p, c, (T*)dk.p, (T*)dg.p);
        else k_kernel_theta_grad<T, 1><<<grid, 128, 0, st>>>((const T*)dx.p, (int)nn, dd, (const T*)dls.p, c, (T*)dk.p, (T*)dg.p);
        launches++;
        ce = cudaGetLastError();
        if (ce == cudaSuccess && k_out) ce = cudaMemcpyAsync(k_out, dk.p, (size_t)nn * nn * sizeof(T), cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess && grad_out) ce = cudaMemcpyAsync(grad_out, dg.p, (size_t)nn * nn * (dd + 1) * sizeof(T), cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) return done(fail(HBEGP_ERR_CUDA, std::string("kernel_theta_grad: ") + cudaGetErrorString(ce)));
        return done(HBEGP_OK);
    }

    // Fills the batched workspaces (K / L / K^-1 and W = L^-1 of every slot) with NaN bit patterns: a test aid that
    // proves no kernel reads a cell nobody wrote (buffers come from cudaMalloc / the pool and are never cleared).
    int debug_poison() override {
        CUDA_TRY(cudaSetDevice(device));
        if (A.p) CUDA_TRY(cudaMemsetAsync(A.p, 0xFF, A.bytes, stream));
        if (W.p) CUDA_TRY(cudaMemsetAsync(W.p, 0xFF, W.bytes, stream));
        if (oz.p) CUDA_TRY(cudaMemsetAsync(oz.p, 0xFF, oz.bytes, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        return HBEGP_OK;
    }

    int debug_factor(double nu, const double* theta, void* k, void* w, void* kinv, int* status) override {
        int nu2, rc;
        if ((rc = nu_to_nu2(nu, &nu2))) return rc;
        CUDA_TRY(cudaSetDevice(device));
        if ((rc = ensure_capacity(1))) return rc;
        fill_params(theta, nullptr, nullptr, h_prm);
        CUDA_TRY(cudaMemcpyAsync(prm.p, h_prm, (size_t)p() * sizeof(T), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemsetAsync(d_status.p, 0, sizeof(int), stream));
        DevBuf tmp;
        if ((rc = tmp.ensure((size_t)n * n * sizeof(T)))) return rc;
        dim3 fg((unsigned)((n + 255) / 256), (unsigned)n);
        const size_t xsm = 2 * (size_t)feat_chunk(d) * TILE * sizeof(T);
        auto copy_out = [&](const T* src, void* dst, int mode) -> int {
            k_sym_fill<T><<<fg, 256, 0, stream>>>(src, np, (int)n, (T*)tmp.p, mode);
            CUDA_TRY(cudaMemcpyAsync(dst, tmp.p, (size_t)n * n * sizeof(T), cudaMemcpyDeviceToHost, stream));
            CUDA_TRY(cudaStreamSynchronize(stream));
            return HBEGP_OK;
        };
        k_scale_x<T><<<dim3((np + 255) / 256, d, 1), 256, 0, stream>>>((const T*)dX.p, (int)n, d, np, (T*)prm.p, p(), (T*)xsT.p);
        if (nu2 == 5) k_assemble<T, 5><<<dim3(ntiles_lower(), 1, 1), 256, xsm, stream>>>((T*)xsT.p, (int)n, d, np, (T*)prm.p, p(), (T*)A.p, mstride(), 0);
        else if (nu2 == 3) k_assemble<T, 3><<<dim3(ntiles_lower(), 1, 1), 256, xsm, stream>>>((T*)xsT.p, (int)n, d, np, (T*)prm.p, p(), (T*)A.p, mstride(), 0);
        else k_assemble<T, 1><<<dim3(ntiles_lower(), 1, 1), 256, xsm, stream>>>((T*)xsT.p, (int)n, d, np, (T*)prm.p, p(), (T*)A.p, mstride(), 0);
        CUDA_TRY(cudaGetLastError());
        if (k && (rc = copy_out((T*)A.p, k, 1))) { tmp.release(); return rc; }
        if ((rc = chol_inv(stream, 0, 1, 0, np))) { tmp.release(); return rc; }
        if (w && (rc = copy_out((T*)W.p, w, 1))) { tmp.release(); return rc; }
        if (kinv) {
            if ((rc = lauum(stream, 0, 1))) { tmp.release(); return rc; }
            if ((rc = copy_out((T*)A.p, kinv, 0))) { tmp.release(); return rc; }
        }
        int hs = 0;
        CUDA_TRY(cudaMemcpyAsync(&hs, d_status.p, sizeof(int), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (status) *status = hs ? HBEGP_NOT_PD : HBEGP_OK;
        tmp.release();
        return HBEGP_OK;
    }
};

template <typename T>
struct ModelT : Model {
    int predict_chunk_rows() const {
        size_t budget = (size_t)1 << 30;  // k* chunk of at most 1 GiB
        long rows = (long)(budget / ((size_t)np * sizeof(T)));
        rows = std::max<long>(128, rows / 128 * 128);
        return (int)std::min<long>(rows, 1 << 16);
    }

    // m <= 64: latency path (see k_kstar_small)
    template <int NU2>
    int predict_small(int m, const T* xs, T* mean, T* var, unsigned long long* nb) {
        Engine<T>* e = static_cast<Engine<T>*>(eng);
        cudaStream_t st = e->stream;
        const int ntiles = np / TILE, nctas = np / 8;
        int rc;
        if ((rc = part.ensure(((size_t)ntiles + nctas) * 64 * sizeof(T)))) return rc;
        if (var && (rc = kstar.ensure((size_t)64 * np * sizeof(T)))) return rc;
        T* pmean = (T*)part.p;
        T* psq = pmean + (size_t)ntiles * 64;
        const size_t sm = ((size_t)m * d + 8 * 16) * sizeof(T);
        k_kstar_small<T, NU2><<<ntiles, 256, sm, st>>>(xs, m, d, (const T*)xsT.p, (int)n, np, (const T*)ls.p, (T)c, (const T*)alpha.p,
                                                      var ? (T*)kstar.p : nullptr, pmean);
        e->launches++;
        if (var) {
            k_wmatvec_small<T><<<dim3(nctas, (m + 15) / 16), 256, 0, st>>>((const T*)W.p, np, (const T*)kstar.p, m, psq);
            e->launches++;
        }
        k_small_finish<T><<<1, 64, 0, st>>>(pmean, ntiles, psq, nctas, m, (T)c, mean, var, nb, (long*)warn_rows.p, (T*)warn_vals.p, kWarnCap);
        e->launches++;
        CUDA_TRY(cudaGetLastError());
        return HBEGP_OK;
    }

    template <int NU2>
    int predict_impl(long m, const T* xs, T* mean, T* var, unsigned long long* nb) {
        Engine<T>* e = static_cast<Engine<T>*>(eng);
        cudaStream_t st = e->stream;
        if (m <= 64 && (size_t)m * d * sizeof(T) <= 40 * 1024) return predict_small<NU2>((int)m, xs, mean, var, nb);
        const size_t ksm = (2 * (size_t)feat_chunk(d) * TILE + TILE) * sizeof(T);
        const int ttiles = np / TILE;
        // The train tiles are split over grid.y in FIXED groups of 16 (1024 training rows); the partial means are summed
        // in group order by k_var_finish.  A fixed group size (instead of one chosen from the number of candidate
        // tiles) makes a candidate's mean independent of how many rows are predicted with it -- the same bits whether
        // the rows arrive in one call, in chunks, or sharded over GPUs -- and keeps the GPU full for few candidates.
        const int tpc = 16, ns = (ttiles + tpc - 1) / tpc;
        int rc;
        if (var == nullptr) {
            const int chunk_cap = 1 << 20;
            for (long row0 = 0; row0 < m; row0 += chunk_cap) {
                const int rows = round_up(std::min<long>(chunk_cap, m - row0), TILE);
                T* pm = nullptr;
                if (ns > 1) {
                    if ((rc = pmean.ensure((size_t)ns * rows * sizeof(T)))) return rc;
                    pm = (T*)pmean.p;
                }
                k_kstar_mean<T, NU2><<<dim3((unsigned)(rows / TILE), ns), 256, ksm, st>>>(xs, m, row0, d, (const T*)xsT.p, (int)n, np,
                                                                                       (const T*)ls.p, (T)c, (const T*)alpha.p, nullptr,
                                                                                       mean, tpc, pm, rows);
                e->launches++;
                if (pm) {
                    k_var_finish<T><<<(rows + 255) / 256, 256, 0, st>>>(nullptr, 0, 0, rows, m, row0, (T)c, nullptr, nb, pm, ns, rows, mean, nullptr, nullptr, 0);
                    e->launches++;
                }
            }
            CUDA_TRY(cudaGetLastError());
            return HBEGP_OK;
        }
        const int chunk = (int)std::min<long>(predict_chunk_rows(), round_up(m, 128));
        if ((rc = kstar.ensure((size_t)chunk * np * sizeof(T)))) return rc;
        if ((rc = part.ensure((size_t)chunk * (np / TILE) * sizeof(T)))) return rc;  // one partial per 64-wide column tile at most
        for (long row0 = 0; row0 < m; row0 += chunk) {
            const int rows = (int)std::min<long>(chunk, round_up(m - row0, 128));
            // The variance kernel is chosen from np alone, never from the row count: a candidate's variance then has
            // the same bits however many rows are predicted with it (f32: 3xTF32 or FFMA sum in different orders).
            // rows is a multiple of 128, so the TF32 tiles are full in M even when rows < 256.
            const bool tf = gemm_uses_tf32<T>(np, np);
            const int bn = tf ? 128 : 64;
            const int ntile = (np + bn - 1) / bn;
            T* pm = nullptr;
            if (ns > 1) {
                if ((rc = pmean.ensure((size_t)ns * rows * sizeof(T)))) return rc;
                pm = (T*)pmean.p;
            }
            k_kstar_mean<T, NU2><<<dim3(rows / TILE, ns), 256, ksm, st>>>(xs, m, row0, d, (const T*)xsT.p, (int)n, np, (const T*)ls.p, (T)c,
                                                                       (const T*)alpha.p, (T*)kstar.p, mean, tpc, pm, rows);
            e->launches++;
            // |W k*|^2 per candidate: U = k* W^T restricted to k <= column tile, squared and row-summed in the epilogue
            GemmArgs<T> g{};
            g.A = (const T*)kstar.p; g.lda = np; g.sA = 0;
            g.B = (const T*)W.p; g.ldb = np; g.sB = 0;
            g.C = nullptr; g.ldc = 0; g.sC = 0;
            g.M = rows; g.N = np; g.K = np; g.kmode = K_LE_N; g.lower_only = 0;
            g.alpha = T(1); g.beta = T(0);
            g.rowsumsq = (T*)part.p; g.ld_rs = ntile; g.s_rs = 0;
            // keep ~48 MB of k* rows resident in L2 while W streams (ncu before: 35 GB of DRAM reads per 1 GB chunk)
            g.raster_group = (int)std::max<size_t>(1, ((size_t)48 << 20) / ((size_t)bn * np * sizeof(T)));
            if constexpr (std::is_same<T, float>::value) {
                if (tf) CUDA_TRY((tf32::launch<true, true>(g, 1, st)));
                else CUDA_TRY((launch_gemm<T, true, true>(g, 1, st)));
            } else CUDA_TRY((launch_gemm<T, true, true>(g, 1, st)));
            e->launches++;
            k_var_finish<T><<<(rows + 255) / 256, 256, 0, st>>>((const T*)part.p, ntile, ntile, rows, m, row0, (T)c, var, nb, pm, ns, rows, mean,
                                                                (long*)warn_rows.p, (T*)warn_vals.p, kWarnCap);
            e->launches++;
            CUDA_TRY(cudaGetLastError());
        }
        return HBEGP_OK;
    }

    int predict_device(long m, const void* xs, void* mean, void* var, long* n_below_device) override {
        if (m < 0 || (m > 0 && (!xs || !mean))) return fail(HBEGP_ERR_INVALID, "predict: bad arguments");
        if (m == 0) return HBEGP_OK;
        Engine<T>* e = static_cast<Engine<T>*>(eng);
        CUDA_TRY(cudaSetDevice(e->device));
        int rc;
        if (var && (rc = ensure_resident())) return rc;  // the mean needs alpha and X^T / l only
        if ((rc = nbelow.ensure(sizeof(unsigned long long)))) return rc;
        if (var && (rc = warn_rows.ensure(kWarnCap * sizeof(long)))) return rc;
        if (var && (rc = warn_vals.ensure(kWarnCap * sizeof(T)))) return rc;
        unsigned long long* nb = n_below_device ? (unsigned long long*)n_below_device : (unsigned long long*)nbelow.p;
        if (var) CUDA_TRY(cudaMemsetAsync(nb, 0, sizeof(unsigned long long), e->stream));
        if (nu2 == 5) return predict_impl<5>(m, (const T*)xs, (T*)mean, (T*)var, nb);
        if (nu2 == 3) return predict_impl<3>(m, (const T*)xs, (T*)mean, (T*)var, nb);
        return predict_impl<1>(m, (const T*)xs, (T*)mean, (T*)var, nb);
    }

    int predict_acquisition(int mode, const hbegp_ynorm* yn, long m, const void* xs, double param, void* out1, void* out2,
                            long* best, long* n_below) override;

    // Rebuilds the evicted factor: K from the model's own scaled inputs and parameters, then the launches that computed W
    // (the recursion over np0 rows, and each append's merge_node on K re-assembled from its tile row r1 / 64), W back
    // into the model.  Rows of W above r1 depend only on rows of K above r1, so the rows of K that were padding when
    // np0 or an earlier append ran and hold data now do not change them.  The engine's workspaces are used when they are
    // large enough for this model's size, temporary ones otherwise; the context's current training data is not touched.
    template <int NU2>
    int rebuild_nu() {
        Engine<T>* e = static_cast<Engine<T>*>(eng);
        const int p = d + 2;
        const size_t msz = (size_t)np * np * sizeof(T);
        DevBuf tA, tW, tldp, tprm, tstatus;
        int rc;
        const bool fits = e->A.bytes >= msz && e->W.bytes >= msz && e->ldp.bytes >= (size_t)(np / TILE) * sizeof(T) && e->d_status.bytes >= sizeof(int);
        auto done = [&](int code) {
            for (DevBuf* b : {&tA, &tW, &tldp, &tprm, &tstatus}) b->release();
            return code;
        };
        if (!fits) {
            if ((rc = tA.ensure(msz)) || (rc = tW.ensure(msz)) || (rc = tldp.ensure((size_t)(np / TILE) * sizeof(T))) ||
                (rc = tstatus.ensure(2 * sizeof(int))))
                return done(rc);
            std::swap(e->A, tA); std::swap(e->W, tW); std::swap(e->ldp, tldp); std::swap(e->d_status, tstatus);
        }
        auto restore = [&] {
            if (!fits) { std::swap(e->A, tA); std::swap(e->W, tW); std::swap(e->ldp, tldp); std::swap(e->d_status, tstatus); }
        };
        if ((rc = tprm.ensure((size_t)p * sizeof(T))) || (rc = W.ensure(msz))) { restore(); return done(rc); }
        std::vector<T> prm_host(p);
        for (int k = 0; k < p; k++) prm_host[k] = (T)prm_h[k];
        cudaStream_t st = e->stream;
        const long save_n = e->n;
        const int save_np = e->np, save_d = e->d;
        e->n = n; e->np = np; e->d = this->d;  // the recursion reads the matrix size from the engine
        cudaError_t ce = cudaMemcpyAsync(tprm.p, prm_host.data(), (size_t)p * sizeof(T), cudaMemcpyHostToDevice, st);
        if (ce == cudaSuccess) ce = cudaMemsetAsync(e->d_status.p, 0, sizeof(int), st);
        auto assemble = [&](int row0) {  // the lower tiles of K from tile row row0 / TILE on
            const int q = row0 / TILE, tile0 = q * (q + 1) / 2, nt = (np / TILE) * (np / TILE + 1) / 2;
            k_assemble<T, NU2><<<dim3(nt - tile0, 1, 1), 256, 2 * (size_t)feat_chunk(this->d) * TILE * sizeof(T), st>>>(
                (const T*)xsT.p, (int)n, this->d, np, (const T*)tprm.p, p, (T*)e->A.p, (long)np * np, tile0);
            e->launches++;
            return cudaGetLastError();
        };
        if (ce == cudaSuccess) ce = assemble(0);
        rc = HBEGP_OK;
        if (ce == cudaSuccess) rc = e->chol_inv(st, 0, 1, 0, np0);
        for (const auto& a : appends) {
            if (ce != cudaSuccess || rc != HBEGP_OK || a.second == a.first) continue;
            if ((ce = assemble(a.first)) == cudaSuccess) rc = e->merge_node(st, 0, 1, 0, a.first, a.second - a.first, typename Engine<T>::Side());
        }
        int hs = 1;
        if (ce == cudaSuccess && rc == HBEGP_OK) ce = cudaMemcpyAsync(W.p, e->W.p, msz, cudaMemcpyDeviceToDevice, st);
        if (ce == cudaSuccess && rc == HBEGP_OK) ce = cudaMemcpyAsync(&hs, e->d_status.p, sizeof(int), cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess && rc == HBEGP_OK) ce = cudaStreamSynchronize(st);
        e->n = save_n; e->np = save_np; e->d = save_d;
        restore();
        if (ce != cudaSuccess) return done(fail(HBEGP_ERR_CUDA, std::string("model rebuild: ") + cudaGetErrorString(ce)));
        if (rc) return done(rc);
        if (hs) return done(fail(HBEGP_ERR_CUDA, "model rebuild: the kernel matrix of a previously fitted model is not positive definite"));
        evicted = false;
        e->n_rebuilds++;
        return done(HBEGP_OK);
    }

    int ensure_resident() override {
        if (!evicted) return HBEGP_OK;
        int rc = (nu2 == 5) ? rebuild_nu<5>() : (nu2 == 3) ? rebuild_nu<3>() : rebuild_nu<1>();
        if (rc == HBEGP_OK) {
            // it is the most recently used model now: move it to the back and let the policy drop another one
            auto& ms = eng->models;
            ms.erase(std::remove(ms.begin(), ms.end(), (Model*)this), ms.end());
            ms.push_back(this);
            eng->evict_old_models();
        }
        return rc;
    }

    int predict_host(long m, const void* xs, void* mean, void* var, long* n_below) override {
        if (m < 0 || (m > 0 && (!xs || !mean))) return fail(HBEGP_ERR_INVALID, "predict: bad arguments");
        if (n_below) *n_below = 0;
        if (m == 0) return HBEGP_OK;
        Engine<T>* e = static_cast<Engine<T>*>(eng);
        CUDA_TRY(cudaSetDevice(e->device));
        int rc;
        if ((rc = xs_tmp.ensure((size_t)m * d * sizeof(T)))) return rc;
        if ((rc = mean_tmp.ensure((size_t)m * sizeof(T)))) return rc;
        if (var && (rc = var_tmp.ensure((size_t)m * sizeof(T)))) return rc;
        CUDA_TRY(cudaMemcpyAsync(xs_tmp.p, xs, (size_t)m * d * sizeof(T), cudaMemcpyHostToDevice, e->stream));
        if ((rc = predict_device(m, xs_tmp.p, mean_tmp.p, var ? var_tmp.p : nullptr, nullptr))) return rc;
        CUDA_TRY(cudaMemcpyAsync(mean, mean_tmp.p, (size_t)m * sizeof(T), cudaMemcpyDeviceToHost, e->stream));
        unsigned long long hb = 0;
        if (var) {
            CUDA_TRY(cudaMemcpyAsync(var, var_tmp.p, (size_t)m * sizeof(T), cudaMemcpyDeviceToHost, e->stream));
            CUDA_TRY(cudaMemcpyAsync(&hb, nbelow.p, sizeof(hb), cudaMemcpyDeviceToHost, e->stream));
        }
        CUDA_TRY(cudaStreamSynchronize(e->stream));
        if (n_below) *n_below = (long)hb;
        return fetch_warn_list((long)hb);
    }

    // Candidate rows in contiguous blocks over the ranks of the context's communicator: every rank passes the same m
    // rows, predicts its block into the send buffer (mean | variance), one ncclAllGather of the device buffers plus a
    // sum all-reduce of the below-warning count, one copy back.
    int predict_sharded(long m, const void* xs, void* mean, void* var, long* n_below) override {
        Engine<T>* e = static_cast<Engine<T>*>(eng);
        if (!e->comm || e->comm_world == 1) return predict_host(m, xs, mean, var, n_below);
        if (m < 0 || (m > 0 && (!xs || !mean))) return fail(HBEGP_ERR_INVALID, "predict_sharded: bad arguments");
        if (n_below) *n_below = 0;
        if (m == 0) return HBEGP_OK;
        Nccl& nc = Nccl::get();
        const int world = e->comm_world, rank = e->comm_rank;
        const long blk = (m + world - 1) / world;
        const long lo = std::min(m, rank * blk), hi = std::min(m, lo + blk), mine = hi - lo;
        const int cols = var ? 2 : 1;
        const size_t blk_bytes = (size_t)cols * blk * sizeof(T);
        CUDA_TRY(cudaSetDevice(e->device));
        int rc;
        if ((rc = e->comm_send.ensure(blk_bytes))) return rc;
        if ((rc = e->comm_recv.ensure(blk_bytes * world))) return rc;
        if ((rc = e->ensure_host_comm(blk_bytes * world))) return rc;
        if ((rc = nbelow.ensure(sizeof(unsigned long long)))) return rc;
        if ((rc = xs_tmp.ensure((size_t)std::max<long>(mine, 1) * d * sizeof(T)))) return rc;
        T* send = (T*)e->comm_send.p;
        CUDA_TRY(cudaMemsetAsync(send, 0, blk_bytes, e->stream));
        CUDA_TRY(cudaMemsetAsync(nbelow.p, 0, sizeof(unsigned long long), e->stream));
        if (mine > 0) {
            CUDA_TRY(cudaMemcpyAsync(xs_tmp.p, (const T*)xs + (size_t)lo * d, (size_t)mine * d * sizeof(T), cudaMemcpyHostToDevice, e->stream));
            if ((rc = predict_device(mine, xs_tmp.p, send, var ? send + blk : nullptr, nullptr))) return rc;
        }
        CUDA_TRY(cudaEventRecord(e->ev_c0, e->stream));
        NCCL_TRY(nc.GroupStart());
        NCCL_TRY(nc.AllGather(send, e->comm_recv.p, blk_bytes, ncclChar, e->comm, e->stream));
        NCCL_TRY(nc.AllReduce(nbelow.p, nbelow.p, 1, ncclUint64, ncclSum, e->comm, e->stream));
        NCCL_TRY(nc.GroupEnd());
        CUDA_TRY(cudaEventRecord(e->ev_c1, e->stream));
        unsigned long long hb = 0;
        CUDA_TRY(cudaMemcpyAsync(e->h_comm, e->comm_recv.p, blk_bytes * world, cudaMemcpyDeviceToHost, e->stream));
        CUDA_TRY(cudaMemcpyAsync(&hb, nbelow.p, sizeof(hb), cudaMemcpyDeviceToHost, e->stream));
        CUDA_TRY(cudaStreamSynchronize(e->stream));
        e->note_collective();
        for (int r = 0; r < world; r++) {
            const long r0 = std::min(m, r * blk), cnt = std::min(m, r0 + blk) - r0;
            const T* src = (const T*)((const char*)e->h_comm + (size_t)r * blk_bytes);
            if (cnt > 0) std::memcpy((T*)mean + r0, src, (size_t)cnt * sizeof(T));
            if (cnt > 0 && var) std::memcpy((T*)var + r0, src + blk, (size_t)cnt * sizeof(T));
        }
        if (n_below) *n_below = (long)hb;
        last_warn_vals.clear();  // the value list is per rank; only the count is exchanged
        last_warn_rows.clear();
        return HBEGP_OK;
    }

    // The (row, value) pairs below the warning level of the prediction that just finished, sorted by row
    // (the device appends them in arrival order).
    int fetch_warn_list(long count) {
        last_warn_vals.clear();
        last_warn_rows.clear();
        if (count <= 0) return HBEGP_OK;
        Engine<T>* e = static_cast<Engine<T>*>(eng);
        const int k = (int)std::min<long>(count, kWarnCap);
        std::vector<long> rows(k);
        std::vector<T> vals(k);
        CUDA_TRY(cudaMemcpyAsync(rows.data(), warn_rows.p, k * sizeof(long), cudaMemcpyDeviceToHost, e->stream));
        CUDA_TRY(cudaMemcpyAsync(vals.data(), warn_vals.p, k * sizeof(T), cudaMemcpyDeviceToHost, e->stream));
        CUDA_TRY(cudaStreamSynchronize(e->stream));
        std::vector<int> order(k);
        for (int i = 0; i < k; i++) order[i] = i;
        std::sort(order.begin(), order.end(), [&](int a, int b) { return rows[a] < rows[b]; });
        for (int i : order) {
            last_warn_rows.push_back(rows[i]);
            last_warn_vals.push_back((double)vals[i]);
        }
        return HBEGP_OK;
    }
};

// predict + acquisition epilogue + arg-best, all on the device; only the requested vectors come back
template <typename T>
int ModelT<T>::predict_acquisition(int mode, const hbegp_ynorm* yn, long m, const void* xs, double param, void* out1,
                                   void* out2, long* best, long* n_below) {
    if (!yn || m < 0 || (m > 0 && !xs) || (mode != 0 && mode != 1)) return fail(HBEGP_ERR_INVALID, "predict_acquisition: bad arguments");
    if (best) *best = -1;
    if (n_below) *n_below = 0;
    if (m == 0) return HBEGP_OK;
    Engine<T>* e = static_cast<Engine<T>*>(eng);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = e->stream;
    int rc;
    if ((rc = xs_tmp.ensure((size_t)m * d * sizeof(T)))) return rc;
    if ((rc = mean_tmp.ensure((size_t)m * sizeof(T)))) return rc;
    if ((rc = var_tmp.ensure((size_t)m * sizeof(T)))) return rc;
    if ((rc = acq1.ensure((size_t)m * sizeof(T)))) return rc;
    if ((rc = acq2.ensure((size_t)m * sizeof(T)))) return rc;
    const int nparts = (int)std::min<long>(1024, (m + 255) / 256);
    if ((rc = argv.ensure((size_t)nparts * sizeof(T)))) return rc;
    if ((rc = argi.ensure((size_t)(nparts + 1) * sizeof(long)))) return rc;
    CUDA_TRY(cudaMemcpyAsync(xs_tmp.p, xs, (size_t)m * d * sizeof(T), cudaMemcpyHostToDevice, st));
    if ((rc = predict_device(m, xs_tmp.p, mean_tmp.p, var_tmp.p, nullptr))) return rc;
    YNorm<T> y;
    y.amplitude = (T)yn->amplitude;
    y.expected = (T)yn->expected;
    y.projection = yn->projection;
    double fmin_n = 0.0;
    T cb = T(0);
    if (mode == 0) fmin_n = (double)y.into((T)param);  // gpr.rs:192-196: fmin projected into normalised space in A
    else cb = (T)param;
    k_acquisition<T><<<(unsigned)((m + 255) / 256), 256, 0, st>>>((const T*)mean_tmp.p, (const T*)var_tmp.p, m, mode, y.projection,
                                                                 y.amplitude, y.expected, fmin_n, cb, (T*)acq1.p, (T*)acq2.p);
    e->launches++;
    const T* key = (mode == 0) ? (const T*)acq2.p : (const T*)acq1.p;
    long hbest = -1;
    if (best) {
        k_argbest_part<T><<<nparts, 256, 0, st>>>(key, m, mode == 0 ? 1 : 0, (T*)argv.p, (long*)argi.p);
        k_argbest_final<T><<<1, 32, 0, st>>>((const T*)argv.p, (const long*)argi.p, nparts, mode == 0 ? 1 : 0, (long*)argi.p + nparts);
        e->launches += 2;
        CUDA_TRY(cudaMemcpyAsync(&hbest, (long*)argi.p + nparts, sizeof(long), cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaGetLastError());
    if (out1) CUDA_TRY(cudaMemcpyAsync(out1, acq1.p, (size_t)m * sizeof(T), cudaMemcpyDeviceToHost, st));
    if (out2 && mode == 0) CUDA_TRY(cudaMemcpyAsync(out2, acq2.p, (size_t)m * sizeof(T), cudaMemcpyDeviceToHost, st));
    unsigned long long hb = 0;
    CUDA_TRY(cudaMemcpyAsync(&hb, nbelow.p, sizeof(hb), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (best) *best = hbest;
    if (n_below) *n_below = (long)hb;
    return fetch_warn_list((long)hb);
}

template <typename T>
int Engine<T>::model_create(double nu, const double* theta, const double* lo, const double* hi, Model** out, double* lml,
                            void* alpha_out, void* kinv_out) {
    int nu2, rc;
    if ((rc = nu_to_nu2(nu, &nu2))) return rc;
    if (!theta || !out) return fail(HBEGP_ERR_INVALID, "model_create: bad arguments");
    *out = nullptr;
    CUDA_TRY(cudaSetDevice(device));
    if ((rc = ensure_capacity(1))) return rc;
    fill_params(theta, lo, hi, h_prm);
    {
        double nz = (double)h_prm[0];  // noise.with_clamped_value(exp(theta_0) rounded through A) (fit.rs:164)
        if (lo && nz < lo[0]) nz = lo[0];
        else if (hi && hi[0] < nz) nz = hi[0];
        next_model_noise = nz;
    }
    const bool want_kinv = kinv_out != nullptr;
    const double t0 = now_ms();
    if ((rc = run_chunk(nu2, 1, false, want_kinv))) return rc;
    if (g_trace_model) fprintf(stderr, "[hbegp] model_create: evaluation %.3f ms\n", now_ms() - t0);
    return finish_model(nu2, out, lml, alpha_out, kinv_out);
}

// Moves the evaluation in batch slot 0 into a model object (fit.rs:166-175 / :56-67).
template <typename T>
int Engine<T>::finish_model(int nu2, Model** out, double* lml, void* alpha_out, void* kinv_out) {
    int rc;
    if (h_status[0] != 0 || !std::isfinite(h_out[0]))
        return fail(HBEGP_NOT_PD, "Kernel matrix must be invertible. (fit.rs:55)");
    if (lml) *lml = h_out[0];
    const double t0 = now_ms();
    ModelT<T>* m = new ModelT<T>();
    m->eng = this;
    m->use_pool(&model_pool);
    m->dtype = dtype;
    m->n = n;
    m->d = d;
    m->np = np;
    m->np0 = np;
    m->nu2 = nu2;
    m->c = (double)h_prm[1];
    m->prm_h.assign(h_prm, h_prm + p());
    m->noise_clamped = next_model_noise;
    auto bail = [&](int code) { delete m; return code; };
    if ((rc = m->W.ensure((size_t)np * np * sizeof(T)))) return bail(rc);
    if ((rc = m->alpha.ensure((size_t)np * sizeof(T)))) return bail(rc);
    if ((rc = m->xsT.ensure((size_t)d * np * sizeof(T)))) return bail(rc);
    if ((rc = m->ls.ensure((size_t)d * sizeof(T)))) return bail(rc);
    if ((rc = m->ldp.ensure((size_t)(np / TILE) * sizeof(T)))) return bail(rc);
    const double t1 = now_ms();
    cudaError_t ce;
    ce = cudaMemcpyAsync(m->W.p, W.p, (size_t)np * np * sizeof(T), cudaMemcpyDeviceToDevice, stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(m->alpha.p, alpha.p, (size_t)np * sizeof(T), cudaMemcpyDeviceToDevice, stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(m->xsT.p, xsT.p, (size_t)d * np * sizeof(T), cudaMemcpyDeviceToDevice, stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(m->ls.p, (T*)prm.p + 2, (size_t)d * sizeof(T), cudaMemcpyDeviceToDevice, stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(m->ldp.p, ldp.p, (size_t)(np / TILE) * sizeof(T), cudaMemcpyDeviceToDevice, stream);
    if (ce == cudaSuccess && alpha_out) ce = cudaMemcpyAsync(alpha_out, alpha.p, (size_t)n * sizeof(T), cudaMemcpyDeviceToHost, stream);
    if (ce != cudaSuccess) { delete m; return fail(HBEGP_ERR_CUDA, std::string("model_create copy: ") + cudaGetErrorString(ce)); }
    if (kinv_out) {
        DevBuf tmp;
        if ((rc = tmp.ensure((size_t)n * n * sizeof(T)))) return bail(rc);
        dim3 fg((unsigned)((n + 255) / 256), (unsigned)n);
        k_sym_fill<T><<<fg, 256, 0, stream>>>((const T*)A.p, np, (int)n, (T*)tmp.p, 0);
        launches++;
        ce = cudaMemcpyAsync(kinv_out, tmp.p, (size_t)n * n * sizeof(T), cudaMemcpyDeviceToHost, stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(stream);
        tmp.release();
        if (ce != cudaSuccess) { delete m; return fail(HBEGP_ERR_CUDA, std::string("model_create kinv: ") + cudaGetErrorString(ce)); }
    }
    ce = cudaStreamSynchronize(stream);
    if (ce != cudaSuccess) { delete m; return fail(HBEGP_ERR_CUDA, std::string("model_create: ") + cudaGetErrorString(ce)); }
    if (g_trace_model) fprintf(stderr, "[hbegp] finish_model: buffers %.3f ms, copies %.3f ms\n", t1 - t0, now_ms() - t1);
    models.push_back(m);
    evict_old_models();
    *out = m;
    return HBEGP_OK;
}

// A model object with its device buffers allocated but not filled: the receiving side of a model broadcast
// (hbegp_multi_model_create: one GPU evaluates, the others receive W, alpha, X^T / l over NVLink).
template <typename T>
Model* Engine<T>::new_empty_model(int nu2, const std::vector<double>& prm_host, double noise_clamped) {
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    ModelT<T>* m = new ModelT<T>();
    m->eng = this;
    m->use_pool(&model_pool);
    m->dtype = dtype;
    m->n = n;
    m->d = d;
    m->np = np;
    m->np0 = np;
    m->nu2 = nu2;
    m->c = prm_host[1];
    m->prm_h = prm_host;
    m->noise_clamped = noise_clamped;
    if (m->W.ensure((size_t)np * np * sizeof(T)) || m->alpha.ensure((size_t)np * sizeof(T)) || m->xsT.ensure((size_t)d * np * sizeof(T)) ||
        m->ls.ensure((size_t)d * sizeof(T)) || m->ldp.ensure((size_t)(np / TILE) * sizeof(T))) {
        delete m;
        return nullptr;
    }
    models.push_back(m);
    evict_old_models();  // replicas follow the same retained-model policy as locally built models
    return m;
}

// Append path of `extend` (SURVEY 8(f) row f3).  The prior model's W11 = L11^-1 over its first r1 rows stays valid
// when those rows are an unchanged prefix of the new data and theta is unchanged, so only the new tile rows are
// assembled and the factorisation is one node of the recursion: O(n^2 k) instead of O(n^3) for k new rows.
template <typename T>
template <int NU2>
int Engine<T>::append_nu(ModelT<T>* prior, int r1, bool want_kinv) {
    cudaStream_t st = stream;
    T* Ab = (T*)A.p;
    T* Wb = (T*)W.p;
    T* xs = (T*)xsT.p;
    T* pr = (T*)prm.p;
    const int q = r1 / TILE, tile0 = q * (q + 1) / 2;
    const size_t xsm = 2 * (size_t)feat_chunk(d) * TILE * sizeof(T);
    if (ntiles_lower() > tile0) {
        k_assemble<T, NU2><<<dim3(ntiles_lower() - tile0, 1, 1), 256, xsm, st>>>(xs, (int)n, d, np, pr, p(), Ab, mstride(), tile0);
        launches++;
    }
    CUDA_TRY(cudaMemcpy2DAsync(Wb, (size_t)np * sizeof(T), prior->W.p, (size_t)prior->np * sizeof(T), (size_t)r1 * sizeof(T), r1,
                               cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ldp.p, prior->ldp.p, (size_t)q * sizeof(T), cudaMemcpyDeviceToDevice, st));
    int rc;
    if (np > r1 && (rc = merge_node(st, 0, 1, 0, r1, np - r1, Side()))) return rc;
    k_trmv_lower<T><<<dim3(np / 8, 1, 1), 256, 0, st>>>(Wb, mstride(), np, (const T*)dY.p, 0, (T*)u.p, np);
    launches++;
    k_trmv_lower_t_part<T><<<dim3(np / TILE, nchunks(), 1), 256, 0, st>>>(Wb, mstride(), np, (T*)u.p, np, (T*)tpart.p, nchunks());
    launches++;
    k_sum_chunks<T><<<dim3((np + 255) / 256, 1, 1), 256, 0, st>>>((T*)tpart.p, nchunks(), np, (T*)alpha.p, np);
    launches++;
    if (want_kinv && (rc = lauum(st, 0, 1))) return rc;
    k_finish<T><<<1, 256, 0, st>>>((const T*)dY.p, (T*)alpha.p, np, (int)n, np, (T*)ldp.p, np / TILE, (double*)gpart.p,
                                  (long)ntiles_lower() * p(), ntiles_lower(), p(), (int*)d_status.p, (double*)d_lml.p,
                                  (double*)d_grad.p, 0);
    launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(h_out, d_lml.p, sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(h_status, d_status.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return HBEGP_OK;
}

// FittedKernel::extend (fit.rs:33-68): the prior model's theta on the context's current data, one evaluation.
template <typename T>
int Engine<T>::model_extend(Model* prior_, Model** out, double* lml, void* alpha_out, void* kinv_out, int* appended) {
    if (!prior_ || !out) return fail(HBEGP_ERR_INVALID, "model_extend: bad arguments");
    *out = nullptr;
    if (appended) *appended = 0;
    ModelT<T>* prior = static_cast<ModelT<T>*>(prior_);
    if (prior->eng != this) return fail(HBEGP_ERR_INVALID, "model_extend: the prior model belongs to another (or a destroyed) context");
    if (n <= 0) return fail(HBEGP_ERR_INVALID, "model_extend: no training data (hbegp_set_data)");
    if (prior->d != d) return fail(HBEGP_ERR_INVALID, "model_extend: the data has a different number of features than the prior model");
    if ((int)prior->prm_h.size() != p()) return fail(HBEGP_ERR_INVALID, "model_extend: prior model without parameters");
    int rc;
    const double t_start = now_ms();
    CUDA_TRY(cudaSetDevice(device));
    if ((rc = ensure_capacity(1))) return rc;
    for (int k = 0; k < p(); k++) h_prm[k] = (T)prior->prm_h[k];
    h_prm[0] = (T)prior->noise_clamped;  // extend evaluates with prior.noise, the CLAMPED value (fit.rs:41-44, gpr.rs:322)
    next_model_noise = prior->noise_clamped;
    // an append reuses the prior factor, which is only valid if it was computed with the same noise
    const bool same_noise = (T)prior->noise_clamped == (T)prior->prm_h[0];
    const int nu2 = prior->nu2;
    const bool want_kinv = kinv_out != nullptr;
    // the append needs at least one complete 64-row leaf of the prior model and the old rows as a prefix
    // (a multiple of 128 rows of the prior are kept so that the appended blocks stay aligned with the 128-wide tiles)
    int r1 = (int)(std::min<long>(prior->n, n) / (2 * TILE)) * (2 * TILE);
    if (prior->evicted) r1 = 0;  // (an evicted prior would have to be refactorised first: no gain)
    if (prior->n > n || !same_noise) r1 = 0;
    if (r1 > 0) {
        CUDA_TRY(cudaMemcpyAsync(prm.p, h_prm, (size_t)p() * sizeof(T), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemsetAsync(d_status.p, 0, sizeof(int), stream));
        CUDA_TRY(cudaMemsetAsync((int*)d_status.p + cap, 0, sizeof(int), stream));
        k_scale_x<T><<<dim3((np + 255) / 256, d, 1), 256, 0, stream>>>((const T*)dX.p, (int)n, d, np, (T*)prm.p, p(), (T*)xsT.p);
        launches++;
        k_prefix_mismatch<T><<<dim3((r1 + 255) / 256, d), 256, 0, stream>>>((const T*)xsT.p, np, (const T*)prior->xsT.p, prior->np, d, r1,
                                                                          (int*)d_status.p + cap);
        launches++;
        int mismatch = 1;
        CUDA_TRY(cudaMemcpyAsync(&mismatch, (int*)d_status.p + cap, sizeof(int), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (mismatch) r1 = 0;
    }
    if (r1 == 0) {  // different rows or row order: the full evaluation
        if ((rc = run_chunk(nu2, 1, false, want_kinv))) return rc;
    } else {
        if (nu2 == 5) rc = append_nu<5>(prior, r1, want_kinv);
        else if (nu2 == 3) rc = append_nu<3>(prior, r1, want_kinv);
        else rc = append_nu<1>(prior, r1, want_kinv);
        if (rc) return rc;
        if (appended) *appended = 1;
    }
    if (g_trace_model) fprintf(stderr, "[hbegp] model_extend: %s %.3f ms\n", r1 ? "append" : "full evaluation", now_ms() - t_start);
    if ((rc = finish_model(nu2, out, lml, alpha_out, kinv_out))) return rc;
    if (r1 > 0) {
        Model* m = *out;
        m->np0 = prior->np0;
        for (const auto& a : prior->appends)
            if (a.first < r1) m->appends.push_back(a);
        m->appends.emplace_back(r1, np);
    }
    return HBEGP_OK;
}

// cudaFuncSetAttribute for every GEMM instantiation up front (never inside a stream capture)
template <typename T>
static int configure_gemms() {
#define HBEGP_CFG(BM, BN, WM, WN, AK, BK_)                                                                        \
    CUDA_TRY(cudaFuncSetAttribute(gemm_kernel<T, BM, BN, WM, WN, AK, BK_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                  (int)GemmCfg<T, BM, BN, WM, WN, AK, BK_>::SMEM_BYTES))
    HBEGP_CFG(64, 64, 32, 32, true, true);
    HBEGP_CFG(64, 64, 32, 32, true, false);
    HBEGP_CFG(64, 64, 32, 32, false, false);
    if constexpr (std::is_same<T, double>::value) {
        HBEGP_CFG(32, 32, 16, 16, true, true);
        HBEGP_CFG(32, 32, 16, 16, true, false);
        HBEGP_CFG(32, 32, 16, 16, false, false);
    } else {
        HBEGP_CFG(32, 32, 32, 16, true, true);
        HBEGP_CFG(32, 32, 32, 16, true, false);
        HBEGP_CFG(32, 32, 32, 16, false, false);
    }
#undef HBEGP_CFG
    if (std::is_same<T, float>::value) {
        CUDA_TRY((tf32::configure<true, true>()));
        CUDA_TRY((tf32::configure<true, false>()));
        CUDA_TRY((tf32::configure<false, false>()));
    } else {
        CUDA_TRY(oz::configure());
    }
    // kernels whose dynamic shared memory grows with the feature count d (two d x 64 operand tiles)
    const int big = (int)kMaxFeatureSmem;
    CUDA_TRY(cudaFuncSetAttribute(k_leaf<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)leaf_smem_bytes<T>()));
    CUDA_TRY(cudaFuncSetAttribute(k_node128_v2<false, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)node128_v2_smem_bytes()));
    CUDA_TRY(cudaFuncSetAttribute(k_assemble<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(cudaFuncSetAttribute(k_assemble<T, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(cudaFuncSetAttribute(k_assemble<T, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(cudaFuncSetAttribute(k_grad_contract<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(cudaFuncSetAttribute(k_grad_contract<T, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(cudaFuncSetAttribute(k_grad_contract<T, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(cudaFuncSetAttribute(k_kstar_mean<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(cudaFuncSetAttribute(k_kstar_mean<T, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(cudaFuncSetAttribute(k_kstar_mean<T, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    return HBEGP_OK;
}

// ------------------------------------------------------------------------------------ restart loop
// The restart loop of gradmin.rs:7-33 / fit.rs:93-134 with all runs advancing in lockstep: one round = one batched
// evaluation of every live run's next point.  `eval` evaluates a batch (the GPU, or a host objective in
// hbegp_fit_runs_with).  With world > 1 every rank runs the same optimisers on the same values: a round's live runs
// are dealt out round-robin, each rank evaluates its share and a sum all-reduce of the zero-padded round record
// (lml, status, gradient per live run) gives everyone the full round -- the load stays balanced while runs finish at
// different times, and the result is bit-identical to the single-process loop.
using BatchEval = std::function<int(int, const double*, double*, double*, int*)>;

// exchange(B, Bm, rc, xbuf): shares one round between the ranks.  xbuf arrives host-packed (B records of p + 2 doubles
// plus a failure flag, zero where this rank has nothing) and must leave as the element-wise sum over all ranks.
using RoundExchange = std::function<int(int, int, int, std::vector<double>&)>;

static int fit_runs_impl(int p, const BatchEval& eval, int n_runs, const double* starts, const double* blo, const double* bhi,
                         int maxeval, int rank, int world, hbegp_allreduce_fn allreduce, void* ar_user,
                         hbegp_run_result* results, double* best_theta, const RoundExchange* exchange = nullptr) {
    if (n_runs < 0 || (n_runs > 0 && (!starts || !blo || !bhi || !results || !best_theta)))
        return fail(HBEGP_ERR_INVALID, "fit_runs: bad arguments");
    if (world < 1 || rank < 0 || rank >= world || (world > 1 && !allreduce && !exchange))
        return fail(HBEGP_ERR_INVALID, "fit_runs: need 0 <= rank < world and, when world > 1, an all-reduce callback or hbegp_comm_init");
    std::vector<double> lb(p), ub(p);
    for (int k = 0; k < p; k++) {
        if (!(blo[k] > 0) || !(bhi[k] >= blo[k])) return fail(HBEGP_ERR_INVALID, "fit_runs: bounds must satisfy 0 < lo <= hi");
        lb[k] = std::log(blo[k]);  // fit.rs:140, kernel.bounds()
        ub[k] = std::log(bhi[k]);
    }
    std::vector<BoundedLbfgs> opt;
    opt.reserve(n_runs);
    for (int r = 0; r < n_runs; r++) {
        opt.emplace_back(p, starts + (size_t)r * p, lb.data(), ub.data(), maxeval);
        results[r].best_lml = -std::numeric_limits<double>::infinity();
        results[r].best_eval = -1;
        results[r].n_evals = 0;
        results[r].final_f = std::numeric_limits<double>::infinity();
        results[r].status = HBEGP_NOT_PD;
        results[r].reserved = 0;
        for (int k = 0; k < p; k++) best_theta[(size_t)r * p + k] = starts[(size_t)r * p + k];
    }
    std::vector<int> live, mine;
    std::vector<double> th, lml, grad, thm, lmlm, gradm, xbuf;
    std::vector<int> st, stm;
    const int w = p + 2;  // round record per live run: lml, status, gradient
    const bool trace = getenv("HBEGP_TRACE") != nullptr;  // per-round batch sizes on stderr
    for (;;) {
        live.clear();
        for (int r = 0; r < n_runs; r++)
            if (!opt[r].done()) live.push_back(r);
        if (live.empty()) break;
        const int B = (int)live.size();
        if (trace) fprintf(stderr, "hbegp fit round: %d live runs\n", B);
        th.resize((size_t)B * p);
        lml.resize(B);
        grad.resize((size_t)B * p);
        st.resize(B);
        for (int b = 0; b < B; b++) std::memcpy(&th[(size_t)b * p], opt[live[b]].ask(), sizeof(double) * p);
        if (world == 1) {
            int rc = eval(B, th.data(), lml.data(), grad.data(), st.data());
            if (rc) return rc;
        } else {
            mine.clear();
            for (int b = rank; b < B; b += world) mine.push_back(b);
            const int Bm = (int)mine.size();
            thm.resize((size_t)Bm * p);
            lmlm.resize(Bm);
            gradm.resize((size_t)Bm * p);
            stm.resize(Bm);
            for (int i = 0; i < Bm; i++) std::memcpy(&thm[(size_t)i * p], &th[(size_t)mine[i] * p], sizeof(double) * p);
            int rc = Bm ? eval(Bm, thm.data(), lmlm.data(), gradm.data(), stm.data()) : HBEGP_OK;
            // a failing rank must still take part in the collective; the error is reported afterwards
            xbuf.assign((size_t)B * w + 1, 0.0);
            xbuf[(size_t)B * w] = rc ? 1.0 : 0.0;
            for (int i = 0; i < Bm && !rc; i++) {
                double* rec = &xbuf[(size_t)mine[i] * w];
                const bool ok = stm[i] == HBEGP_OK;
                rec[0] = ok ? lmlm[i] : 0.0;
                rec[1] = (double)stm[i];
                for (int k = 0; k < p; k++) rec[2 + k] = ok ? gradm[(size_t)i * p + k] : 0.0;
            }
            if (exchange) {
                int xrc = (*exchange)(B, Bm, rc, xbuf);
                if (xrc) return xrc;
            } else if (allreduce(ar_user, xbuf.data(), (long)xbuf.size())) {
                return fail(HBEGP_ERR_INVALID, "fit_runs: the all-reduce callback failed");
            }
            if (rc) return rc;
            if (xbuf[(size_t)B * w] != 0.0) return fail(HBEGP_ERR_CUDA, "fit_runs: the evaluation failed on another rank");
            for (int b = 0; b < B; b++) {
                const double* rec = &xbuf[(size_t)b * w];
                lml[b] = rec[0];
                st[b] = (int)rec[1];
                std::memcpy(&grad[(size_t)b * p], rec + 2, sizeof(double) * p);
            }
        }
        for (int b = 0; b < B; b++) {
            const int r = live[b];
            hbegp_run_result& R = results[r];
            const bool ok = st[b] == HBEGP_OK;
            // capture rule of fit.rs:115-125: first success, then strictly larger LML only
            if (ok && (R.best_eval < 0 || lml[b] > R.best_lml)) {
                R.best_lml = lml[b];
                R.best_eval = R.n_evals;
                R.status = HBEGP_OK;
                std::memcpy(&best_theta[(size_t)r * p], &th[(size_t)b * p], sizeof(double) * p);
            }
            R.n_evals++;
            double f = ok ? -lml[b] : std::numeric_limits<double>::infinity();
            for (int k = 0; k < p; k++) grad[(size_t)b * p + k] = ok ? -grad[(size_t)b * p + k] : 0.0;
            opt[r].tell(f, &grad[(size_t)b * p]);
            if (opt[r].done()) R.final_f = opt[r].f();
        }
    }
    return HBEGP_OK;
}

// ------------------------------------------------------------------------------------ exchange between GPUs (NCCL)
// One round of the balanced restart loop: this rank's records are packed ON THE DEVICE from the evaluation's result
// buffers into the zero-filled round record (positions rank, rank + world, ... like the dealing in fit_runs_impl), one
// ncclAllReduce(sum) over NVLink shares the round -- every element is summed with zeros only, so all ranks see
// bit-identical values -- and one device-to-host copy brings it back.
static int nccl_exchange_round(EngineBase* e, int B, int Bm, int rc_eval, std::vector<double>& xbuf) {
    Nccl& nc = Nccl::get();
    const int p = e->d + 2, w = p + 2;
    const size_t count = (size_t)B * w + 1;
    CUDA_TRY(cudaSetDevice(e->device));
    int rc;
    if ((rc = e->comm_send.ensure(count * sizeof(double)))) return rc;
    if ((rc = e->ensure_host_comm(count * sizeof(double)))) return rc;
    double* d_round = (double*)e->comm_send.p;
    if (rc_eval == HBEGP_OK && Bm > 0 && e->last_eval_cnt == Bm) {
        CUDA_TRY(cudaMemsetAsync(d_round, 0, count * sizeof(double), e->stream));
        k_pack_round<<<Bm, 64, 0, e->stream>>>(e->dev_lml(), e->dev_grad(), e->dev_status(), Bm, p, e->comm_rank, e->comm_world, d_round);
        e->launches++;
        CUDA_TRY(cudaGetLastError());
    } else {
        // nothing evaluated here this round, a failed evaluation (flag only), or results spread over several chunks:
        // the host-packed record goes up as it is
        std::memcpy(e->h_comm, xbuf.data(), count * sizeof(double));
        CUDA_TRY(cudaMemcpyAsync(d_round, e->h_comm, count * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    }
    CUDA_TRY(cudaEventRecord(e->ev_c0, e->stream));
    NCCL_TRY(nc.AllReduce(d_round, d_round, count, ncclDouble, ncclSum, e->comm, e->stream));
    CUDA_TRY(cudaEventRecord(e->ev_c1, e->stream));
    CUDA_TRY(cudaMemcpyAsync(e->h_comm, d_round, count * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    e->note_collective();
    std::memcpy(xbuf.data(), e->h_comm, count * sizeof(double));
    return HBEGP_OK;
}

// ------------------------------------------------------------------------------------ batched-objective rendezvous
// Keeps the caller's own optimiser in the loop (the reference's NLopt L-BFGS, src/util/gradmin.rs:35-60, one instance
// per restart): every run's objective callback submits its theta and blocks; when all runs that are still live have
// submitted, the last arrival evaluates the whole round with ONE batched GPU call and wakes the others.  The rows
// of a round are ordered by run index, like the lockstep loop of fit_runs_impl, and the capture rule of
// fit.rs:115-125 is recorded per run.
struct Batcher {
    EngineBase* eng = nullptr;
    double nu = 2.5;
    int n_runs = 0, p = 0;
    std::vector<double> lo, hi;
    bool have_bounds = false;
    std::mutex mu;
    std::condition_variable cv;
    std::vector<char> live, submitted;
    std::vector<double> theta, lml, grad;  // per run
    std::vector<int> status;
    std::vector<long long> round_of;  // generation in which run r's pending submission was answered
    long long generation = 0;
    int rc_last = HBEGP_OK;
    std::string err_last;
    std::vector<hbegp_run_result> results;
    std::vector<double> best_theta;
    long long rounds = 0, evals = 0;

    // with `mu` held: is a round complete (every live run has submitted, and there is at least one)?
    bool round_ready() const {
        int waiting = 0;
        for (int r = 0; r < n_runs; r++) {
            if (live[r] && !submitted[r]) return false;
            if (live[r]) waiting++;
        }
        return waiting > 0;
    }

    // with `mu` held (every other participant is blocked on `cv`): evaluate the round and publish it
    void evaluate_round() {
        std::vector<int> rows;
        for (int r = 0; r < n_runs; r++)
            if (live[r] && submitted[r]) rows.push_back(r);
        const int B = (int)rows.size();
        std::vector<double> th((size_t)B * p), l(B), g((size_t)B * p);
        std::vector<int> st(B);
        for (int b = 0; b < B; b++) std::memcpy(&th[(size_t)b * p], &theta[(size_t)rows[b] * p], sizeof(double) * p);
        rc_last = eng->eval_batch(nu, B, th.data(), have_bounds ? lo.data() : nullptr, have_bounds ? hi.data() : nullptr, l.data(),
                                  g.data(), st.data());
        if (rc_last) err_last = g_last_error;
        for (int b = 0; b < B; b++) {
            const int r = rows[b];
            lml[r] = rc_last ? -std::numeric_limits<double>::infinity() : l[b];
            status[r] = rc_last ? HBEGP_NOT_PD : st[b];
            for (int k = 0; k < p; k++) grad[(size_t)r * p + k] = rc_last ? 0.0 : g[(size_t)b * p + k];
            hbegp_run_result& R = results[r];
            if (!rc_last && st[b] == HBEGP_OK && (R.best_eval < 0 || l[b] > R.best_lml)) {  // fit.rs:115-125
                R.best_lml = l[b];
                R.best_eval = R.n_evals;
                R.status = HBEGP_OK;
                std::memcpy(&best_theta[(size_t)r * p], &theta[(size_t)r * p], sizeof(double) * p);
            }
            R.n_evals++;
            submitted[r] = 0;
            round_of[r] = generation;
        }
        generation++;
        rounds++;
        evals += B;
        cv.notify_all();
    }
};

}  // namespace hbegp

// =================================================================================== C ABI
using namespace hbegp;

struct hbegp_ctx {
    EngineBase* eng;
};
struct hbegp_model {
    Model* m;
};

template <typename A>
static int ynorm_fit_t(int projection, long n, const A* y, const double* ko, A* out_y, hbegp_ynorm* out) {
    YNorm<A> yn;
    yn.fit(projection, y, n, ko != nullptr, ko ? (A)*ko : A(0), out_y);
    out->amplitude = (double)yn.amplitude;
    out->expected = (double)yn.expected;
    out->projection = projection;
    return HBEGP_OK;
}

template <typename A>
static int ynorm_apply_t(const hbegp_ynorm* h, int op, long n, const A* a, const A* b, A* out) {
    YNorm<A> yn;
    yn.amplitude = (A)h->amplitude;
    yn.expected = (A)h->expected;
    yn.projection = h->projection;
    for (long i = 0; i < n; i++) {
        switch (op) {
            case 0: out[i] = yn.into(a[i]); break;
            case 1: out[i] = yn.location_from(a[i]); break;
            case 2: out[i] = yn.mean_from(a[i], b[i]); break;
            case 3: out[i] = yn.std_from(a[i], b[i]); break;
            default: out[i] = yn.cv_from(a[i], b[i]); break;
        }
    }
    return HBEGP_OK;
}

extern "C" {

const char* hbegp_version(void) { return "hbegp 0.1.0 (sm_100a)"; }
const char* hbegp_last_error(void) { return g_last_error.c_str(); }

int hbegp_ctx_create(int device, int dtype, void* stream, hbegp_ctx** out) {
    if (!out) return fail(HBEGP_ERR_INVALID, "ctx_create: out is null");
    *out = nullptr;
    if (dtype != HBEGP_F64 && dtype != HBEGP_F32) return fail(HBEGP_ERR_INVALID, "ctx_create: dtype must be HBEGP_F64 or HBEGP_F32");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        return fail(HBEGP_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(ce));
    if (device < 0 || device >= ndev) return fail(HBEGP_ERR_INVALID, "ctx_create: bad device index");
    CUDA_TRY(cudaSetDevice(device));
    EngineBase* e = (dtype == HBEGP_F64) ? static_cast<EngineBase*>(new Engine<double>()) : static_cast<EngineBase*>(new Engine<float>());
    e->device = device;
    e->dtype = dtype;
    if (stream) {
        e->stream = (cudaStream_t)stream;
    } else {
        ce = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
        if (ce != cudaSuccess) { delete e; return fail(HBEGP_ERR_CUDA, cudaGetErrorString(ce)); }
        e->own_stream = true;
    }
    {
        int rc = (dtype == HBEGP_F64) ? configure_gemms<double>() : configure_gemms<float>();
        if (rc) { delete e; return rc; }
    }
    {
        const char* t = getenv("HBEGP_TF32");
        tf32::enabled() = !(t && atoi(t) == 0);
        if (dtype == HBEGP_F32 && tf32::enabled() && !tf32::encode_fn()) {
            delete e;
            return fail(HBEGP_ERR_CUDA, "ctx_create: cuTensorMapEncodeTiled is not available from this driver (set HBEGP_TF32=0)");
        }
    }
    constexpr int STREAM_GROUPS = 16;  // the most a batch is split into (Engine::n_groups)
    for (int i = 0; i < STREAM_GROUPS; i++) {
        cudaStream_t s;
        cudaEvent_t ev;
        if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
            delete e;
            return fail(HBEGP_ERR_CUDA, "ctx_create: could not create streams");
        }
        e->sub.push_back(s);
        e->sub_done.push_back(ev);
        cudaStream_t s2;
        cudaEvent_t ea, eb;
        if (cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ea, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&eb, cudaEventDisableTiming) != cudaSuccess) {
            delete e;
            return fail(HBEGP_ERR_CUDA, "ctx_create: could not create side streams");
        }
        e->side.push_back(s2);
        e->side_a.push_back(ea);
        e->side_b.push_back(eb);
    }
    if (cudaEventCreateWithFlags(&e->fork_ev, cudaEventDisableTiming) != cudaSuccess) { delete e; return fail(HBEGP_ERR_CUDA, "ctx_create: event"); }
    if (cudaStreamCreateWithFlags(&e->main_side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->main_a, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->main_b, cudaEventDisableTiming) != cudaSuccess) {
        delete e;
        return fail(HBEGP_ERR_CUDA, "ctx_create: side stream");
    }
    *out = new hbegp_ctx{e};
    return HBEGP_OK;
}

int hbegp_ctx_destroy(hbegp_ctx* ctx) {
    if (!ctx) return HBEGP_OK;
    EngineBase* e = ctx->eng;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    for (Model* m : e->models) {  // models outliving their context keep answering with HBEGP_ERR_INVALID
        m->release_all();
        m->use_pool(nullptr);
        m->eng = nullptr;
    }
    e->models.clear();
    for (auto s : e->sub) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
    for (auto ev : e->sub_done) cudaEventDestroy(ev);
    for (auto s2 : e->side) { cudaStreamSynchronize(s2); cudaStreamDestroy(s2); }
    for (auto ev : e->side_a) cudaEventDestroy(ev);
    for (auto ev : e->side_b) cudaEventDestroy(ev);
    if (e->main_side) { cudaStreamSynchronize(e->main_side); cudaStreamDestroy(e->main_side); }
    if (e->main_a) cudaEventDestroy(e->main_a);
    if (e->main_b) cudaEventDestroy(e->main_b);
    if (e->fork_ev) cudaEventDestroy(e->fork_ev);
    if (e->comm) Nccl::get().CommDestroy(e->comm);
    e->comm_send.release();
    e->comm_recv.release();
    if (e->h_comm) cudaFreeHost(e->h_comm);
    if (e->ev_c0) cudaEventDestroy(e->ev_c0);
    if (e->ev_c1) cudaEventDestroy(e->ev_c1);
    if (e->own_stream) cudaStreamDestroy(e->stream);
    delete e;
    delete ctx;
    return HBEGP_OK;
}

int hbegp_ctx_set_workspace_limit(hbegp_ctx* ctx, unsigned long long bytes) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    ctx->eng->ws_limit = (size_t)bytes;
    return HBEGP_OK;
}

long long hbegp_ctx_launch_count(hbegp_ctx* ctx) { return ctx ? ctx->eng->launches : 0; }

int hbegp_ctx_set_resident_models(hbegp_ctx* ctx, int max_resident) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    ctx->eng->resident_limit = max_resident;
    ctx->eng->evict_old_models();
    return HBEGP_OK;
}

int hbegp_ctx_model_stats(hbegp_ctx* ctx, int* live, int* resident, long long* evictions, long long* rebuilds) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    int r = 0;
    for (Model* m : ctx->eng->models) r += m->evicted ? 0 : 1;
    if (live) *live = (int)ctx->eng->models.size();
    if (resident) *resident = r;
    if (evictions) *evictions = ctx->eng->n_evictions;
    if (rebuilds) *rebuilds = ctx->eng->n_rebuilds;
    return HBEGP_OK;
}

int hbegp_set_data(hbegp_ctx* ctx, long n, int d, const void* x, const void* y) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    return ctx->eng->set_data(n, d, x, y, false);
}
int hbegp_set_data_device(hbegp_ctx* ctx, long n, int d, const void* x, const void* y) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    return ctx->eng->set_data(n, d, x, y, true);
}

int hbegp_lml_grad_batch(hbegp_ctx* ctx, double nu, int B, const double* theta, const double* lo, const double* hi,
                         double* lml, double* grad, int* status) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    return ctx->eng->eval_batch(nu, B, theta, lo, hi, lml, grad, status);
}

int hbegp_fit_runs(hbegp_ctx* ctx, double nu, int n_runs, const double* starts, const double* bounds_lo,
                   const double* bounds_hi, int maxeval, hbegp_run_result* results, double* best_theta) {
    return hbegp_fit_runs_sharded(ctx, nu, n_runs, starts, bounds_lo, bounds_hi, maxeval, 0, 1, nullptr, nullptr, results, best_theta);
}

int hbegp_fit_runs_sharded(hbegp_ctx* ctx, double nu, int n_runs, const double* starts, const double* bounds_lo,
                           const double* bounds_hi, int maxeval, int rank, int world, hbegp_allreduce_fn allreduce,
                           void* allreduce_user, hbegp_run_result* results, double* best_theta) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    if (ctx->eng->n <= 0) return fail(HBEGP_ERR_INVALID, "no training data: call hbegp_set_data first");
    EngineBase* e = ctx->eng;
    BatchEval eval = [&](int B, const double* th, double* lml, double* grad, int* st) {
        return e->eval_batch(nu, B, th, bounds_lo, bounds_hi, lml, grad, st);
    };
    if (world > 1 && !allreduce) {
        if (!e->comm || e->comm_world != world || e->comm_rank != rank)
            return fail(HBEGP_ERR_INVALID, "fit_runs_sharded: no all-reduce callback and no matching communicator (hbegp_comm_init)");
        RoundExchange ex = [e](int B, int Bm, int rc, std::vector<double>& xbuf) { return nccl_exchange_round(e, B, Bm, rc, xbuf); };
        return fit_runs_impl(e->d + 2, eval, n_runs, starts, bounds_lo, bounds_hi, maxeval, rank, world, nullptr, nullptr, results,
                             best_theta, &ex);
    }
    return fit_runs_impl(e->d + 2, eval, n_runs, starts, bounds_lo, bounds_hi, maxeval, rank, world, allreduce, allreduce_user,
                         results, best_theta);
}

// ---- communicator (multi-process mode: one context per rank)
int hbegp_comm_unique_id(void* id_out) {
    if (!id_out) return fail(HBEGP_ERR_INVALID, "comm_unique_id: null output");
    Nccl& nc = Nccl::get();
    if (!nc.ok()) return fail(HBEGP_ERR_CUDA, nc.error);
    ncclUniqueId id;
    NCCL_TRY(nc.GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == HBEGP_COMM_ID_BYTES, "ncclUniqueId size");
    std::memcpy(id_out, &id, sizeof(id));
    return HBEGP_OK;
}

static int comm_attach(EngineBase* e, ncclComm_t comm, int rank, int world) {
    CUDA_TRY(cudaSetDevice(e->device));  // the timing events belong to this context's device
    e->comm = comm;
    e->comm_rank = rank;
    e->comm_world = world;
    if (!e->ev_c0) {
        CUDA_TRY(cudaEventCreate(&e->ev_c0));
        CUDA_TRY(cudaEventCreate(&e->ev_c1));
    }
    return HBEGP_OK;
}

int hbegp_comm_init(hbegp_ctx* ctx, int world, int rank, const void* id) {
    if (!ctx || !id || world < 1 || rank < 0 || rank >= world) return fail(HBEGP_ERR_INVALID, "comm_init: bad arguments");
    EngineBase* e = ctx->eng;
    if (e->comm) return fail(HBEGP_ERR_INVALID, "comm_init: this context already has a communicator");
    Nccl& nc = Nccl::get();
    if (!nc.ok()) return fail(HBEGP_ERR_CUDA, nc.error);
    CUDA_TRY(cudaSetDevice(e->device));
    ncclUniqueId uid;
    std::memcpy(&uid, id, sizeof(uid));
    ncclComm_t comm = nullptr;
    NCCL_TRY(nc.CommInitRank(&comm, world, uid, rank));
    return comm_attach(e, comm, rank, world);
}

int hbegp_comm_info(hbegp_ctx* ctx, int* rank, int* world, int* nccl_version, double* collective_ms, long long* n_collectives) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    EngineBase* e = ctx->eng;
    if (rank) *rank = e->comm_rank;
    if (world) *world = e->comm ? e->comm_world : 1;
    if (nccl_version) {
        *nccl_version = 0;
        if (Nccl::get().ok()) Nccl::get().GetVersion(nccl_version);
    }
    if (collective_ms) *collective_ms = e->coll_ms_total;
    if (n_collectives) *n_collectives = e->n_collectives;
    return HBEGP_OK;
}

// B thetas known to every rank; rank r evaluates thetas r, r + world, ...; one ncclAllGather of the per-rank record
// blocks (device buffers) and one device-to-host copy give every rank all B results.
int hbegp_lml_grad_batch_sharded(hbegp_ctx* ctx, double nu, int B, const double* theta, const double* lo, const double* hi,
                                 double* lml, double* grad, int* status) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    EngineBase* e = ctx->eng;
    if (!e->comm || e->comm_world == 1) return e->eval_batch(nu, B, theta, lo, hi, lml, grad, status);
    if (B < 0 || (B > 0 && (!theta || !lml))) return fail(HBEGP_ERR_INVALID, "lml_grad_batch_sharded: bad arguments");
    if (B == 0) return HBEGP_OK;
    Nccl& nc = Nccl::get();
    const int p = e->d + 2, w = p + 2, world = e->comm_world, rank = e->comm_rank;
    const int blk = (B + world - 1) / world;          // records per rank (zero padded)
    const size_t blk_count = (size_t)blk * w + 1;     // + this rank's failure flag
    std::vector<double> th, l, g;
    std::vector<int> st;
    int Bm = 0;
    for (int b = rank; b < B; b += world) Bm++;
    th.resize((size_t)Bm * p);
    l.resize(Bm);
    g.resize((size_t)Bm * p);
    st.resize(Bm);
    for (int i = 0; i < Bm; i++) std::memcpy(&th[(size_t)i * p], theta + (size_t)(rank + i * world) * p, sizeof(double) * p);
    int rc_eval = Bm ? e->eval_batch(nu, Bm, th.data(), lo, hi, l.data(), g.data(), st.data()) : HBEGP_OK;
    const std::string eval_err = rc_eval ? g_last_error : std::string();
    CUDA_TRY(cudaSetDevice(e->device));
    int rc;
    if ((rc = e->comm_send.ensure(blk_count * sizeof(double)))) return rc;
    if ((rc = e->comm_recv.ensure(blk_count * world * sizeof(double)))) return rc;
    if ((rc = e->ensure_host_comm(blk_count * world * sizeof(double)))) return rc;
    double* d_send = (double*)e->comm_send.p;
    CUDA_TRY(cudaMemsetAsync(d_send, 0, blk_count * sizeof(double), e->stream));
    if (rc_eval == HBEGP_OK && Bm > 0 && e->last_eval_cnt == Bm) {
        k_pack_round<<<Bm, 64, 0, e->stream>>>(e->dev_lml(), e->dev_grad(), e->dev_status(), Bm, p, 0, 1, d_send);
        e->launches++;
        CUDA_TRY(cudaGetLastError());
    } else {
        double* hs = (double*)e->h_comm;
        std::memset(hs, 0, blk_count * sizeof(double));
        for (int i = 0; i < Bm && !rc_eval; i++) {
            const bool ok = st[i] == HBEGP_OK;
            hs[(size_t)i * w] = ok ? l[i] : 0.0;
            hs[(size_t)i * w + 1] = ok ? 0.0 : 1.0;
            for (int k = 0; k < p; k++) hs[(size_t)i * w + 2 + k] = ok ? g[(size_t)i * p + k] : 0.0;
        }
        hs[(size_t)blk * w] = rc_eval ? 1.0 : 0.0;
        CUDA_TRY(cudaMemcpyAsync(d_send, hs, blk_count * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    }
    CUDA_TRY(cudaEventRecord(e->ev_c0, e->stream));
    NCCL_TRY(nc.AllGather(d_send, e->comm_recv.p, blk_count, ncclDouble, e->comm, e->stream));
    CUDA_TRY(cudaEventRecord(e->ev_c1, e->stream));
    CUDA_TRY(cudaMemcpyAsync(e->h_comm, e->comm_recv.p, blk_count * world * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    e->note_collective();
    if (rc_eval) return fail(rc_eval, eval_err);
    const double* all = (const double*)e->h_comm;
    for (int r = 0; r < world; r++)
        if (all[(size_t)r * blk_count + (size_t)blk * w] != 0.0) return fail(HBEGP_ERR_CUDA, "lml_grad_batch_sharded: the evaluation failed on another rank");
    for (int b = 0; b < B; b++) {
        const double* rec = all + (size_t)(b % world) * blk_count + (size_t)(b / world) * w;
        const bool bad = rec[1] != 0.0;
        lml[b] = bad ? -std::numeric_limits<double>::infinity() : rec[0];
        if (status) status[b] = bad ? HBEGP_NOT_PD : HBEGP_OK;
        if (grad) std::memcpy(grad + (size_t)b * p, rec + 2, sizeof(double) * p);
    }
    return HBEGP_OK;
}

int hbegp_fit_runs_with(hbegp_batch_objective_fn objective, void* objective_user, int p, int n_runs, const double* starts,
                        const double* bounds_lo, const double* bounds_hi, int maxeval, int rank, int world,
                        hbegp_allreduce_fn allreduce, void* allreduce_user, hbegp_run_result* results, double* best_theta) {
    if (!objective || p < 1) return fail(HBEGP_ERR_INVALID, "fit_runs_with: bad arguments");
    BatchEval eval = [&](int B, const double* th, double* lml, double* grad, int* st) {
        int rc = objective(objective_user, B, p, th, lml, grad, st);
        return rc ? fail(HBEGP_ERR_INVALID, "fit_runs_with: the objective callback failed") : HBEGP_OK;
    };
    return fit_runs_impl(p, eval, n_runs, starts, bounds_lo, bounds_hi, maxeval, rank, world, allreduce, allreduce_user, results,
                         best_theta);
}

struct hbegp_batcher {
    Batcher b;
};

int hbegp_batcher_create(hbegp_ctx* ctx, double nu, int n_runs, const double* bounds_lo, const double* bounds_hi,
                         hbegp_batcher** out) {
    if (!ctx || !out || n_runs <= 0) return fail(HBEGP_ERR_INVALID, "batcher_create: bad arguments");
    *out = nullptr;
    if (ctx->eng->n <= 0) return fail(HBEGP_ERR_INVALID, "no training data: call hbegp_set_data first");
    int nu2, rc;
    if ((rc = nu_to_nu2(nu, &nu2))) return rc;
    hbegp_batcher* h = new hbegp_batcher();
    Batcher& b = h->b;
    b.eng = ctx->eng;
    b.nu = nu;
    b.n_runs = n_runs;
    b.p = ctx->eng->d + 2;
    b.have_bounds = bounds_lo && bounds_hi;
    if (b.have_bounds) {
        b.lo.assign(bounds_lo, bounds_lo + b.p);
        b.hi.assign(bounds_hi, bounds_hi + b.p);
    }
    b.live.assign(n_runs, 1);
    b.submitted.assign(n_runs, 0);
    b.theta.assign((size_t)n_runs * b.p, 0.0);
    b.grad.assign((size_t)n_runs * b.p, 0.0);
    b.lml.assign(n_runs, 0.0);
    b.status.assign(n_runs, 0);
    b.round_of.assign(n_runs, -1);
    b.results.resize(n_runs);
    b.best_theta.assign((size_t)n_runs * b.p, 0.0);
    for (auto& R : b.results) {
        R.best_lml = -std::numeric_limits<double>::infinity();
        R.best_eval = -1;
        R.n_evals = 0;
        R.final_f = std::numeric_limits<double>::infinity();
        R.status = HBEGP_NOT_PD;
        R.reserved = 0;
    }
    *out = h;
    return HBEGP_OK;
}

int hbegp_batcher_eval(hbegp_batcher* h, int run, const double* theta, double* lml, double* grad, int* status) {
    if (!h || !theta || !lml || run < 0 || run >= h->b.n_runs) return fail(HBEGP_ERR_INVALID, "batcher_eval: bad arguments");
    Batcher& b = h->b;
    std::unique_lock<std::mutex> lk(b.mu);
    if (!b.live[run]) return fail(HBEGP_ERR_INVALID, "batcher_eval: this run has already left the batcher");
    if (b.submitted[run]) return fail(HBEGP_ERR_INVALID, "batcher_eval: run submitted twice (one thread per run)");
    std::memcpy(&b.theta[(size_t)run * b.p], theta, sizeof(double) * b.p);
    b.submitted[run] = 1;
    const long long my_gen = b.generation;
    if (b.round_ready()) b.evaluate_round();
    else b.cv.wait(lk, [&] { return b.round_of[run] >= my_gen; });
    const int rc = b.rc_last;
    if (rc) return fail(rc, "batcher_eval: the batched evaluation failed: " + b.err_last);
    *lml = b.lml[run];
    if (status) *status = b.status[run];
    if (grad) std::memcpy(grad, &b.grad[(size_t)run * b.p], sizeof(double) * b.p);
    return HBEGP_OK;
}

int hbegp_batcher_leave(hbegp_batcher* h, int run, double final_f) {
    if (!h || run < 0 || run >= h->b.n_runs) return fail(HBEGP_ERR_INVALID, "batcher_leave: bad arguments");
    Batcher& b = h->b;
    std::unique_lock<std::mutex> lk(b.mu);
    if (!b.live[run]) return HBEGP_OK;
    b.live[run] = 0;
    b.submitted[run] = 0;
    b.results[run].final_f = final_f;
    if (b.round_ready()) b.evaluate_round();  // the others were only waiting for this run
    return HBEGP_OK;
}

int hbegp_batcher_results(hbegp_batcher* h, hbegp_run_result* results, double* best_theta, long long* n_rounds) {
    if (!h) return fail(HBEGP_ERR_INVALID, "batcher_results: null batcher");
    Batcher& b = h->b;
    std::unique_lock<std::mutex> lk(b.mu);
    if (results) std::memcpy(results, b.results.data(), sizeof(hbegp_run_result) * b.n_runs);
    if (best_theta) std::memcpy(best_theta, b.best_theta.data(), sizeof(double) * b.best_theta.size());
    if (n_rounds) *n_rounds = b.rounds;
    return HBEGP_OK;
}

int hbegp_batcher_destroy(hbegp_batcher* h) {
    delete h;
    return HBEGP_OK;
}

int hbegp_pick_best_run(int n_runs, const hbegp_run_result* results) {
    int best = -1;
    for (int r = 0; r < n_runs; r++) {
        if (results[r].status != HBEGP_OK || results[r].best_eval < 0) continue;
        if (best < 0 || results[r].best_lml > results[best].best_lml) best = r;
    }
    return best;
}

int hbegp_model_create(hbegp_ctx* ctx, double nu, const double* theta, const double* lo, const double* hi,
                       hbegp_model** out, double* lml, void* alpha_out, void* kinv_out) {
    if (!ctx || !out) return fail(HBEGP_ERR_INVALID, "null context / out");
    Model* m = nullptr;
    int rc = ctx->eng->model_create(nu, theta, lo, hi, &m, lml, alpha_out, kinv_out);
    *out = nullptr;
    if (rc) return rc;
    *out = new hbegp_model{m};
    return HBEGP_OK;
}

int hbegp_model_extend(hbegp_ctx* ctx, hbegp_model* prior, hbegp_model** out, double* lml, void* alpha_out, void* kinv_out,
                       int* appended) {
    if (!ctx || !prior || !prior->m || !out) return fail(HBEGP_ERR_INVALID, "hbegp_model_extend: bad arguments");
    Model* m = nullptr;
    *out = nullptr;
    int rc = ctx->eng->model_extend(prior->m, &m, lml, alpha_out, kinv_out, appended);
    if (rc) return rc;
    *out = new hbegp_model{m};
    return HBEGP_OK;
}

int hbegp_model_destroy(hbegp_model* model) {
    if (!model) return HBEGP_OK;
    if (model->m) {
        if (model->m->eng) {
            cudaSetDevice(model->m->eng->device);
            cudaStreamSynchronize(model->m->eng->stream);
        }
        delete model->m;
    }
    delete model;
    return HBEGP_OK;
}

long hbegp_model_n(const hbegp_model* model) { return (model && model->m) ? model->m->n : 0; }
int hbegp_model_dim(const hbegp_model* model) { return (model && model->m) ? model->m->d : 0; }

int hbegp_predict_warn_values(const hbegp_model* model, int cap, double* values_out, long* rows_out) {
    if (!model || !model->m || cap < 0 || (cap > 0 && !values_out)) return fail(HBEGP_ERR_INVALID, "predict_warn_values: bad arguments");
    const int k = (int)std::min<size_t>((size_t)cap, model->m->last_warn_vals.size());
    for (int i = 0; i < k; i++) {
        values_out[i] = model->m->last_warn_vals[i];
        if (rows_out) rows_out[i] = model->m->last_warn_rows[i];
    }
    return k;
}

int hbegp_kernel_matrix(hbegp_ctx* ctx, double nu, int d, const double* theta, long n1, const void* x1, long n2, const void* x2,
                        void* k_out) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    return ctx->eng->kernel_matrix(nu, d, theta, n1, x1, n2, x2, k_out);
}

int hbegp_kernel_theta_grad(hbegp_ctx* ctx, double nu, int d, const double* theta, long n, const void* x, void* k_out,
                            void* grad_out) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    return ctx->eng->kernel_theta_grad(nu, d, theta, n, x, k_out, grad_out);
}

int hbegp_kernel_diag(int dtype, int d, const double* theta, long n, void* diag_out) {
    // Product<ConstantKernel, Matern>::diag = c * 1 (product_kernel.rs:72-74, constant_kernel.rs:40-42,
    // matern_kernel.rs:137-139); no device work
    if (d <= 0 || !theta || n < 0 || (n > 0 && !diag_out)) return fail(HBEGP_ERR_INVALID, "kernel_diag: bad arguments");
    if (dtype == HBEGP_F64) {
        const double c = std::exp(theta[0]);
        for (long i = 0; i < n; i++) ((double*)diag_out)[i] = c * 1.0;
    } else if (dtype == HBEGP_F32) {
        const float c = (float)std::exp(theta[0]);
        for (long i = 0; i < n; i++) ((float*)diag_out)[i] = c * 1.0f;
    } else {
        return fail(HBEGP_ERR_INVALID, "kernel_diag: bad dtype");
    }
    return HBEGP_OK;
}

int hbegp_lbfgs_set_tolerances(double ftol, double gtol) {
    lbfgs_tolerances().ftol = ftol;
    lbfgs_tolerances().gtol = gtol;
    return HBEGP_OK;
}

int hbegp_predict(hbegp_model* model, long m, const void* xs, void* mean, void* var, long* n_below_warn) {
    if (!model) return fail(HBEGP_ERR_INVALID, "null model");
    if (!model->m->eng) return fail(HBEGP_ERR_INVALID, "the model's context has been destroyed");
    return model->m->predict_host(m, xs, mean, var, n_below_warn);
}

int hbegp_predict_sharded(hbegp_model* model, long m, const void* xs, void* mean, void* var, long* n_below_warn) {
    if (!model || !model->m) return fail(HBEGP_ERR_INVALID, "null model");
    if (!model->m->eng) return fail(HBEGP_ERR_INVALID, "the model's context has been destroyed");
    return model->m->predict_sharded(m, xs, mean, var, n_below_warn);
}

int hbegp_predict_device(hbegp_model* model, long m, const void* xs_device, void* mean_device, void* var_device,
                         long* n_below_warn_device) {
    if (!model) return fail(HBEGP_ERR_INVALID, "null model");
    if (!model->m->eng) return fail(HBEGP_ERR_INVALID, "the model's context has been destroyed");
    return model->m->predict_device(m, xs_device, mean_device, var_device, n_below_warn_device);
}

int hbegp_predict_mean_ei(hbegp_model* model, const hbegp_ynorm* yn, long m, const void* xs, double fmin, void* mean_out,
                          void* ei_out, long* best_index, long* n_below_warn) {
    if (!model) return fail(HBEGP_ERR_INVALID, "null model");
    if (!model->m->eng) return fail(HBEGP_ERR_INVALID, "the model's context has been destroyed");
    return model->m->predict_acquisition(0, yn, m, xs, fmin, mean_out, ei_out, best_index, n_below_warn);
}

int hbegp_predict_confidence_bound(hbegp_model* model, const hbegp_ynorm* yn, long m, const void* xs, double cb, void* out,
                                   long* best_index, long* n_below_warn) {
    if (!model) return fail(HBEGP_ERR_INVALID, "null model");
    if (!model->m->eng) return fail(HBEGP_ERR_INVALID, "the model's context has been destroyed");
    return model->m->predict_acquisition(1, yn, m, xs, cb, out, nullptr, best_index, n_below_warn);
}

int hbegp_minimize_by_gradient(hbegp_objective_fn objective, void* user, int n, double* x, const double* lo,
                               const double* hi, int maxeval, double* f_out) {
    if (!objective || !x || !lo || !hi || n <= 0) return fail(HBEGP_ERR_INVALID, "minimize_by_gradient: bad arguments");
    BoundedLbfgs opt(n, x, lo, hi, maxeval);
    std::vector<double> g(n);
    while (!opt.done()) {
        double f = objective(opt.ask(), g.data(), user);
        opt.tell(f, g.data());
    }
    std::memcpy(x, opt.x(), sizeof(double) * n);
    if (f_out) *f_out = opt.f();
    return opt.evals();
}

void hbegp_rng_seed(unsigned long long seed, unsigned long long state[4]) { Xoshiro256::seed(seed, state); }

void hbegp_rng_fork(unsigned long long state[4], unsigned long long child[4]) {
    Xoshiro256 r;
    std::memcpy(r.s, state, sizeof(r.s));
    for (int i = 0; i < 4; i++) child[i] = r.next();
    std::memcpy(state, r.s, sizeof(r.s));
    if (!(child[0] | child[1] | child[2] | child[3])) Xoshiro256::seed(0, child);
}

double hbegp_rng_uniform(unsigned long long state[4], double lo, double hi) {
    Xoshiro256 r;
    std::memcpy(r.s, state, sizeof(r.s));
    double v = r.uniform_inclusive(lo, hi);
    std::memcpy(state, r.s, sizeof(r.s));
    return v;
}

int hbegp_ynorm_fit(int dtype, int projection, long n, const void* y, const double* known_optimum, void* y_out,
                    hbegp_ynorm* out) {
    if (n <= 0 || !y || !y_out || !out || (projection != HBEGP_PROJ_LINEAR && projection != HBEGP_PROJ_LOG))
        return fail(HBEGP_ERR_INVALID, "ynorm_fit: bad arguments");
    out->dtype = dtype;
    if (dtype == HBEGP_F64) return ynorm_fit_t<double>(projection, n, (const double*)y, known_optimum, (double*)y_out, out);
    if (dtype == HBEGP_F32) return ynorm_fit_t<float>(projection, n, (const float*)y, known_optimum, (float*)y_out, out);
    return fail(HBEGP_ERR_INVALID, "ynorm_fit: bad dtype");
}

int hbegp_ynorm_apply(const hbegp_ynorm* yn, int op, long n, const void* a, const void* b, void* out) {
    if (!yn || n < 0 || op < 0 || op > 4 || (n > 0 && (!a || !out)) || (op >= 2 && n > 0 && !b))
        return fail(HBEGP_ERR_INVALID, "ynorm_apply: bad arguments");
    if (yn->dtype == HBEGP_F64) return ynorm_apply_t<double>(yn, op, n, (const double*)a, (const double*)b, (double*)out);
    return ynorm_apply_t<float>(yn, op, n, (const float*)a, (const float*)b, (float*)out);
}

int hbegp_estimate_amplitude(int dtype, long n, const void* y, const double* bounds, double out[3]) {
    if (n <= 0 || !y || !out) return fail(HBEGP_ERR_INVALID, "estimate_amplitude: bad arguments");
    if (dtype == HBEGP_F64) estimate_amplitude<double>((const double*)y, n, bounds, out);
    else estimate_amplitude<float>((const float*)y, n, bounds, out);
    if (!(out[1] <= out[0] && out[0] <= out[2])) return fail(HBEGP_ERR_INVALID, "estimate_amplitude: start outside bounds (gpr.rs:449 unwrap)");
    return HBEGP_OK;
}

double hbegp_expected_improvement(double mean, double std, double fmin) { return expected_improvement(mean, std, fmin); }

int hbegp_expected_improvement_a(int dtype, long m, const void* mean, const void* var, double fmin, void* ei_out) {
    if (m < 0 || (m > 0 && (!mean || !var || !ei_out))) return fail(HBEGP_ERR_INVALID, "expected_improvement_a: bad arguments");
    if (dtype == HBEGP_F64) {
        const double *mu = (const double*)mean, *v = (const double*)var;
        double* o = (double*)ei_out;
        for (long i = 0; i < m; i++) o[i] = expected_improvement(mu[i], std::sqrt(v[i]), fmin);
    } else {
        const float *mu = (const float*)mean, *v = (const float*)var;
        float* o = (float*)ei_out;
        for (long i = 0; i < m; i++) o[i] = (float)expected_improvement((double)mu[i], (double)std::sqrt(v[i]), fmin);
    }
    return HBEGP_OK;
}

double hbegp_normal_inverse_cdf(double p, double mean, double std) { return mean + std * norm_ppf(p); }

int hbegp_bench_phase(hbegp_ctx* ctx, double nu, int B, const double* theta, int phase, int reps, float* ms_out) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    if (ctx->eng->n <= 0) return fail(HBEGP_ERR_INVALID, "no training data: call hbegp_set_data first");
    return ctx->eng->bench_phase(nu, B, theta, phase, reps, ms_out);
}

int hbegp_debug_poison(hbegp_ctx* ctx) {
    if (!ctx) return fail(HBEGP_ERR_INVALID, "null context");
    return ctx->eng->debug_poison();
}

int hbegp_debug_factor(hbegp_ctx* ctx, double nu, const double* theta, void* k, void* w, void* kinv, int* status) {
    if (!ctx || !theta) return fail(HBEGP_ERR_INVALID, "debug_factor: bad arguments");
    if (ctx->eng->n <= 0) return fail(HBEGP_ERR_INVALID, "no training data: call hbegp_set_data first");
    return ctx->eng->debug_factor(nu, theta, k, w, kinv, status);
}

}  // extern "C"

// =================================================================================== single-process multi-GPU
// The reference is ONE process (src/bin/hbetune/main.rs:255-355), so a drop-in estimator needs a handle that spans the
// GPUs of the box without any help from the host language: hbegp_multi owns one context per device and their NCCL
// communicators.  Work is split only where the path shards (SURVEY 8e): the thetas of a batched evaluation / the live
// runs of a fit round are dealt round-robin to the GPUs and evaluated concurrently (one host thread per GPU; the
// results come back to the one process, so no collective is needed there), candidate rows of a prediction go out in
// contiguous blocks.  What does travel between GPUs travels over NVLink with NCCL on device buffers: the training data
// (ncclBroadcast at set_data) and the fitted model (W = L^-1, alpha, X^T / l: one evaluation on GPU 0, broadcast to the
// replicas -- 134 MB at n = 4096, cheaper than n^3 flops per replica).
struct hbegp_multi {
    std::vector<hbegp_ctx*> ctx;
    std::vector<ncclComm_t> comms;
    int dtype = HBEGP_F64;
};
struct hbegp_multi_model {
    hbegp_multi* mm = nullptr;
    std::vector<hbegp_model*> models;
};

template <typename F>
static int on_all_gpus(int n, F&& f) {  // f(i) -> status, one host thread per GPU; first failure wins
    std::vector<int> rc(n, HBEGP_OK);
    std::vector<std::string> err(n);
    std::vector<std::thread> th;
    for (int i = 1; i < n; i++)
        th.emplace_back([&, i] {
            rc[i] = f(i);
            if (rc[i]) err[i] = g_last_error;
        });
    rc[0] = f(0);
    if (rc[0]) err[0] = g_last_error;
    for (auto& t : th) t.join();
    for (int i = 0; i < n; i++)
        if (rc[i]) return fail(rc[i], "GPU " + std::to_string(i) + ": " + err[i]);
    return HBEGP_OK;
}

extern "C" {

int hbegp_multi_create(int n_gpus, const int* devices, int dtype, hbegp_multi** out) {
    if (!out || n_gpus < 1) return fail(HBEGP_ERR_INVALID, "multi_create: bad arguments");
    *out = nullptr;
    hbegp_multi* mm = new hbegp_multi();
    mm->dtype = dtype;
    std::vector<int> devs(n_gpus);
    for (int i = 0; i < n_gpus; i++) devs[i] = devices ? devices[i] : i;
    for (int i = 0; i < n_gpus; i++) {
        hbegp_ctx* c = nullptr;
        int rc = hbegp_ctx_create(devs[i], dtype, nullptr, &c);
        if (rc) {
            hbegp_multi_destroy(mm);
            return rc;
        }
        mm->ctx.push_back(c);
    }
    if (n_gpus > 1) {
        Nccl& nc = Nccl::get();
        if (!nc.ok()) {
            hbegp_multi_destroy(mm);
            return fail(HBEGP_ERR_CUDA, nc.error);
        }
        mm->comms.assign(n_gpus, nullptr);
        ncclResult_t r = nc.CommInitAll(mm->comms.data(), n_gpus, devs.data());
        if (r != ncclSuccess) {
            mm->comms.clear();
            hbegp_multi_destroy(mm);
            return fail(HBEGP_ERR_CUDA, std::string("ncclCommInitAll: ") + nc.GetErrorString(r));
        }
        for (int i = 0; i < n_gpus; i++) {
            int rc = comm_attach(mm->ctx[i]->eng, mm->comms[i], i, n_gpus);  // the context owns (and destroys) its communicator
            if (rc) {
                hbegp_multi_destroy(mm);
                return rc;
            }
        }
    }
    *out = mm;
    return HBEGP_OK;
}

int hbegp_multi_destroy(hbegp_multi* mm) {
    if (!mm) return HBEGP_OK;
    for (hbegp_ctx* c : mm->ctx) hbegp_ctx_destroy(c);
    delete mm;
    return HBEGP_OK;
}

int hbegp_multi_n_gpus(const hbegp_multi* mm) { return mm ? (int)mm->ctx.size() : 0; }
hbegp_ctx* hbegp_multi_ctx(hbegp_multi* mm, int i) { return (mm && i >= 0 && i < (int)mm->ctx.size()) ? mm->ctx[i] : nullptr; }

// Group-broadcast `bytes` from GPU 0's buffer to every replica's (NCCL over NVLink), then wait for all streams.
static int multi_broadcast(hbegp_multi* mm, const std::vector<void*>& bufs, size_t bytes) {
    const int G = (int)mm->ctx.size();
    if (G == 1 || bytes == 0) return HBEGP_OK;
    Nccl& nc = Nccl::get();
    EngineBase* e0 = mm->ctx[0]->eng;
    CUDA_TRY(cudaSetDevice(e0->device));
    CUDA_TRY(cudaEventRecord(e0->ev_c0, e0->stream));
    NCCL_TRY(nc.GroupStart());
    for (int i = 0; i < G; i++) {
        EngineBase* e = mm->ctx[i]->eng;
        NCCL_TRY(nc.Broadcast(bufs[0], bufs[i], bytes, ncclChar, 0, e->comm, e->stream));
    }
    NCCL_TRY(nc.GroupEnd());
    CUDA_TRY(cudaSetDevice(e0->device));
    CUDA_TRY(cudaEventRecord(e0->ev_c1, e0->stream));
    for (int i = 0; i < G; i++) {
        EngineBase* e = mm->ctx[i]->eng;
        CUDA_TRY(cudaSetDevice(e->device));
        CUDA_TRY(cudaStreamSynchronize(e->stream));
    }
    e0->note_collective();
    return HBEGP_OK;
}

int hbegp_multi_set_data(hbegp_multi* mm, long n, int d, const void* x, const void* y) {
    if (!mm) return fail(HBEGP_ERR_INVALID, "null multi-GPU handle");
    const int G = (int)mm->ctx.size();
    int rc = mm->ctx[0]->eng->set_data(n, d, x, y, false);  // one host-to-device copy ...
    if (rc) return rc;
    std::vector<void*> bx(G), by(G);
    for (int i = 0; i < G; i++) {
        EngineBase* e = mm->ctx[i]->eng;
        if (i > 0 && (rc = e->alloc_data(n, d))) return rc;
        bx[i] = e->dev_x();
        by[i] = e->dev_y();
    }
    const size_t es = mm->ctx[0]->eng->elem_size();
    if ((rc = multi_broadcast(mm, bx, (size_t)n * d * es))) return rc;  // ... then NVLink to the replicas
    return multi_broadcast(mm, by, (size_t)n * es);
}

// B thetas dealt round-robin over the GPUs, evaluated concurrently, results gathered by the host threads.
static int multi_eval(hbegp_multi* mm, double nu, int B, const double* theta, const double* lo, const double* hi, double* lml,
                      double* grad, int* status) {
    const int G = (int)mm->ctx.size();
    if (B <= 0) return HBEGP_OK;
    const int p = mm->ctx[0]->eng->d + 2;
    if (G == 1 || B == 1) return mm->ctx[0]->eng->eval_batch(nu, B, theta, lo, hi, lml, grad, status);
    return on_all_gpus(G, [&](int i) -> int {
        std::vector<int> mine;
        for (int b = i; b < B; b += G) mine.push_back(b);
        const int Bm = (int)mine.size();
        if (!Bm) return HBEGP_OK;
        std::vector<double> th((size_t)Bm * p), l(Bm), g(grad ? (size_t)Bm * p : 0);
        std::vector<int> st(Bm);
        for (int k = 0; k < Bm; k++) std::memcpy(&th[(size_t)k * p], theta + (size_t)mine[k] * p, sizeof(double) * p);
        int rc = mm->ctx[i]->eng->eval_batch(nu, Bm, th.data(), lo, hi, l.data(), grad ? g.data() : nullptr, st.data());
        if (rc) return rc;
        for (int k = 0; k < Bm; k++) {
            lml[mine[k]] = l[k];
            if (status) status[mine[k]] = st[k];
            if (grad) std::memcpy(grad + (size_t)mine[k] * p, &g[(size_t)k * p], sizeof(double) * p);
        }
        return HBEGP_OK;
    });
}

int hbegp_multi_lml_grad_batch(hbegp_multi* mm, double nu, int B, const double* theta, const double* lo, const double* hi,
                               double* lml, double* grad, int* status) {
    if (!mm) return fail(HBEGP_ERR_INVALID, "null multi-GPU handle");
    if (B < 0 || (B > 0 && (!theta || !lml))) return fail(HBEGP_ERR_INVALID, "multi_lml_grad_batch: bad arguments");
    if (mm->ctx[0]->eng->n <= 0) return fail(HBEGP_ERR_INVALID, "no training data: call hbegp_multi_set_data first");
    return multi_eval(mm, nu, B, theta, lo, hi, lml, grad, status);
}

int hbegp_multi_fit_runs(hbegp_multi* mm, double nu, int n_runs, const double* starts, const double* bounds_lo,
                         const double* bounds_hi, int maxeval, hbegp_run_result* results, double* best_theta) {
    if (!mm) return fail(HBEGP_ERR_INVALID, "null multi-GPU handle");
    if (mm->ctx[0]->eng->n <= 0) return fail(HBEGP_ERR_INVALID, "no training data: call hbegp_multi_set_data first");
    BatchEval eval = [&](int B, const double* th, double* lml, double* grad, int* st) {
        return multi_eval(mm, nu, B, th, bounds_lo, bounds_hi, lml, grad, st);
    };
    return fit_runs_impl(mm->ctx[0]->eng->d + 2, eval, n_runs, starts, bounds_lo, bounds_hi, maxeval, 0, 1, nullptr, nullptr, results,
                         best_theta);
}

int hbegp_multi_model_create(hbegp_multi* mm, double nu, const double* theta, const double* lo, const double* hi,
                             hbegp_multi_model** out, double* lml, void* alpha_out, void* kinv_out) {
    if (!mm || !out) return fail(HBEGP_ERR_INVALID, "multi_model_create: bad arguments");
    *out = nullptr;
    const int G = (int)mm->ctx.size();
    hbegp_model* m0 = nullptr;
    int rc = hbegp_model_create(mm->ctx[0], nu, theta, lo, hi, &m0, lml, alpha_out, kinv_out);
    if (rc) return rc;
    hbegp_multi_model* h = new hbegp_multi_model();
    h->mm = mm;
    h->models.push_back(m0);
    Model* src = m0->m;
    for (int i = 1; i < G; i++) {
        Model* r = mm->ctx[i]->eng->new_empty_model(src->nu2, src->prm_h, src->noise_clamped);
        if (!r) {
            hbegp_multi_model_destroy(h);
            return fail(HBEGP_ERR_NOMEM, "multi_model_create: could not allocate the replica on GPU " + std::to_string(i));
        }
        r->np0 = src->np0;
        r->appends = src->appends;
        h->models.push_back(new hbegp_model{r});
    }
    struct Part {
        DevBuf Model::*buf;
        size_t bytes;
    };
    const size_t es = mm->ctx[0]->eng->elem_size(), np = (size_t)src->np;
    const Part parts[] = {{&Model::W, np * np * es}, {&Model::alpha, np * es}, {&Model::xsT, (size_t)src->d * np * es},
                          {&Model::ls, (size_t)src->d * es}, {&Model::ldp, (np / TILE) * es}};
    for (const Part& part : parts) {
        std::vector<void*> bufs(G);
        for (int i = 0; i < G; i++) bufs[i] = (h->models[i]->m->*(part.buf)).p;
        if ((rc = multi_broadcast(mm, bufs, part.bytes))) {
            hbegp_multi_model_destroy(h);
            return rc;
        }
    }
    *out = h;
    return HBEGP_OK;
}

int hbegp_multi_model_destroy(hbegp_multi_model* h) {
    if (!h) return HBEGP_OK;
    for (hbegp_model* m : h->models) hbegp_model_destroy(m);
    delete h;
    return HBEGP_OK;
}

hbegp_model* hbegp_multi_model_replica(hbegp_multi_model* h, int i) {
    return (h && i >= 0 && i < (int)h->models.size()) ? h->models[i] : nullptr;
}

int hbegp_multi_predict(hbegp_multi_model* h, long m, const void* xs, void* mean, void* var, long* n_below_warn) {
    if (!h) return fail(HBEGP_ERR_INVALID, "null multi-GPU model");
    if (m < 0 || (m > 0 && (!xs || !mean))) return fail(HBEGP_ERR_INVALID, "multi_predict: bad arguments");
    if (n_below_warn) *n_below_warn = 0;
    if (m == 0) return HBEGP_OK;
    const int G = (int)h->models.size();
    if (G == 1 || m < 256) return hbegp_predict(h->models[0], m, xs, mean, var, n_below_warn);
    const size_t es = h->mm->ctx[0]->eng->elem_size();
    const int d = h->models[0]->m->d;
    const long blk = (m + G - 1) / G;
    std::vector<long> below(G, 0);
    int rc = on_all_gpus(G, [&](int i) -> int {
        const long r0 = std::min(m, i * blk), cnt = std::min(m, r0 + blk) - r0;
        if (cnt <= 0) return HBEGP_OK;
        return hbegp_predict(h->models[i], cnt, (const char*)xs + (size_t)r0 * d * es, (char*)mean + (size_t)r0 * es,
                             var ? (char*)var + (size_t)r0 * es : nullptr, &below[i]);
    });
    if (rc) return rc;
    if (n_below_warn)
        for (long b : below) *n_below_warn += b;
    return HBEGP_OK;
}

}  // extern "C"
