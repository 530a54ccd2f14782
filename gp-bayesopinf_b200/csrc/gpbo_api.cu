// C ABI of libgpbo.so (see include/gpbo.h): workspace handle, wave scheduling over the
// (GP x start) batch, the lock-step multi-start optimiser driver, and the posterior-moment path.
#include "../../include/gpbo.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <unordered_map>
#include <vector>

#include "kernels_predict.cuh"
#include "kernels_sqrtw.cuh"
#include "kernels_posterior.cuh"
#include "kernels_small.cuh"
#include "lbfgsb.h"

using namespace gpbo;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return fail(GPBO_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));      \
    } while (0)

// Device (cudaMalloc) or pinned host (cudaMallocHost) allocation that only grows and frees itself.  Not copyable: a
// copy would free the same pointer twice.
template <bool Pinned>
struct Buf {
    void* p = nullptr;
    size_t bytes = 0;
    Buf() = default;
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    ~Buf() { release(); }
    cudaError_t ensure(size_t need) {
        if (need <= bytes) return cudaSuccess;
        release();
        cudaError_t e = Pinned ? cudaMallocHost(&p, need) : cudaMalloc(&p, need);
        if (e == cudaSuccess) bytes = need;
        else p = nullptr;
        return e;
    }
    void release() {
        if (p) { if (Pinned) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr; bytes = 0;
    }
    template <class T> T* as() const { return static_cast<T*>(p); }
};
using DevBuf = Buf<false>;
using PinnedBuf = Buf<true>;

struct ProfRec { int cls; cudaEvent_t e0, e1; };

// Optimiser pool: every (GP, start) pair's L-BFGS-B state machine (host side, ~800 B each).
struct OptPool {
    std::vector<gpbo::Lbfgsb> opt;
    long long evals = 0;
    int rounds = 0;
};

// bounds_log [3][2] and opts {factr, pgtol, maxiter, maxfun, maxls} (NULL: scipy's defaults) of the optimiser entry
// points
int parse_lbfgsb_args(const double* bounds_log, const double* opts, LbOptions* o, double lo[3], double hi[3]) {
    for (int i = 0; i < 3; ++i) {
        lo[i] = bounds_log[2 * i];
        hi[i] = bounds_log[2 * i + 1];
        if (!(lo[i] <= hi[i])) return fail(GPBO_EINVAL, "empty bound interval");
    }
    if (opts) {
        o->factr = opts[0]; o->pgtol = opts[1]; o->maxiter = (int)opts[2]; o->maxfun = (int)opts[3]; o->maxls = (int)opts[4];
    }
    return GPBO_OK;
}

// The identity map 0 ... n-1 of pairs to GPs, copied to the device array gp_dev on stream s.  The stream is
// synchronised so that the host vector outlives the copy.
int copy_identity(cudaStream_t s, int* gp_dev, int n) {
    std::vector<int> id(n);
    for (int i = 0; i < n; ++i) id[i] = i;
    CUDA_TRY(cudaMemcpyAsync(gp_dev, id.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

// Run-time switches for A/B measurements and diagnostics (DESIGN.md §11; the defaults are the measured best), read
// once per process.  The on / off switches count as set whatever their value.
struct Switches {
    bool no_tma;          // GPBO_NO_TMA=1: LDGSTS staging instead of TMA in the main loops of the four dominant kernels
    int overlap_max;      // GPBO_OVERLAP_MAX=n: inverse rows on the side stream up to n pairs per wave (0: never; SMs)
    int side_split_div;   // GPBO_SIDE_SPLIT_DIV=k: side-stream split-K partials use 1/k of the SMs (1: bit-identical)
    int split_max;        // GPBO_SPLIT_MAX: split-K policy: most chunks (16),
    int split_min;        // GPBO_SPLIT_MIN: fewest slices per chunk (4),
    bool quant_split;     // GPBO_NO_QUANT_SPLIT=1: quantisation-aware splitting off
    int trtri_lpt;        // GPBO_TRTRI_LPT=0: pair-major instead of longest-first tile order in trtri_row
    bool no_sweep;        // GPBO_NO_SWEEP=1: prediction TRSM by per-column launches instead of the persistent row sweep
    int sweep_mode;       // GPBO_SWEEP_MODE: how the sweeps are cut (cross_sweep_kernel's grid)
    bool no_toeplitz;     // GPBO_NO_TOEPLITZ=1: general K_zz generator even for equispaced estimation grids
    bool ns_plain;        // GPBO_NS_PLAIN=1: unscaled Newton-Schulz iteration
    bool debug_ns;        // GPBO_DEBUG_NS=1: Newton-Schulz residual trace on stderr
    bool small_dbg;       // GPBO_SMALL_DBG=1: per-phase cycle counters of the in-shared small-matrix kernels on stderr
};

const Switches& switches() {
    auto set = [](const char* name) { return std::getenv(name) != nullptr; };
    auto num = [](const char* name, int dflt) { const char* v = std::getenv(name); return v ? std::atoi(v) : dflt; };
    static const Switches sw{set("GPBO_NO_TMA"), num("GPBO_OVERLAP_MAX", -1), std::max(1, num("GPBO_SIDE_SPLIT_DIV", 1)),
                             num("GPBO_SPLIT_MAX", 16), std::max(1, num("GPBO_SPLIT_MIN", 4)), !set("GPBO_NO_QUANT_SPLIT"),
                             num("GPBO_TRTRI_LPT", 1), set("GPBO_NO_SWEEP"), num("GPBO_SWEEP_MODE", 0),
                             set("GPBO_NO_TOEPLITZ"), set("GPBO_NS_PLAIN"), set("GPBO_DEBUG_NS"), set("GPBO_SMALL_DBG")};
    return sw;
}

// ---- run-time values to template arguments: f gets std::integral_constant<int, V> for the first V equal to v, else
// for the last V
template <int V, int... Rest, class F>
decltype(auto) dispatch(int v, F&& f) {
    if constexpr (sizeof...(Rest) == 0) return f(std::integral_constant<int, V>{});
    else return v == V ? f(std::integral_constant<int, V>{}) : dispatch<Rest...>(v, f);
}
template <class F> decltype(auto) with_bool(bool b, F&& f) { return b ? f(std::true_type{}) : f(std::false_type{}); }
template <class F> decltype(auto) with_generator(int gen, F&& f) { return dispatch<0, 1, 2, 3>(gen, f); }
template <class F> decltype(auto) with_family(int fam, F&& f) { return dispatch<0, 3, 5>(fam, f); }
template <class F> decltype(auto) with_small_block(int n, F&& f) { return dispatch<64, 256>(n <= 64 ? 64 : 256, f); }
template <class F> decltype(auto) with_asm_kind(int kind, F&& f) { return dispatch<0, 1, 2, 3, 4, 5, 6>(kind, f); }

// Element generator (AsmSelect index) of the factorisation for RBF order rbf_order (0: sklearn's, 1: rbf_eval's):
// Matern-3/2 (2) and Matern-5/2 (3) always use sklearn's order; only generator 1 works on unscaled abscissae.
int generator(int family, int rbf_order) { return family == 0 ? rbf_order : (family == 3 ? 2 : 3); }

}  // namespace

struct gpbo_ctx {
    int device = 0;
    int family = 0;                  // 0 RBF (the reference's kernel); 3 / 5: Matern nu = 3/2, 5/2
    size_t limit = 0;
    cudaStream_t stream = nullptr;   // used by the *_host entry points
    long long launches = 0;
    bool profiling = false;
    std::vector<ProfRec> recs;
    std::vector<cudaEvent_t> ev_pool;   // recycled timing events: no cudaEventCreate inside a timed region
    int sm_count = 0;
    PinnedBuf h_ns;                     // residual read-back of the Newton-Schulz iteration
    std::vector<cudaEvent_t> ns_events;
    int small_max = SMALL_DEFAULT;      // training sizes up to this run on the in-shared small-matrix path (0: never)
    DevBuf sm_counter, sm_starts, sm_theta, sm_fun, sm_ints, sm_dbg;
    int G_res = 0, m_res = 0;           // shape of the problem resident in t_dev / y_dev (gpbo_problem_upload_host)
    double prof_ms[GPBO_NCLASS] = {0};
    long long prof_n[GPBO_NCLASS] = {0};
    // wave workspace
    DevBuf A, D, DT, ts, z, alpha, pp, logdet, part, status;
    // per-call device copies of host inputs / outputs
    DevBuf t_dev, y_dev, ypad, theta_dev, gpof_dev, lml_dev, grad_dev, st_dev;
    // prediction
    DevBuf X, trow, tsrc, out1, out2, cov_dev, sweep_flags, kzz_tab, kzz_flag;
    // sqrtW (Newton-Schulz)
    DevBuf nsY, nsZ, nsT, nsTT, nsYn, nsZn, nsPart, nsNorm, nsResid, w_dev;
    int w_G = 0, w_n = 0;            // shape of the sqrtW stack currently resident in w_dev
    DevBuf wp_lhs, wp_rhs, wp_olhs, wp_orhs;
    DevBuf pg_gram, pg_proj, pg_regs, pg_means, pg_chol, pg_status, pg_tmp;      // posterior grid (kernels_posterior.cuh)
    // split-K partial tiles (small batches)
    DevBuf pre, pre2;             // pre2: partials of the inverse rows when they run on the side stream
    // side stream + events: in the latency-bound regime (few pairs) the inverse rows W = L^-1 run in the shadow of the
    // factorisation's dependency chain (eval_wave)
    cudaStream_t side = nullptr;
    std::vector<cudaEvent_t> diag_events;
    cudaEvent_t side_done = nullptr;
    DevBuf asm_consts, asm_xs;  // per-matrix constants / scaled abscissae of the stand-alone assembly (asm_prep_kernel)
    // TMA tensor maps of the wave buffers (A, D, DT), re-encoded when a buffer moves or the padded size changes
    TmaMaps tmaps;
    const void* tm_A = nullptr; const void* tm_D = nullptr; const void* tm_DT = nullptr;
    size_t tm_bytes_A = 0, tm_bytes_D = 0;
    int tm_mpad = 0;
    bool tma_ok = false;
    // staging of the pair evaluations (eval_pairs)
    PinnedBuf h_theta, h_lml, h_grad, h_gpof;
    std::unordered_map<const void*, size_t> smem_opted;   // kernel -> dynamic shared memory opted into (smem_opt_in)
};

namespace {

enum { C_PREP = 0, C_DIAG, C_PANEL, C_TRSV, C_TRTRI, C_LAUUM, C_FINAL, C_CROSS, C_SCHUR, C_MEAN, C_ASM, C_SQRTW, C_SMALL, C_STD };

template <class F>
inline void launch(gpbo_ctx* c, int cls, cudaStream_t s, F&& f) {
    if (c->profiling) {
        ProfRec r;
        r.cls = cls;
        cudaEvent_t* ev[2] = {&r.e0, &r.e1};
        for (cudaEvent_t* e : ev) {
            if (c->ev_pool.empty()) cudaEventCreate(e);
            else { *e = c->ev_pool.back(); c->ev_pool.pop_back(); }
        }
        cudaEventRecord(r.e0, s);
        f();
        cudaEventRecord(r.e1, s);
        c->recs.push_back(r);
    } else {
        f();
    }
    c->launches += 1;
}

// A launch with more than 48 KB of dynamic shared memory needs the kernel's opt-in on the device first; call this with
// the kernel just before its launch (and before an occupancy query, which counts 0 resident CTAs without it).  A handle
// belongs to one device, so its own record says what is already set.  The attribute is only ever raised, so another
// handle on the same device cannot lower it under this one.
template <class K>
int smem_opt_in(gpbo_ctx* c, K* kernel, size_t bytes) {
    const void* f = reinterpret_cast<const void*>(kernel);
    if (bytes <= 48 * 1024) return GPBO_OK;
    size_t& opted = c->smem_opted[f];
    if (opted >= bytes) return GPBO_OK;
    cudaFuncAttributes fa;
    CUDA_TRY(cudaFuncGetAttributes(&fa, f));
    if ((size_t)fa.maxDynamicSharedSizeBytes < bytes)
        CUDA_TRY(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    opted = bytes;
    return GPBO_OK;
}

inline int pad_to_tile(int m) { return (m + TB - 1) / TB * TB; }

size_t pair_bytes(int m_pad) {
    const size_t T = m_pad / TB;
    const size_t ntiles = T * (T + 1) / 2;
    return (size_t)m_pad * m_pad * 8 + 2 * T * TB * TB * 8 + 3 * (size_t)m_pad * 8 + T * 8 + ntiles * 32 +
           sizeof(PairParams) + 16;
}

int resolve_limit(gpbo_ctx* c) {
    if (c->limit == 0) {
        size_t fr = 0, tot = 0;
        CUDA_TRY(cudaMemGetInfo(&fr, &tot));
        c->limit = (size_t)(0.8 * (double)fr);
    }
    return GPBO_OK;
}

int sm_count(gpbo_ctx* c) {
    if (c->sm_count == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, c->device) != cudaSuccess || n <= 0) n = 148;
        c->sm_count = n;
    }
    return c->sm_count;
}

// Pairs per wave for `want` pairs: as many as fit the workspace limit, then the `want` pairs are spread evenly over
// the resulting number of waves (2048 pairs at a capacity of 1030 run as 1024 + 1024, not 1030 + 1018), each wave a
// multiple of the SM count when that costs no extra wave (kernels with one CTA per pair then fill whole rounds; at a
// capacity of 1100 on 148 SMs: 1036 + 1012).
int wave_capacity(gpbo_ctx* c, int m_pad, size_t extra_per_pair, size_t reserved, int want) {
    if (resolve_limit(c)) return -1;
    const size_t per = pair_bytes(m_pad) + extra_per_pair;
    if (c->limit <= reserved + per) return 0;
    size_t cap = (c->limit - reserved) / per;
    if (cap >= (size_t)want) return want;
    const size_t nw = ((size_t)want + cap - 1) / cap;
    size_t even = ((size_t)want + nw - 1) / nw;
    const size_t sms = (size_t)sm_count(c);
    const size_t up = (even + sms - 1) / sms * sms;
    if (up <= cap) even = up;
    return (int)even;
}

// ---- workspace accounting ---------------------------------------------------------------------------------
// Every operation sizes its waves as if it owned the whole workspace limit; the large buffers of OTHER operations
// that are still cached (DevBuf never shrinks on its own) are released when the sum would exceed the limit, and a
// buffer of this operation that is larger than now needed is given back if that is what it takes.
struct Need { DevBuf* b; size_t bytes; };

std::vector<DevBuf*> big_buffers(gpbo_ctx* c) {
    return {&c->A, &c->D, &c->DT, &c->X, &c->pre, &c->nsY, &c->nsZ, &c->nsT, &c->nsTT, &c->nsYn, &c->nsZn,
            &c->cov_dev, &c->w_dev, &c->wp_olhs};
}

int fit_buffers(gpbo_ctx* c, cudaStream_t s, const std::vector<Need>& needs) {
    int rc = resolve_limit(c);
    if (rc) return rc;
    auto used = [&](const DevBuf* b) {
        for (const Need& n : needs)
            if (n.b == b) return true;
        return false;
    };
    auto total = [&]() {
        size_t tot = 0;
        for (DevBuf* b : big_buffers(c))
            if (!used(b)) tot += b->bytes;
        for (const Need& n : needs) tot += std::max(n.b->bytes, n.bytes);
        return tot;
    };
    if (total() > c->limit) {
        CUDA_TRY(cudaStreamSynchronize(s));
        for (DevBuf* b : big_buffers(c))
            if (!used(b) && b->bytes) {
                if (b == &c->w_dev) { c->w_G = 0; c->w_n = 0; }     // the resident sqrtW stack is gone
                b->release();
            }
        if (total() > c->limit)
            for (const Need& n : needs)
                if (n.b->bytes > n.bytes) {
                    if (n.b == &c->w_dev) { c->w_G = 0; c->w_n = 0; }
                    n.b->release();
                }
    }
    for (const Need& n : needs) CUDA_TRY(n.b->ensure(n.bytes));
    return GPBO_OK;
}

// extra: further large buffers of the operation (prediction: X; fixed outputs kept alive: cov_dev, w_dev)
int ensure_wave(gpbo_ctx* c, cudaStream_t s, int m_pad, int cap, std::vector<Need> extra = {}) {
    const size_t T = m_pad / TB, ntiles = T * (T + 1) / 2;
    extra.push_back({&c->A, (size_t)cap * m_pad * m_pad * 8});
    extra.push_back({&c->D, (size_t)cap * T * TB * TB * 8});
    extra.push_back({&c->DT, (size_t)cap * T * TB * TB * 8});
    extra.push_back({&c->pre, c->pre.bytes});          // split-K scratch: sized on demand, kept
    int rc0 = fit_buffers(c, s, extra);
    if (rc0) return rc0;
    CUDA_TRY(c->ts.ensure((size_t)cap * m_pad * 8));
    CUDA_TRY(c->z.ensure((size_t)cap * m_pad * 8));
    CUDA_TRY(c->alpha.ensure((size_t)cap * m_pad * 8));
    CUDA_TRY(c->pp.ensure((size_t)cap * sizeof(PairParams)));
    CUDA_TRY(c->logdet.ensure((size_t)cap * T * 8));
    CUDA_TRY(c->part.ensure((size_t)cap * ntiles * 32));
    CUDA_TRY(c->status.ensure((size_t)cap * 4));
    return GPBO_OK;
}

MatArgs mat_args(gpbo_ctx* c, int m, int m_pad) {
    MatArgs a;
    a.A = c->A.as<double>();
    a.mat_stride = (long)m_pad * m_pad;
    a.lda = m_pad;
    a.m = m;
    a.T = m_pad / TB;
    a.D = c->D.as<double>();
    a.DT = c->DT.as<double>();
    a.logdet = c->logdet.as<double>();
    a.status = c->status.as<int>();
    a.pp = c->pp.as<PairParams>();
    a.ts = c->ts.as<double>();
    // trtri rows launch their tiles longest-first: -2.4 % trtri time at 148 pairs, -1.6 % at 256 (m = 8192,
    // profiles/r02c_trtri_order.txt); GPBO_TRTRI_LPT=0 restores the pair-major order
    a.flags = switches().trtri_lpt;
    return a;
}

// ---- TMA tensor maps ------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled is a driver-API entry point; it is fetched through the runtime (no -lcuda at link time).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// 2-D map over `rows` rows of `cols` doubles (row-major, contiguous), box = one operand slice (16 x 128), 128-byte swizzle.
bool encode_slice_map(CUtensorMap* map, void* base, size_t rows, size_t cols) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn || rows == 0 || rows > 0xffffffffull) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)cols * 8};
    const cuuint32_t box[2] = {BK, TB};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// (Re-)encode the maps of the wave buffers.  GPBO_NO_TMA=1 keeps the LDGSTS staging everywhere (A/B measurements).
void update_tma_maps(gpbo_ctx* c, int m_pad) {
    if (switches().no_tma) { c->tma_ok = false; return; }
    if (c->tma_ok && c->tm_A == c->A.p && c->tm_D == c->D.p && c->tm_DT == c->DT.p && c->tm_mpad == m_pad &&
        c->tm_bytes_A == c->A.bytes && c->tm_bytes_D == c->D.bytes)
        return;
    const size_t rows_a = c->A.bytes / ((size_t)m_pad * 8), rows_d = std::min(c->D.bytes, c->DT.bytes) / ((size_t)TB * 8);
    c->tma_ok = encode_slice_map(&c->tmaps.A, c->A.p, rows_a, (size_t)m_pad) &&
                encode_slice_map(&c->tmaps.D, c->D.p, rows_d, TB) && encode_slice_map(&c->tmaps.DT, c->DT.p, rows_d, TB);
    c->tm_A = c->A.p; c->tm_D = c->D.p; c->tm_DT = c->DT.p; c->tm_mpad = m_pad;
    c->tm_bytes_A = c->A.bytes; c->tm_bytes_D = c->D.bytes;
}

// Split-K policy: with fewer than ~one CTA per SM in a launch whose tiles run a k-loop of nk_max slices, the loop
// is cut into up to 16 chunks of >= 4 slices computed by separate CTAs (splitk_partial_kernel) first.
// Returns a PreAcc with buf == nullptr when the fused kernels should run their own loop.
int plan_split(gpbo_ctx* c, cudaStream_t s, const MatArgs& a, int mode, int idx, int nb, int ntile, int nk_max,
               const double* X, long x_stride, PreAcc* out, DevBuf* prebuf = nullptr) {
    if (!prebuf) prebuf = &c->pre;
    const Switches& sw = switches();
    // partials of the side stream (prebuf == pre2) fill only 1/div of the SMs, the rest stays free for the chain
    out->buf = nullptr; out->nsplit = 1; out->chunk = nk_max;
    const int g_sm_count = prebuf == &c->pre2 ? std::max(1, sm_count(c) / sw.side_split_div) : sm_count(c);
    const long units = (long)nb * ntile;
    if (units <= 0 || nk_max < 16) return GPBO_OK;
    // tuning knobs (defaults measured on B200, see DESIGN.md): at most SPLIT_MAX chunks of at least SPLIT_MIN slices
    int nsplit = (int)std::min<long>(sw.split_max, g_sm_count / units);
    nsplit = std::min(nsplit, nk_max / sw.split_min);
    if (nsplit < 2 && units <= 4L * g_sm_count) {
        // between one and a few CTAs per SM the launch is quantised: 256 tiles on 148 SMs take two tile times, 1.73
        // would do.  Cutting every tile into ns k-chunks takes ceil(units ns / SMs) / ns tile times (4 chunks: 1.75);
        // pick the ns that minimises that plus ~2 % per chunk for writing / re-reading the partial accumulators.
        double best = (double)((units + g_sm_count - 1) / g_sm_count);
        int best_ns = 1;
        for (int ns = 2; sw.quant_split && ns <= 8 && nk_max / ns >= 2 * sw.split_min; ++ns) {
            const double cost = (double)((units * ns + g_sm_count - 1) / g_sm_count) / ns + 0.02 * ns;
            if (cost < 0.97 * best) { best = cost; best_ns = ns; }
        }
        nsplit = best_ns;
    }
    if (nsplit < 2) return GPBO_OK;
    const int chunk = (nk_max + nsplit - 1) / nsplit;
    nsplit = (nk_max + chunk - 1) / chunk;
    CUDA_TRY(prebuf->ensure((size_t)units * nsplit * 64 * NTHR * 8));
    if (int rc = smem_opt_in(c, splitk_partial_kernel, MAIN_SMEM)) return rc;
    launch(c, mode == 1 ? C_TRTRI : (mode == 2 ? C_CROSS : C_PANEL), s, [&] {
        splitk_partial_kernel<<<(unsigned)(units * nsplit), NTHR, MAIN_SMEM, s>>>(a, mode, idx, ntile, nsplit, chunk,
                                                                                 prebuf->as<double>(), X, x_stride);
    });
    out->buf = prebuf->as<double>(); out->nsplit = nsplit; out->chunk = chunk;
    return GPBO_OK;
}

// Factor K(theta) for nb pairs and solve for alpha with element generator gen (generator()).
// solve_alpha = false: neither z = L^-1 y nor alpha is computed (the caller gets both from the inverse factor after
// trtri: z_from_inverse_kernel, alpha_from_inverse_kernel).
int factor_wave(gpbo_ctx* c, cudaStream_t s, const MatArgs& a, const double* t_dev, const double* ypad,
                const double* theta_dev, const int* gpof_dev, int nb, int gen, bool solve_alpha = true,
                const cudaEvent_t* diag_events = nullptr) {
    launch(c, C_PREP, s, [&] {
        prep_pairs_kernel<<<nb, 256, 0, s>>>(theta_dev, gpof_dev, t_dev, a.m, a.lda, gen == 1 ? 1 : 0,
                                             c->pp.as<PairParams>(), c->ts.as<double>(), c->status.as<int>(),
                                             a.band ? c->z.as<double>() : nullptr);
    });
    CrossArgs none{nullptr, 0, 0, 0, 0};
    for (int j = 0; j < a.T; ++j) {
        PreAcc pre;
        int rc = plan_split(c, s, a, 0, j, nb, a.T - j, j * (TB / BK), nullptr, 0, &pre);
        if (rc) return rc;
        const TmaMaps& tm = c->tmaps;
        rc = with_generator(gen, [&](auto g) { return with_bool(c->tma_ok, [&](auto tma) {
            auto diag = chol_diag_kernel<g, tma>;
            auto panel = chol_panel_kernel<g, false, tma>;
            if (int e = smem_opt_in(c, diag, MAIN_SMEM + SMEM_ALIGN_PAD)) return e;
            launch(c, C_DIAG, s, [&] { diag<<<nb, NTHR, MAIN_SMEM + SMEM_ALIGN_PAD, s>>>(a, j, pre, tm); });
            if (diag_events) CUDA_TRY(cudaEventRecord(diag_events[j], s));      // L row j, D_j, DT_j are final
            if (j < a.T - 1) {
                const int grid = nb * (a.T - 1 - j);
                if (int e = smem_opt_in(c, panel, TILE_SMEM + SMEM_ALIGN_PAD)) return e;
                launch(c, C_PANEL, s, [&] {
                    panel<<<grid, NTHR, TILE_SMEM + SMEM_ALIGN_PAD, s>>>(a, j, nullptr, 0, 0, none, pre, tm);
                });
            }
            return GPBO_OK;
        }); });
        if (rc) return rc;
    }
    if (solve_alpha) {
        launch(c, C_TRSV, s, [&] { trsv_fwd_kernel<<<nb, TRSV_THR, 0, s>>>(a, ypad, c->z.as<double>()); });
        launch(c, C_TRSV, s, [&] { trsv_bwd_kernel<<<nb, TRSV_THR, 0, s>>>(a, c->z.as<double>(), c->alpha.as<double>()); });
    }
    CUDA_TRY(cudaGetLastError());
    return GPBO_OK;
}

int eval_wave(gpbo_ctx* c, cudaStream_t s, const double* t_dev, const double* ypad, int m, int m_pad,
              const double* theta_dev, const int* gpof_dev, int nb, bool with_grad, double* lml, double* grad,
              int* status) {
    MatArgs a = mat_args(c, m, m_pad);
    // RBF: the factorisation and the inverse rows skip the exactly-zero blocks left of the factor's profile
    // (kernels_chol.cuh, band_first).  The per-block intervals of ts take 2 T of the pair's m_pad = 128 T doubles of z,
    // which holds nothing until z_from_inverse_kernel / trsv_fwd_kernel run after the last of those kernels.
    if (generator(c->family, 0) == 0) a.band = c->z.as<double>();
    update_tma_maps(c, m_pad);
    // Few pairs in flight: the factorisation is a chain of T dependent (partials -> diagonal block -> panel) steps that
    // leaves most SMs idle, and row i of W = L^-1 needs only what exists once diagonal block i is done -- so the inverse
    // rows run on a side stream, each behind the event of "its" diagonal block, in the shadow of the chain (single pair,
    // m = 4096: 8.9 -> 7.4 ms per evaluation; the optimiser's tail is a sequence of such evaluations).  With many pairs
    // every launch fills the GPU and the two streams would only compete, so the rows stay on the main stream.
    // Measured gain at m = 4096: 17 % at 1 pair, 13 % at 8, 6 % at 56, 3 % at 96, 2 % at 148 (one diagonal-block CTA per
    // SM); the default limit is the SM count (profiles/r02d_tail_overlap.txt).
    const int overlap_max = switches().overlap_max >= 0 ? switches().overlap_max : sm_count(c);
    const bool overlap = with_grad && nb <= overlap_max && a.T >= 4;
    if (overlap) {
        if (!c->side) {
            // lowest priority: its CTAs take an SM only when the factorisation chain (on the handle's own stream: highest
            // priority) has none waiting
            int least = 0, greatest = 0;
            CUDA_TRY(cudaDeviceGetStreamPriorityRange(&least, &greatest));
            CUDA_TRY(cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, least));
        }
        if (!c->side_done) CUDA_TRY(cudaEventCreateWithFlags(&c->side_done, cudaEventDisableTiming));
        while ((int)c->diag_events.size() < a.T) {
            cudaEvent_t e;
            CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            c->diag_events.push_back(e);
        }
    }
    int rc = factor_wave(c, s, a, t_dev, ypad, theta_dev, gpof_dev, nb, generator(c->family, 0), !with_grad,
                         overlap ? c->diag_events.data() : nullptr);
    if (rc) return rc;
    const int ntiles = a.T * (a.T + 1) / 2;
    if (with_grad) {
        cudaStream_t st = overlap ? c->side : s;
        for (int i = 1; i < a.T; ++i) {
            if (overlap) CUDA_TRY(cudaStreamWaitEvent(st, c->diag_events[i], 0));
            PreAcc pre;
            rc = plan_split(c, st, a, 1, i, nb, i, i * (TB / BK), nullptr, 0, &pre, overlap ? &c->pre2 : nullptr);
            if (rc) return rc;
            rc = with_bool(c->tma_ok, [&](auto tma) {
                auto row = trtri_row_kernel<tma>;
                if (int e = smem_opt_in(c, row, TILE_SMEM + SMEM_ALIGN_PAD)) return e;
                launch(c, C_TRTRI, st, [&] { row<<<nb * i, NTHR, TILE_SMEM + SMEM_ALIGN_PAD, st>>>(a, i, pre, c->tmaps); });
                return GPBO_OK;
            });
            if (rc) return rc;
        }
        if (overlap) {
            CUDA_TRY(cudaEventRecord(c->side_done, st));
            CUDA_TRY(cudaStreamWaitEvent(s, c->side_done, 0));
        }
        launch(c, C_TRSV, s, [&] { z_from_inverse_kernel<<<nb * a.T, NTHR, 0, s>>>(a, ypad, c->z.as<double>()); });
        launch(c, C_TRSV, s, [&] {
            alpha_from_inverse_kernel<<<nb * a.T, NTHR, 0, s>>>(a, c->z.as<double>(), c->alpha.as<double>());
        });
        rc = with_family(c->family, [&](auto fam) { return with_bool(c->tma_ok, [&](auto tma) {
            auto lauum = lauum_grad_kernel<fam, tma>;
            if (int e = smem_opt_in(c, lauum, MAIN_SMEM + SMEM_ALIGN_PAD)) return e;
            launch(c, C_LAUUM, s, [&] {
                lauum<<<nb * ntiles, NTHR, MAIN_SMEM + SMEM_ALIGN_PAD, s>>>(a, c->alpha.as<double>(), c->part.as<double>(),
                                                                          ntiles, c->tmaps);
            });
            return GPBO_OK;
        }); });
        if (rc) return rc;
    }
    launch(c, C_FINAL, s, [&] {
        finalize_kernel<<<nb, NTHR, 0, s>>>(a, ypad, c->alpha.as<double>(), c->part.as<double>(), ntiles, lml, grad, status,
                                            with_grad ? 1 : 0);
    });
    CUDA_TRY(cudaGetLastError());
    return GPBO_OK;
}

// ---- small-matrix path (kernels_small.cuh) ---------------------------------------------------------------
bool small_path_ok(const gpbo_ctx* c, int m) { return m <= c->small_max && m <= SMALL_MAX; }

// CTAs that can be resident at once for the small kernels (persistent grids are sized to this); the kernel's shared
// memory opt-in must already be in place
template <class K>
int small_resident(gpbo_ctx* c, K kernel, int nt, size_t smem) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, nt, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    return per_sm * sm_count(c);
}

// GPBO_SMALL_DBG=1: per-phase cycle counters of the in-shared kernels, printed to stderr after every launch
long long* small_dbg_begin(gpbo_ctx* c, cudaStream_t s) {
    if (!switches().small_dbg) return nullptr;
    if (c->sm_dbg.ensure(16 * 8) != cudaSuccess) return nullptr;
    cudaMemsetAsync(c->sm_dbg.p, 0, 16 * 8, s);
    return c->sm_dbg.as<long long>();
}
void small_dbg_end(gpbo_ctx* c, cudaStream_t s, const char* what, int m) {
    if (!switches().small_dbg || !c->sm_dbg.p) return;
    long long h[16];
    cudaMemcpyAsync(h, c->sm_dbg.p, sizeof(h), cudaMemcpyDeviceToHost, s);
    cudaStreamSynchronize(s);
    std::fprintf(stderr, "[gpbo small %s m=%d] cycles: fill %lld chol32 %lld panel %lld trailing %lld diaginv %lld "
                         "blockrows %lld z_alpha %lld traces %lld | optimiser %lld over %lld feeds\n",
                 what, m, h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], h[8], h[9]);
}

// LML (+ gradient) of B pairs, one CTA per pair, one launch.  All pointers device.
int small_lml_grad_device(gpbo_ctx* c, cudaStream_t s, const double* t, const double* y, int m, const double* theta,
                          const int* gp_of, int B, double* lml, double* grad, int* status) {
    SmallProblem pr{t, y, m, small_pad(m), small_dbg_begin(c, s)};
    const size_t smem = small_smem_bytes(pr.n);
    int rc = with_small_block(pr.n, [&](auto nt) { return with_family(c->family, [&](auto fam) {
        auto k = small_lml_grad_kernel<nt, fam>;
        if (int e = smem_opt_in(c, k, smem)) return e;
        launch(c, C_SMALL, s, [&] {
            k<<<std::min(B, 8 * small_resident(c, k, nt, smem)), nt.value, smem, s>>>(pr, theta, gp_of, B, lml, grad,
                                                                                      status);
        });
        return GPBO_OK;
    }); });
    if (rc) return rc;
    small_dbg_end(c, s, "lml_grad", m);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

// The whole multi-start fit as one persistent kernel.  t_dev / y_dev hold the problem; starts / gp_of / outputs HOST.
int small_fit_device(gpbo_ctx* c, cudaStream_t s, int G, int m, const double* bounds_log, const double* starts,
                     const int* gp_of, int B, const double* opts, double* theta_opt, double* fun, int* nfev, int* nit,
                     int* opt_status, long long* total_evals, int* rounds) {
    (void)G;
    LbOptions o;
    SmallBox box;
    int rc = parse_lbfgsb_args(bounds_log, opts, &o, box.lo, box.hi);
    if (rc) return rc;
    CUDA_TRY(c->sm_counter.ensure(4));
    CUDA_TRY(c->sm_starts.ensure((size_t)B * 24));
    CUDA_TRY(c->sm_theta.ensure((size_t)B * 24));
    CUDA_TRY(c->sm_fun.ensure((size_t)B * 8));
    CUDA_TRY(c->sm_ints.ensure((size_t)B * 16));
    CUDA_TRY(cudaMemsetAsync(c->sm_counter.p, 0, 4, s));
    CUDA_TRY(cudaMemcpyAsync(c->sm_starts.p, starts, (size_t)B * 24, cudaMemcpyHostToDevice, s));
    int* d_gp = c->sm_ints.as<int>();
    int* d_nfev = d_gp + B;
    int* d_nit = d_nfev + B;
    int* d_st = d_nit + B;
    if (gp_of) {
        CUDA_TRY(cudaMemcpyAsync(d_gp, gp_of, (size_t)B * 4, cudaMemcpyHostToDevice, s));
    } else {
        rc = copy_identity(s, d_gp, B);
        if (rc) return rc;
    }
    SmallProblem pr{c->t_dev.as<double>(), c->y_dev.as<double>(), m, small_pad(m), small_dbg_begin(c, s)};
    const size_t smem = small_smem_bytes(pr.n);
    rc = with_small_block(pr.n, [&](auto nt) { return with_family(c->family, [&](auto fam) {
        auto k = small_fit_kernel<nt, fam>;
        if (int e = smem_opt_in(c, k, smem)) return e;
        launch(c, C_SMALL, s, [&] {
            k<<<std::min(B, small_resident(c, k, nt, smem)), nt.value, smem, s>>>(
                pr, c->sm_starts.as<double>(), d_gp, B, box, o, c->sm_counter.as<int>(), c->sm_theta.as<double>(),
                c->sm_fun.as<double>(), d_nfev, d_nit, d_st);
        });
        return GPBO_OK;
    }); });
    if (rc) return rc;
    small_dbg_end(c, s, "fit", m);
    CUDA_TRY(cudaGetLastError());
    std::vector<int> h_nfev(B), h_nit(B), h_st(B);
    CUDA_TRY(cudaMemcpyAsync(theta_opt, c->sm_theta.p, (size_t)B * 24, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(fun, c->sm_fun.p, (size_t)B * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h_nfev.data(), d_nfev, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h_nit.data(), d_nit, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h_st.data(), d_st, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    long long ev = 0;
    int longest = 0;
    for (int b = 0; b < B; ++b) {
        ev += h_nfev[b];
        longest = std::max(longest, h_nfev[b]);
        if (nfev) nfev[b] = h_nfev[b];
        if (nit) nit[b] = h_nit[b];
        if (opt_status) opt_status[b] = h_st[b];
    }
    if (total_evals) *total_evals = ev;
    if (rounds) *rounds = longest;       // no lock-step here: the longest chain of evaluations of any pair
    return GPBO_OK;
}

int make_ypad(gpbo_ctx* c, cudaStream_t s, const double* y_dev, int G, int m, int m_pad) {
    CUDA_TRY(c->ypad.ensure((size_t)G * m_pad * 8));
    launch(c, C_PREP, s, [&] { pad_rows_kernel<<<G, 256, 0, s>>>(y_dev, m, m_pad, c->ypad.as<double>()); });
    return GPBO_OK;
}

// All pairs, in waves.  All pointers are device pointers.
int lml_grad_device(gpbo_ctx* c, cudaStream_t s, const double* t, const double* y, int G, int m, const double* theta,
                    const int* gp_of, int B, double* lml, double* grad, int* status) {
    if (!c || !t || !y || !theta || !lml || G <= 0 || m <= 0 || B < 0) return fail(GPBO_EINVAL, "lml_grad: bad argument");
    if (B == 0) return GPBO_OK;
    if (!gp_of) return fail(GPBO_EINVAL, "lml_grad: internal: gp_of must be materialised");
    CUDA_TRY(cudaSetDevice(c->device));
    if (small_path_ok(c, m)) return small_lml_grad_device(c, s, t, y, m, theta, gp_of, B, lml, grad, status);
    const int m_pad = pad_to_tile(m);
    const size_t reserved = (size_t)G * m_pad * 8 + (1 << 20);
    const int cap = wave_capacity(c, m_pad, 0, reserved, B);
    if (cap <= 0) return fail(GPBO_ENOMEM, "lml_grad: one pair does not fit the workspace limit");
    int rc = ensure_wave(c, s, m_pad, cap);
    if (rc) return rc;
    rc = make_ypad(c, s, y, G, m, m_pad);
    if (rc) return rc;
    for (int w0 = 0; w0 < B; w0 += cap) {
        const int nb = std::min(cap, B - w0);
        rc = eval_wave(c, s, t, c->ypad.as<double>(), m, m_pad, theta + 3 * (size_t)w0, gp_of + w0, nb,
                       grad != nullptr, lml + w0, grad ? grad + 3 * (size_t)w0 : nullptr, status ? status + w0 : nullptr);
        if (rc) return rc;
    }
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

// sqrtW = (C + eta I)^(-1/2) for G matrices (device pointers); status / iters are HOST arrays (may be NULL).
int sqrtw_device(gpbo_ctx* c, cudaStream_t s, const double* cov, int G, int n, double eta, double* out, int* status,
                 int* iters) {
    CUDA_TRY(cudaSetDevice(c->device));
    int rc = resolve_limit(c);
    if (rc) return rc;
    const int ld = pad_to_tile(n), T = ld / TB, ntiles = T * (T + 1) / 2;
    const size_t mat = (size_t)ld * ld * 8;
    const int nfull = T * T;
    const size_t per = 6 * mat + (size_t)nfull * 8 + 64;
    // the input / output stacks count against the limit when they are the library's own staging buffers
    const bool own_io = (cov == c->cov_dev.as<double>()) && (out == c->w_dev.as<double>());
    const size_t fixed = own_io ? c->cov_dev.bytes + c->w_dev.bytes : 0;
    if (c->limit < fixed + per) return fail(GPBO_ENOMEM, "sqrtw: one matrix does not fit the workspace limit");
    int cap = (int)std::min<size_t>((size_t)G, (c->limit - fixed) / per);
    {
        std::vector<Need> needs = {{&c->nsY, cap * mat}, {&c->nsZ, cap * mat}, {&c->nsT, cap * mat},
                                   {&c->nsTT, cap * mat}, {&c->nsYn, cap * mat}, {&c->nsZn, cap * mat}};
        if (own_io) { needs.push_back({&c->cov_dev, c->cov_dev.bytes}); needs.push_back({&c->w_dev, c->w_dev.bytes}); }
        rc = fit_buffers(c, s, needs);
        if (rc) return rc;
    }
    CUDA_TRY(c->nsPart.ensure((size_t)cap * nfull * 8));
    CUDA_TRY(c->nsNorm.ensure((size_t)cap * 8));
    CUDA_TRY(c->nsResid.ensure((size_t)cap * 8));
    if (int e = smem_opt_in(c, ns_gemm_kernel, MAIN_SMEM)) return e;       // both products of every iteration below
    const int maxit = 90;
    const bool debug_ns = switches().debug_ns;
    const bool plain_ns = switches().ns_plain;       // unscaled iteration (for comparison runs)
    std::vector<double> prev(cap), lk(cap);
    std::vector<char> done(cap);
    // residual read-back: pinned, one slot per iteration, checked ONE iteration late so that the host never drains
    // the GPU queue (iteration k+1's first product is already enqueued when iteration k's residual is looked at)
    CUDA_TRY(c->h_ns.ensure((size_t)(maxit + 1) * cap * 8));
    double* h_ns = c->h_ns.as<double>();
    while ((int)c->ns_events.size() < maxit + 1) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->ns_events.push_back(e);
    }
    for (int w0 = 0; w0 < G; w0 += cap) {
        const int nb = std::min(cap, G - w0);
        const double* Cw = cov + (size_t)w0 * n * n;
        NsArgs a;
        a.Y = c->nsY.as<double>(); a.Z = c->nsZ.as<double>(); a.T = c->nsT.as<double>(); a.TT = c->nsTT.as<double>();
        a.Yn = c->nsYn.as<double>(); a.Zn = c->nsZn.as<double>();
        a.stride = (long)ld * ld; a.ld = ld; a.n = n; a.part = c->nsPart.as<double>();
        unsigned long long* norm = c->nsNorm.as<unsigned long long>();
        CUDA_TRY(cudaMemsetAsync(norm, 0, (size_t)nb * 8, s));
        launch(c, C_SQRTW, s, [&] { ns_norm_kernel<<<dim3((n + 7) / 8, nb), NTHR, 0, s>>>(Cw, n, eta, norm); });
        launch(c, C_SQRTW, s, [&] { ns_init_kernel<<<dim3(ld, nb), NTHR, 0, s>>>(Cw, n, eta, norm, a); });
        // scaling bound l_0 = sqrt(eta / s) per matrix; the batch is stepped with the smallest bound (safe for all)
        double* h_norm = h_ns + (size_t)maxit * cap;
        CUDA_TRY(cudaMemcpyAsync(h_norm, norm, (size_t)nb * 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        double l = 1.0;
        for (int p = 0; p < nb; ++p) {
            const double sp = h_norm[p];
            const double lp = (eta > 0.0 && sp > 0.0 && std::isfinite(sp)) ? std::sqrt(std::min(1.0, eta / sp)) : 1e-8;
            l = std::min(l, std::max(lp, 1e-8));
        }
        if (plain_ns) l = 1.0;
        for (int p = 0; p < nb; ++p) { done[p] = 0; prev[p] = HUGE_VAL; if (status) status[w0 + p] = 0; if (iters) iters[w0 + p] = maxit; }
        // Convergence bookkeeping for the residual of iteration `it`, looked at one iteration late: Y, Z then already
        // hold iterate it + 1, produced with scaling mu_used.  Only an UNSCALED step (mu = 1) is known to improve a
        // nearly converged iterate (E_{k+1} = 3/4 E_k^2 + 1/4 E_k^3); a scaled step deliberately moves eigenvalues
        // near 1 down to the lower bound, so after one nothing is accepted.  Returns whether every matrix is finished
        // and the largest residual of the still running ones.
        auto judge = [&](int it, double mu_used, double* worst) {
            const double* resid = h_ns + (size_t)it * cap;
            bool all_done = true;
            *worst = 0.0;
            if (debug_ns) std::fprintf(stderr, "[gpbo sqrtw] it %d r0 %.6e mu %.6f\n", it, std::sqrt(resid[0]), mu_used);
            for (int p = 0; p < nb; ++p) {
                if (done[p]) continue;
                const double r = std::sqrt(resid[p]);
                if (!std::isfinite(r)) {                       // an eigenvalue <= 0 made Z blow up
                    done[p] = 2;
                } else if (mu_used == 1.0 &&
                           (0.75 * r * r <= 1e-11 * std::sqrt((double)ld) || (prev[p] < 0.05 && r >= 0.25 * prev[p]))) {
                    // converged: the next iterate (already in Y, Z) has a residual <= 0.75 r^2; or the quadratic
                    // phase has stalled at the rounding floor ~ cond * eps -- the reference's eigh result is no
                    // more accurate there
                    done[p] = 1;
                    if (iters) iters[w0 + p] = it + 1;
                }
                prev[p] = r;
                if (!done[p]) { all_done = false; *worst = std::max(*worst, r); }
            }
            return all_done;
        };
        auto fmap = [](double mu, double x) { return 0.5 * mu * x * (3.0 - mu * mu * x * x); };
        double mu_prev = 1.0;
        // a positive definite input is within ||I - T|| < 1 after about log(1 / l_0) / log(2.6) scaled steps; one whose
        // residual is still >= 0.9 long after that has an eigenvalue <= 0 (the reference's ValueError case)
        const int it_hopeless = (int)std::ceil(std::log(1.0 / l) / std::log(2.5)) + 14;
        for (int it = 0; it < maxit; ++it) {
            launch(c, C_SQRTW, s, [&] { ns_gemm_kernel<<<dim3(nb * nfull, 1), NTHR, MAIN_SMEM, s>>>(a, nfull, 0, 0.0, 0.0); });
            launch(c, C_SQRTW, s, [&] { ns_resid_kernel<<<nb, NTHR, 0, s>>>(a.part, nfull, c->nsResid.as<double>()); });
            CUDA_TRY(cudaMemcpyAsync(h_ns + (size_t)it * cap, c->nsResid.p, (size_t)nb * 8, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaEventRecord(c->ns_events[it], s));
            // The first residual is waited for: it decides whether the input needs scaling at all (a well conditioned
            // matrix must not have its eigenvalues near 1 thrown down by a scaled step).  Afterwards the residuals are
            // read ONE iteration late, when the next product is already enqueued: the host never drains the queue.
            double worst = 0.0;
            if (it == 0) {
                CUDA_TRY(cudaEventSynchronize(c->ns_events[0]));
                for (int p = 0; p < nb; ++p) {
                    const double r = std::sqrt(h_ns[p]);
                    worst = std::isfinite(r) ? std::max(worst, r) : HUGE_VAL;
                }
                // spectrum of T_0 within [1 - r, 1 + r] (r = Frobenius norm of I - T): x >= sqrt(1 - r)
                if (worst < 1.0) l = std::max(l, std::sqrt(1.0 - worst));
            } else {
                CUDA_TRY(cudaEventSynchronize(c->ns_events[it - 1]));
                if (judge(it - 1, mu_prev, &worst)) break;    // Y, Z hold iterate `it`: one unscaled step past it - 1
                if (it > it_hopeless && worst >= 0.9) {
                    for (int p = 0; p < nb; ++p)
                        if (!done[p]) done[p] = 2;
                    break;
                }
                // x_{it-1} in [sqrt(1 - r), sqrt(1 + r)] -> after the step with mu_prev: x_it >= min of the images
                if (worst < 1.0) {
                    const double lo = std::min(fmap(mu_prev, std::sqrt(1.0 - worst)),
                                               fmap(mu_prev, std::min(1.0, std::sqrt(1.0 + worst))));
                    if (std::isfinite(lo)) l = std::max(l, std::min(1.0, lo));
                }
            }
            if (it == maxit - 1) {                            // out of iterations: the last residual decides directly
                CUDA_TRY(cudaEventSynchronize(c->ns_events[it]));
                const double* resid = h_ns + (size_t)it * cap;
                for (int p = 0; p < nb; ++p)
                    if (!done[p] && std::sqrt(resid[p]) <= 1e-11 * std::sqrt((double)ld)) done[p] = 1;
                break;
            }
            const double mu = (plain_ns || l > 1.0 - 1e-3) ? 1.0 : std::sqrt(3.0 / (1.0 + l + l * l));
            const double ca = 1.5 * mu, cb = 0.5 * mu * mu * mu;
            l = std::min(1.0, fmap(mu, l));
            mu_prev = mu;
            launch(c, C_SQRTW, s, [&] { ns_gemm_kernel<<<dim3(nb * ntiles, 2), NTHR, MAIN_SMEM, s>>>(a, ntiles, 1, ca, cb); });
            std::swap(a.Y, a.Yn);
            std::swap(a.Z, a.Zn);
        }
        for (int p = 0; p < nb; ++p)
            if (done[p] != 1 && status) status[w0 + p] = 1;
        launch(c, C_SQRTW, s, [&] { ns_out_kernel<<<dim3(n, nb), NTHR, 0, s>>>(a, norm, out + (size_t)w0 * n * n); });
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------
extern "C" {

int gpbo_version(void) { return 100; }
const char* gpbo_last_error(void) { return g_err.c_str(); }

int gpbo_create(gpbo_ctx** out, int device, size_t max_workspace_bytes) {
    if (!out) return fail(GPBO_EINVAL, "gpbo_create: out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(GPBO_ECUDA, std::string("gpbo_create: no CUDA device (") + cudaGetErrorString(e) + ")");
    if (device < 0 || device >= n) return fail(GPBO_EINVAL, "gpbo_create: bad device index");
    CUDA_TRY(cudaSetDevice(device));
    gpbo_ctx* c = new gpbo_ctx();
    c->device = device;
    c->limit = max_workspace_bytes;
    {
        int least = 0, greatest = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CUDA_TRY(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, greatest));
    }
    *out = c;
    return GPBO_OK;
}

int gpbo_destroy(gpbo_ctx* c) {
    if (!c) return GPBO_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto& r : c->recs) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : c->ns_events) cudaEventDestroy(e);
    for (cudaEvent_t e : c->diag_events) cudaEventDestroy(e);
    if (c->side_done) cudaEventDestroy(c->side_done);
    if (c->side) cudaStreamDestroy(c->side);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;                           // the device and pinned buffers free themselves
    return GPBO_OK;
}

long long gpbo_launch_count(const gpbo_ctx* c) { return c ? c->launches : 0; }

int gpbo_set_kernel_family(gpbo_ctx* c, int twice_nu) {
    if (!c) return fail(GPBO_EINVAL, "set_kernel_family: ctx is NULL");
    if (twice_nu != 0 && twice_nu != 3 && twice_nu != 5)
        return fail(GPBO_EINVAL, "set_kernel_family: 0 (RBF), 3 (Matern-3/2) or 5 (Matern-5/2)");
    c->family = twice_nu;
    return GPBO_OK;
}

int gpbo_get_stream(gpbo_ctx* c, void** stream) {
    if (!c || !stream) return fail(GPBO_EINVAL, "get_stream: bad argument");
    *stream = static_cast<void*>(c->stream);
    return GPBO_OK;
}

int gpbo_set_small_path(gpbo_ctx* c, int max_m) {
    if (!c || max_m < 0) return fail(GPBO_EINVAL, "set_small_path: bad argument");
    c->small_max = std::min(max_m, (int)SMALL_MAX);
    return GPBO_OK;
}

int gpbo_wave_capacity(gpbo_ctx* c, int m) {
    if (!c || m <= 0) return fail(GPBO_EINVAL, "wave_capacity: bad argument");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(GPBO_ECUDA, "cudaSetDevice failed");
    return wave_capacity(c, pad_to_tile(m), 0, 1 << 20, 1 << 30);
}

int gpbo_profile_enable(gpbo_ctx* c, int on) {
    if (!c) return fail(GPBO_EINVAL, "profile_enable: ctx is NULL");
    for (auto& r : c->recs) { c->ev_pool.push_back(r.e0); c->ev_pool.push_back(r.e1); }
    c->recs.clear();
    for (int i = 0; i < GPBO_NCLASS; ++i) { c->prof_ms[i] = 0; c->prof_n[i] = 0; }
    c->profiling = on != 0;
    return GPBO_OK;
}

int gpbo_profile_get(gpbo_ctx* c, double* ms, long long* launches) {
    if (!c || !ms || !launches) return fail(GPBO_EINVAL, "profile_get: bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaDeviceSynchronize());
    for (auto& r : c->recs) {
        float f = 0.f;
        cudaEventElapsedTime(&f, r.e0, r.e1);
        c->prof_ms[r.cls] += f;
        c->prof_n[r.cls] += 1;
        c->ev_pool.push_back(r.e0);
        c->ev_pool.push_back(r.e1);
    }
    c->recs.clear();
    for (int i = 0; i < GPBO_NCLASS; ++i) { ms[i] = c->prof_ms[i]; launches[i] = c->prof_n[i]; }
    return GPBO_OK;
}

static int assemble_impl(gpbo_ctx* c, int fam, int kind, const double* t1, long t1_stride, int n1, const double* t2,
                         long t2_stride, int n2, const double* theta, int B, double* out, void* stream) {
    if (!c || !t1 || !t2 || !theta || !out || n1 <= 0 || n2 <= 0 || B <= 0 || kind < 0 || kind > 6)
        return fail(GPBO_EINVAL, "assemble: bad argument");
    if (fam != 0 && fam != 3 && fam != 5) return fail(GPBO_EINVAL, "assemble: twice_nu must be 3 or 5");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const long os = (long)n1 * n2;
    const bool sym = (t1 == t2 && t1_stride == t2_stride && n1 == n2);
    if ((kind == 0 || kind == 1) && n1 != n2) return fail(GPBO_EINVAL, "assemble: the train kinds 0 / 1 need n1 == n2");
    const bool scaled = fam != 0 || kind == 0 || kind == 2 || kind == 6;       // AsmScaled: the generator works on t / ell
    CUDA_TRY(c->asm_consts.ensure((size_t)B * sizeof(AsmConsts)));
    if (scaled) CUDA_TRY(c->asm_xs.ensure((size_t)B * ((size_t)n1 + (sym ? 0 : n2)) * 8));
    const AsmConsts* kc = c->asm_consts.as<AsmConsts>();
    double* xs1 = c->asm_xs.as<double>();
    double* xs2 = sym ? xs1 : xs1 + (size_t)B * n1;
    const double* a1 = scaled ? xs1 : t1;
    const double* a2 = scaled ? xs2 : t2;
    const long s1 = scaled ? n1 : t1_stride, s2 = scaled ? n2 : t2_stride;
    // threads per CTA of the general kernel: one per column pair, 64 ... 256
    const int gthr = std::min(NTHR, std::max(64, ((n2 + 1) / 2 + 31) / 32 * 32));
    const int nt = (n1 + SYM_T - 1) / SYM_T;
    const dim3 gs(nt * (nt + 1) / 2, B);
    const dim3 gg((n2 + 2 * gthr - 1) / (2 * gthr), (n1 + ASM_ROWS - 1) / ASM_ROWS, B);
    int rc = with_family(fam, [&](auto f) { return with_asm_kind(kind, [&](auto k) {
        auto sym_kernel = assemble_sym2_kernel<f, k>;
        if (int e = sym ? smem_opt_in(c, sym_kernel, SYM2_SMEM) : GPBO_OK) return e;
        launch(c, C_ASM, s, [&] {   // one record for the pre-pass, the assembly and the diagonal
            asm_prep_kernel<<<dim3((std::max(n1, n2) + 255) / 256, B), 256, 0, s>>>(
                theta, t1, t1_stride, n1, t2, t2_stride, n2, scaled, sym, c->asm_consts.as<AsmConsts>(), xs1, xs2);
            if (sym) sym_kernel<<<gs, NTHR, SYM2_SMEM, s>>>(a1, s1, n1, kc, out, os);
            else assemble_general_kernel<f, k><<<gg, gthr, 0, s>>>(a1, s1, n1, a2, s2, n2, kc, out, os);
            if (!sym && (kind == 0 || kind == 1)) asm_diag_kernel<<<dim3((n1 + 255) / 256, B), 256, 0, s>>>(kc, n1, out, os);
        });
        return GPBO_OK;
    }); });
    if (rc) return rc;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

int gpbo_assemble(gpbo_ctx* c, int kind, const double* t1, long t1_stride, int n1, const double* t2, long t2_stride,
                  int n2, const double* theta, int B, double* out, void* stream) {
    return assemble_impl(c, 0, kind, t1, t1_stride, n1, t2, t2_stride, n2, theta, B, out, stream);
}

int gpbo_assemble_matern(gpbo_ctx* c, int twice_nu, int kind, const double* t1, long t1_stride, int n1, const double* t2,
                         long t2_stride, int n2, const double* theta, int B, double* out, void* stream) {
    if (twice_nu != 3 && twice_nu != 5) return fail(GPBO_EINVAL, "assemble_matern: twice_nu must be 3 or 5");
    return assemble_impl(c, twice_nu, kind, t1, t1_stride, n1, t2, t2_stride, n2, theta, B, out, stream);
}

int gpbo_lml_grad(gpbo_ctx* c, const double* t, const double* y, int G, int m, const double* theta, const int* gp_of,
                  int B, double* lml, double* grad, int* status, void* stream) {
    if (!c) return fail(GPBO_EINVAL, "lml_grad: ctx is NULL");
    if (!gp_of && B != G) return fail(GPBO_EINVAL, "lml_grad: gp_of is NULL but B != G");
    if (!gp_of) {
        // identity map: materialise it so waves can be sliced uniformly (copied on the caller's stream, so it is
        // ordered against earlier work of a non-blocking stream)
        CUDA_TRY(cudaSetDevice(c->device));
        CUDA_TRY(c->gpof_dev.ensure((size_t)B * 4));
        int rc = copy_identity(static_cast<cudaStream_t>(stream), c->gpof_dev.as<int>(), B);
        if (rc) return rc;
        gp_of = c->gpof_dev.as<int>();
    }
    return lml_grad_device(c, static_cast<cudaStream_t>(stream), t, y, G, m, theta, gp_of, B, lml, grad, status);
}

static bool all_finite(const double* v, size_t n) {
    for (size_t i = 0; i < n; ++i)
        if (!std::isfinite(v[i])) return false;
    return true;
}

// Host inputs are validated like scikit-learn validates X and y (GaussianProcessRegressor.fit -> validate_data):
// the kernels' exp fast path maps a NaN abscissa to a finite element instead of propagating it.
static int upload_problem(gpbo_ctx* c, cudaStream_t s, const double* t, const double* y, int G, int m) {
    if (!all_finite(t, (size_t)G * m) || !all_finite(y, (size_t)G * m))
        return fail(GPBO_EINVAL, "input contains NaN or infinity (t or y)");
    c->G_res = 0; c->m_res = 0;       // t_dev / y_dev are about to change: a resident problem is no longer valid
    CUDA_TRY(c->t_dev.ensure((size_t)G * m * 8));
    CUDA_TRY(c->y_dev.ensure((size_t)G * m * 8));
    CUDA_TRY(cudaMemcpyAsync(c->t_dev.p, t, (size_t)G * m * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(c->y_dev.p, y, (size_t)G * m * 8, cudaMemcpyHostToDevice, s));
    return GPBO_OK;
}

// LML (+ gradient; grad == NULL: the LML-only path) of n pairs against the problem in t_dev / y_dev (G GPs of m
// points).  theta [n][3] and gp_of [n] (NULL: pair b uses GP b) are HOST inputs staged through the pinned h_* buffers;
// lml [n], grad [n][3] and status [n] (may be NULL) are HOST outputs.
static int eval_pairs(gpbo_ctx* c, cudaStream_t s, int G, int m, const double* theta, const int* gp_of, int n,
                      double* lml, double* grad, int* status) {
    CUDA_TRY(c->h_theta.ensure((size_t)n * 24));
    CUDA_TRY(c->h_gpof.ensure((size_t)n * 4));
    CUDA_TRY(c->h_lml.ensure((size_t)n * 8));
    CUDA_TRY(c->h_grad.ensure((size_t)n * 24));
    CUDA_TRY(c->theta_dev.ensure((size_t)n * 24));
    CUDA_TRY(c->gpof_dev.ensure((size_t)n * 4));
    CUDA_TRY(c->lml_dev.ensure((size_t)n * 8));
    CUDA_TRY(c->grad_dev.ensure((size_t)n * 24));
    CUDA_TRY(c->st_dev.ensure((size_t)n * 4));
    std::memcpy(c->h_theta.p, theta, (size_t)n * 24);
    CUDA_TRY(cudaMemcpyAsync(c->theta_dev.p, c->h_theta.p, (size_t)n * 24, cudaMemcpyHostToDevice, s));
    if (gp_of) {
        std::memcpy(c->h_gpof.p, gp_of, (size_t)n * 4);
        CUDA_TRY(cudaMemcpyAsync(c->gpof_dev.p, c->h_gpof.p, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    } else if (int rc = copy_identity(s, c->gpof_dev.as<int>(), n)) {
        return rc;
    }
    int rc = lml_grad_device(c, s, c->t_dev.as<double>(), c->y_dev.as<double>(), G, m, c->theta_dev.as<double>(),
                             c->gpof_dev.as<int>(), n, c->lml_dev.as<double>(), grad ? c->grad_dev.as<double>() : nullptr,
                             c->st_dev.as<int>());
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->h_lml.p, c->lml_dev.p, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    if (grad) CUDA_TRY(cudaMemcpyAsync(c->h_grad.p, c->grad_dev.p, (size_t)n * 24, cudaMemcpyDeviceToHost, s));
    if (status) CUDA_TRY(cudaMemcpyAsync(status, c->st_dev.p, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    std::memcpy(lml, c->h_lml.p, (size_t)n * 8);
    if (grad) std::memcpy(grad, c->h_grad.p, (size_t)n * 24);
    return GPBO_OK;
}

int gpbo_lml_grad_host(gpbo_ctx* c, const double* t, const double* y, int G, int m, const double* theta,
                       const int* gp_of, int B, double* lml, double* grad, int* status) {
    if (!c || !t || !y || !theta || !lml || G <= 0 || m <= 0 || B <= 0)
        return fail(GPBO_EINVAL, "lml_grad_host: bad argument");
    if (!gp_of && B != G) return fail(GPBO_EINVAL, "lml_grad_host: gp_of is NULL but B != G");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    int rc = upload_problem(c, s, t, y, G, m);
    if (rc) return rc;
    if (gp_of)
        for (int b = 0; b < B; ++b)
            if (gp_of[b] < 0 || gp_of[b] >= G) return fail(GPBO_EINVAL, "gp_of entry out of range");
    return eval_pairs(c, s, G, m, theta, gp_of, B, lml, grad, status);
}

static int pool_init(OptPool& pool, int B, const double* bounds_log, const double* starts, const double* opts) {
    LbOptions o;
    double lo[3], hi[3];
    int rc = parse_lbfgsb_args(bounds_log, opts, &o, lo, hi);
    if (rc) return rc;
    pool.opt.assign(B, Lbfgsb());
    for (int b = 0; b < B; ++b) pool.opt[b].init(starts + 3 * (size_t)b, lo, hi, o);
    pool.evals = 0;
    pool.rounds = 0;
    return GPBO_OK;
}

// The running pairs' indices idx[n] and trial points theta[n][3]; returns n.
static int pool_live(const OptPool& pool, int* idx, double* theta) {
    int n = 0;
    const int B = (int)pool.opt.size();
    for (int b = 0; b < B; ++b) {
        const Lbfgsb& o = pool.opt[b];
        if (!o.running()) continue;
        idx[n] = b;
        theta[3 * n] = o.x[0]; theta[3 * n + 1] = o.x[1]; theta[3 * n + 2] = o.x[2];
        ++n;
    }
    return n;
}

static int pool_feed(OptPool& pool, int n, const int* idx, const double* lml, const double* grad) {
    const int B = (int)pool.opt.size();
    for (int k = 0; k < n; ++k) {
        const int b = idx[k];
        if (b < 0 || b >= B || !pool.opt[b].running()) return fail(GPBO_EINVAL, "optpool_feed: pair is not running");
        double gneg[3] = {-grad[3 * k], -grad[3 * k + 1], -grad[3 * k + 2]};
        pool.opt[b].feed(-lml[k], gneg);         // obj_func = (-lml, -grad), _gpr.py:300-307
    }
    pool.evals += n;
    if (n > 0) pool.rounds += 1;
    return GPBO_OK;
}

static void pool_result(const OptPool& pool, double* theta_opt, double* fun, int* nfev, int* nit, int* opt_status,
                        long long* total_evals, int* rounds) {
    const int B = (int)pool.opt.size();
    for (int b = 0; b < B; ++b) {
        const Lbfgsb& o = pool.opt[b];
        o.current_best(theta_opt + 3 * (size_t)b, fun + b);
        if (nfev) nfev[b] = o.nfev;
        if (nit) nit[b] = o.nit;
        if (opt_status) opt_status[b] = o.status;
    }
    if (total_evals) *total_evals = pool.evals;
    if (rounds) *rounds = pool.rounds;
}

int gpbo_fit_host(gpbo_ctx* c, const double* t, const double* y, int G, int m, const double* bounds_log,
                  const double* starts, const int* gp_of, int B, const double* opts, double* theta_opt, double* fun,
                  int* nfev, int* nit, int* opt_status, long long* total_evals, int* rounds) {
    if (!c || !t || !y || !bounds_log || !starts || !theta_opt || !fun || G <= 0 || m <= 0 || B <= 0)
        return fail(GPBO_EINVAL, "fit_host: bad argument");
    if (!gp_of && B != G) return fail(GPBO_EINVAL, "fit_host: gp_of is NULL but B != G");
    if (gp_of)
        for (int b = 0; b < B; ++b)
            if (gp_of[b] < 0 || gp_of[b] >= G) return fail(GPBO_EINVAL, "fit_host: gp_of entry out of range");
    OptPool pool;
    int rc = pool_init(pool, B, bounds_log, starts, opts);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    rc = upload_problem(c, s, t, y, G, m);
    if (rc) return rc;
    if (small_path_ok(c, m)) {
        // reference-size problems: the whole multi-start fit runs as ONE persistent kernel, optimiser on device
        rc = small_fit_device(c, s, G, m, bounds_log, starts, gp_of, B, opts, theta_opt, fun, nfev, nit, opt_status,
                              total_evals, rounds);
        return rc;
    }
    std::vector<int> idx(B), gp(B);
    std::vector<double> theta(3 * (size_t)B), lml(B), grad(3 * (size_t)B);
    for (int n; (n = pool_live(pool, idx.data(), theta.data())) > 0;) {
        for (int k = 0; k < n; ++k) gp[k] = gp_of ? gp_of[idx[k]] : idx[k];
        rc = eval_pairs(c, s, G, m, theta.data(), gp.data(), n, lml.data(), grad.data(), nullptr);
        if (rc) return rc;
        rc = pool_feed(pool, n, idx.data(), lml.data(), grad.data());
        if (rc) return rc;
    }
    pool_result(pool, theta_opt, fun, nfev, nit, opt_status, total_evals, rounds);
    return GPBO_OK;
}

// ---- optimiser pool + resident problem: the pieces of gpbo_fit_host, exposed so that a multi-GPU driver can
// interleave one all-gather per lock-step round (sharding.py) ------------------------------------------------
struct gpbo_optpool { OptPool pool; };

int gpbo_optpool_create(gpbo_optpool** out, int B, const double* bounds_log, const double* starts, const double* opts) {
    if (!out || B <= 0 || !bounds_log || !starts) return fail(GPBO_EINVAL, "optpool_create: bad argument");
    gpbo_optpool* h = new gpbo_optpool();
    int rc = pool_init(h->pool, B, bounds_log, starts, opts);
    if (rc) { delete h; return rc; }
    *out = h;
    return GPBO_OK;
}

int gpbo_optpool_destroy(gpbo_optpool* h) {
    delete h;
    return GPBO_OK;
}

int gpbo_optpool_live(gpbo_optpool* h, int* idx, double* theta, int* n_live) {
    if (!h || !idx || !theta || !n_live) return fail(GPBO_EINVAL, "optpool_live: bad argument");
    *n_live = pool_live(h->pool, idx, theta);
    return GPBO_OK;
}

int gpbo_optpool_feed(gpbo_optpool* h, int n, const int* idx, const double* lml, const double* grad) {
    if (!h || n < 0 || (n > 0 && (!idx || !lml || !grad))) return fail(GPBO_EINVAL, "optpool_feed: bad argument");
    return pool_feed(h->pool, n, idx, lml, grad);
}

int gpbo_optpool_result(gpbo_optpool* h, double* theta_opt, double* fun, int* nfev, int* nit, int* opt_status,
                        long long* total_evals, int* rounds) {
    if (!h || !theta_opt || !fun) return fail(GPBO_EINVAL, "optpool_result: bad argument");
    pool_result(h->pool, theta_opt, fun, nfev, nit, opt_status, total_evals, rounds);
    return GPBO_OK;
}

int gpbo_problem_upload_host(gpbo_ctx* c, const double* t, const double* y, int G, int m) {
    if (!c || !t || !y || G <= 0 || m <= 0) return fail(GPBO_EINVAL, "problem_upload_host: bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    int rc = upload_problem(c, c->stream, t, y, G, m);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->G_res = G; c->m_res = m;
    return GPBO_OK;
}

int gpbo_lml_grad_resident_host(gpbo_ctx* c, const double* theta, const int* gp_of, int B, double* lml, double* grad,
                                int* status) {
    if (!c || !theta || !gp_of || !lml || !grad || B < 0) return fail(GPBO_EINVAL, "lml_grad_resident_host: bad argument");
    if (c->G_res <= 0) return fail(GPBO_EINVAL, "lml_grad_resident_host: no resident problem (gpbo_problem_upload_host)");
    if (B == 0) return GPBO_OK;
    for (int b = 0; b < B; ++b)
        if (gp_of[b] < 0 || gp_of[b] >= c->G_res) return fail(GPBO_EINVAL, "lml_grad_resident_host: gp_of entry out of range");
    CUDA_TRY(cudaSetDevice(c->device));
    return eval_pairs(c, c->stream, c->G_res, c->m_res, theta, gp_of, B, lml, grad, status);
}

int gpbo_lbfgsb_minimize(gpbo_objective_fn fn, void* user, const double* x0, const double* bounds_log,
                         const double* opts, double* x, double* f, int* nfev, int* nit, int* status) {
    if (!fn || !x0 || !bounds_log || !x || !f) return fail(GPBO_EINVAL, "lbfgsb_minimize: bad argument");
    LbOptions o;
    double lo[3], hi[3];
    int rc = parse_lbfgsb_args(bounds_log, opts, &o, lo, hi);
    if (rc) return rc;
    Lbfgsb opt;
    opt.init(x0, lo, hi, o);
    while (opt.running()) {
        double g[3];
        const double fv = fn(opt.x, g, user);
        opt.feed(fv, g);
    }
    for (int i = 0; i < 3; ++i) x[i] = opt.x[i];
    *f = opt.f;
    if (nfev) *nfev = opt.nfev;
    if (nit) *nit = opt.nit;
    if (status) *status = opt.status;
    return GPBO_OK;
}

// Posterior moments for G GPs (pairs == GPs).  mode 0: predict (mean, std; sklearn order);
// mode 1: lstsq (state, ddt, cov; rbf_eval order).  All pointers device.
static int moments_device(gpbo_ctx* c, cudaStream_t s, int mode, const double* t, const double* y, int G, int m,
                          const double* theta, const double* trow_src, long src_stride, int n, double* out1,
                          double* out2, double* cov, double* alpha_out, int* status) {
    CUDA_TRY(cudaSetDevice(c->device));
    const int m_pad = pad_to_tile(m), n_pad = pad_to_tile(n), xT = n_pad / TB;
    const bool need_x = (mode == 0) || (cov != nullptr);
    const size_t extra = (need_x ? (size_t)n_pad * m_pad * 8 : 0) + (size_t)n_pad * 8;
    // the covariance output (when it is the library's own staging buffer) lives beside the waves
    const bool own_cov = cov && cov == c->cov_dev.as<double>();
    const size_t reserved = (size_t)G * m_pad * 8 + (1 << 20) + (own_cov ? c->cov_dev.bytes : 0);
    const int cap = wave_capacity(c, m_pad, extra, reserved, G);
    if (cap <= 0) return fail(GPBO_ENOMEM, "moments: one GP does not fit the workspace limit");
    std::vector<Need> more;
    if (need_x) more.push_back({&c->X, (size_t)cap * n_pad * m_pad * 8});
    if (own_cov) more.push_back({&c->cov_dev, c->cov_dev.bytes});
    int rc = ensure_wave(c, s, m_pad, cap, more);
    if (rc) return rc;
    CUDA_TRY(c->trow.ensure((size_t)cap * n_pad * 8));
    CUDA_TRY(c->gpof_dev.ensure((size_t)G * 4));
    rc = copy_identity(s, c->gpof_dev.as<int>(), G);
    if (rc) return rc;
    rc = make_ypad(c, s, y, G, m, m_pad);
    if (rc) return rc;
    const int gen = generator(c->family, mode == 0 ? 0 : 1);
    const int order = gen == 1 ? 1 : 0;        // abscissae order of the evaluation points, as of the training points
    MatArgs a = mat_args(c, m, m_pad);
    update_tma_maps(c, m_pad);
    for (int w0 = 0; w0 < G; w0 += cap) {
        const int nb = std::min(cap, G - w0);
        rc = factor_wave(c, s, a, t, c->ypad.as<double>(), theta + 3 * (size_t)w0, c->gpof_dev.as<int>() + w0, nb, gen);
        if (rc) return rc;
        launch(c, C_PREP, s, [&] {
            scale_rows_kernel<<<nb, 256, 0, s>>>(trow_src + (size_t)w0 * src_stride, src_stride, n, n_pad, order,
                                                 c->pp.as<PairParams>(), c->trow.as<double>());
        });
        CrossArgs cr{c->trow.as<double>(), n, n_pad, mode == 0 ? 0 : 1, c->family};
        dim3 mgrid((n + NTHR / 32 - 1) / (NTHR / 32), nb);
        launch(c, C_MEAN, s, [&] {
            mean_kernel<<<mgrid, NTHR, 0, s>>>(a, cr, c->alpha.as<double>(), out1 + (size_t)w0 * n, n);
        });
        if (mode == 1) {
            CrossArgs cr2 = cr;
            cr2.kind = 2;
            launch(c, C_MEAN, s, [&] {
                mean_kernel<<<mgrid, NTHR, 0, s>>>(a, cr2, c->alpha.as<double>(), out2 + (size_t)w0 * n, n);
            });
        }
        if (need_x) {
            CrossArgs crx = cr;
            crx.kind = mode == 0 ? 0 : 2;
            const long xs = (long)n_pad * m_pad;
            const int units = nb * xT;
            if (!switches().no_sweep && 2 * units >= sm_count(c)) {
                // enough row tiles to fill the GPU: one persistent launch, the sweeps cut into equal cost ranges
                CUDA_TRY(c->sweep_flags.ensure((size_t)units * 4));
                CUDA_TRY(cudaMemsetAsync(c->sweep_flags.p, 0, (size_t)units * 4, s));
                // grid: GPBO_SWEEP_MODE 0 (default): one CTA per SM, the sweeps cut along j into equal cost ranges;
                // 1: whole units only, spread evenly (256 units -> 128 CTAs x 2, all CTAs in lock-step over j).
                // Measured on 8 GPs x m = m' = 4096: 19.0 ms (0.78 of the DMMA peak) against 22.0 ms (0.67).
                const int rounds = (units + sm_count(c) - 1) / sm_count(c);
                const int grid = switches().sweep_mode == 0 ? std::min(units, sm_count(c)) : (units + rounds - 1) / rounds;
                if (int e = smem_opt_in(c, cross_sweep_kernel, TILE_SMEM)) return e;
                launch(c, C_CROSS, s, [&] {
                    cross_sweep_kernel<<<grid, NTHR, TILE_SMEM, s>>>(a, c->X.as<double>(), xs, xT, units, crx,
                                                                     c->sweep_flags.as<int>());
                });
            } else {
                for (int j = 0; j < a.T; ++j) {
                    PreAcc pre;
                    rc = plan_split(c, s, a, 2, j, nb, xT, j * (TB / BK), c->X.as<double>(), xs, &pre);
                    if (rc) return rc;
                    // the prediction instance exists for generator 0 and LDGSTS staging only
                    auto panel = chol_panel_kernel<0, true, false>;
                    if (int e = smem_opt_in(c, panel, TILE_SMEM + SMEM_ALIGN_PAD)) return e;
                    launch(c, C_CROSS, s, [&] {
                        panel<<<nb * xT, NTHR, TILE_SMEM + SMEM_ALIGN_PAD, s>>>(a, j, c->X.as<double>(), xs, xT, crx, pre,
                                                                              c->tmaps);
                    });
                }
            }
            if (mode == 0) {
                launch(c, C_STD, s, [&] {
                    std_kernel<<<mgrid, NTHR, 0, s>>>(a, c->X.as<double>(), xs, n, out2 + (size_t)w0 * n, n);
                });
            } else {
                const int ntiles = xT * (xT + 1) / 2;
                // N2: equispaced estimation points -> K_zz from a per-GP table of m' values indexed by the lag
                double* ktab = nullptr;
                int* kflag = nullptr;
                if (!switches().no_toeplitz) {
                    CUDA_TRY(c->kzz_tab.ensure((size_t)cap * n_pad * 8));
                    CUDA_TRY(c->kzz_flag.ensure((size_t)cap * 4));
                    ktab = c->kzz_tab.as<double>();
                    kflag = c->kzz_flag.as<int>();
                    launch(c, C_PREP, s, [&] {
                        kzz_table_kernel<<<nb, NTHR, 0, s>>>(trow_src + (size_t)w0 * src_stride, src_stride, crx,
                                                             c->pp.as<PairParams>(), ktab, kflag);
                    });
                }
                if (int e = smem_opt_in(c, schur_kernel, MAIN_SMEM)) return e;
                launch(c, C_SCHUR, s, [&] {
                    schur_kernel<<<nb * ntiles, NTHR, MAIN_SMEM, s>>>(a, c->X.as<double>(), xs, crx, ntiles,
                                                                      cov + (size_t)w0 * n * n, (long)n * n, ktab, kflag);
                });
            }
        }
        if (alpha_out)
            CUDA_TRY(cudaMemcpy2DAsync(alpha_out + (size_t)w0 * m, (size_t)m * 8, c->alpha.p, (size_t)m_pad * 8,
                                       (size_t)m * 8, nb, cudaMemcpyDeviceToDevice, s));
        if (status)
            CUDA_TRY(cudaMemcpyAsync(status + w0, c->status.p, (size_t)nb * 4, cudaMemcpyDeviceToDevice, s));
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

// sqrtW of the G covariances in cov_dev into w_dev, which then holds the resident weight stack of step 3; copied to
// the HOST array sqrtw.
static int sqrtw_resident(gpbo_ctx* c, cudaStream_t s, int G, int n, double eta, double* sqrtw, int* status, int* iters) {
    int rc = sqrtw_device(c, s, c->cov_dev.as<double>(), G, n, eta, c->w_dev.as<double>(), status, iters);
    if (rc) return rc;
    c->w_G = G; c->w_n = n;
    CUDA_TRY(cudaMemcpyAsync(sqrtw, c->w_dev.p, (size_t)G * n * n * 8, cudaMemcpyDeviceToHost, s));
    return GPBO_OK;
}

static int moments_host(gpbo_ctx* c, int mode, const double* t, const double* y, int G, int m, const double* theta,
                        const double* pts, long pts_stride, int n, double* o1, double* o2, double* cov, double* alpha,
                        int* status, double eta = 0.0, double* sqrtw = nullptr, int* w_status = nullptr,
                        int* w_iters = nullptr) {
    if (!c || !t || !y || !theta || !pts || !o1 || !o2 || G <= 0 || m <= 0 || n <= 0)
        return fail(GPBO_EINVAL, "moments_host: bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    int rc = upload_problem(c, s, t, y, G, m);
    if (rc) return rc;
    CUDA_TRY(c->theta_dev.ensure((size_t)G * 24));
    CUDA_TRY(cudaMemcpyAsync(c->theta_dev.p, theta, (size_t)G * 24, cudaMemcpyHostToDevice, s));
    const size_t npts = pts_stride == 0 ? (size_t)n : (size_t)G * pts_stride;
    if (!all_finite(pts, npts)) return fail(GPBO_EINVAL, "evaluation points contain NaN or infinity");
    CUDA_TRY(c->tsrc.ensure(npts * 8));
    CUDA_TRY(cudaMemcpyAsync(c->tsrc.p, pts, npts * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(c->out1.ensure((size_t)G * n * 8));
    CUDA_TRY(c->out2.ensure((size_t)G * n * 8));
    CUDA_TRY(c->st_dev.ensure((size_t)G * 4));
    if (cov) {
        rc = fit_buffers(c, s, {{&c->cov_dev, (size_t)G * n * n * 8}});
        if (rc) return rc;
    }
    if (alpha) CUDA_TRY(c->grad_dev.ensure((size_t)G * m * 8));
    rc = moments_device(c, s, mode, c->t_dev.as<double>(), c->y_dev.as<double>(), G, m, c->theta_dev.as<double>(),
                        c->tsrc.as<double>(), pts_stride, n, c->out1.as<double>(), c->out2.as<double>(),
                        cov ? c->cov_dev.as<double>() : nullptr, alpha ? c->grad_dev.as<double>() : nullptr,
                        c->st_dev.as<int>());
    if (rc) return rc;
    if (sqrtw) {
        if (!cov) return fail(GPBO_EINVAL, "lstsq_weights: cov output is required when sqrtw is requested");
        rc = fit_buffers(c, s, {{&c->cov_dev, c->cov_dev.bytes}, {&c->w_dev, (size_t)G * n * n * 8}});
        if (rc) return rc;
        rc = sqrtw_resident(c, s, G, n, eta, sqrtw, w_status, w_iters);
        if (rc) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(o1, c->out1.p, (size_t)G * n * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(o2, c->out2.p, (size_t)G * n * 8, cudaMemcpyDeviceToHost, s));
    if (cov) CUDA_TRY(cudaMemcpyAsync(cov, c->cov_dev.p, (size_t)G * n * n * 8, cudaMemcpyDeviceToHost, s));
    if (alpha) CUDA_TRY(cudaMemcpyAsync(alpha, c->grad_dev.p, (size_t)G * m * 8, cudaMemcpyDeviceToHost, s));
    if (status) CUDA_TRY(cudaMemcpyAsync(status, c->st_dev.p, (size_t)G * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

int gpbo_predict_host(gpbo_ctx* c, const double* t, const double* y, int G, int m, const double* theta,
                      const double* t_star, long tstar_stride, int n_star, double* mean, double* std, double* alpha,
                      int* status) {
    return moments_host(c, 0, t, y, G, m, theta, t_star, tstar_stride, n_star, mean, std, nullptr, alpha, status);
}

int gpbo_lstsq_moments_host(gpbo_ctx* c, const double* t, const double* y, int G, int m, const double* theta,
                            const double* t_est, long test_stride, int n_est, double* state, double* ddt, double* cov,
                            int* status) {
    return moments_host(c, 1, t, y, G, m, theta, t_est, test_stride, n_est, state, ddt, cov, nullptr, status);
}

int gpbo_lstsq_weights_host(gpbo_ctx* c, const double* t, const double* y, int G, int m, const double* theta,
                            const double* t_est, long test_stride, int n_est, double eta, double* state, double* ddt,
                            double* cov, double* sqrtw, int* status, int* w_status, int* w_iters) {
    if (!sqrtw || !cov) return fail(GPBO_EINVAL, "lstsq_weights_host: cov and sqrtw outputs are required");
    return moments_host(c, 1, t, y, G, m, theta, t_est, test_stride, n_est, state, ddt, cov, nullptr, status, eta, sqrtw,
                        w_status, w_iters);
}

int gpbo_sqrtw(gpbo_ctx* c, const double* cov, int G, int n, double eta, double* sqrtw, int* status, int* iters,
               void* stream) {
    if (!c || !cov || !sqrtw || G <= 0 || n <= 0) return fail(GPBO_EINVAL, "sqrtw: bad argument");
    return sqrtw_device(c, static_cast<cudaStream_t>(stream), cov, G, n, eta, sqrtw, status, iters);
}

int gpbo_sqrtw_host(gpbo_ctx* c, const double* cov, int G, int n, double eta, double* sqrtw, int* status, int* iters) {
    if (!c || !cov || !sqrtw || G <= 0 || n <= 0) return fail(GPBO_EINVAL, "sqrtw_host: bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    const size_t bytes = (size_t)G * n * n * 8;
    int rc = fit_buffers(c, s, {{&c->cov_dev, bytes}, {&c->w_dev, bytes}});
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->cov_dev.p, cov, bytes, cudaMemcpyHostToDevice, s));
    rc = sqrtw_resident(c, s, G, n, eta, sqrtw, status, iters);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

// Step 3's A_g = sqrtW[g] @ lhs and b_g = sqrtW[g] @ rhs[g] for all g into wp_olhs / wp_orhs.  sqrtw (HOST; NULL: the
// resident stack in w_dev, which must be G x n x n), lhs [n][d] and rhs [G][n] are HOST arrays; `who` names the
// entry point in the error message.
static int weighted_products(gpbo_ctx* c, cudaStream_t s, const char* who, const double* sqrtw, int G, int n,
                             const double* lhs, int d, const double* rhs) {
    if (sqrtw) {
        CUDA_TRY(c->w_dev.ensure((size_t)G * n * n * 8));
        CUDA_TRY(cudaMemcpyAsync(c->w_dev.p, sqrtw, (size_t)G * n * n * 8, cudaMemcpyHostToDevice, s));
        c->w_G = G; c->w_n = n;
    } else if (c->w_G != G || c->w_n != n || !c->w_dev.p) {
        return fail(GPBO_EINVAL, std::string(who) + ": sqrtw is NULL but the resident weight stack has another shape "
                                                    "(call gpbo_lstsq_weights_host / gpbo_sqrtw_host for the same G, n first)");
    }
    CUDA_TRY(c->wp_lhs.ensure((size_t)n * d * 8));
    CUDA_TRY(c->wp_rhs.ensure((size_t)G * n * 8));
    CUDA_TRY(c->wp_olhs.ensure((size_t)G * n * d * 8));
    CUDA_TRY(c->wp_orhs.ensure((size_t)G * n * 8));
    CUDA_TRY(cudaMemcpyAsync(c->wp_lhs.p, lhs, (size_t)n * d * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(c->wp_rhs.p, rhs, (size_t)G * n * 8, cudaMemcpyHostToDevice, s));
    launch(c, C_SQRTW, s, [&] {
        weighted_products_kernel<<<dim3((n + NTHR / 32 - 1) / (NTHR / 32), G), NTHR, 0, s>>>(
            c->w_dev.as<double>(), n, c->wp_lhs.as<double>(), d, c->wp_rhs.as<double>(), c->wp_olhs.as<double>(),
            c->wp_orhs.as<double>());
    });
    CUDA_TRY(cudaGetLastError());
    return GPBO_OK;
}

int gpbo_weighted_products_host(gpbo_ctx* c, const double* sqrtw, int G, int n, const double* lhs, int d,
                                const double* rhs, double* out_lhs, double* out_rhs) {
    if (!c || !lhs || !rhs || !out_lhs || !out_rhs || G <= 0 || n <= 0 || d <= 0)
        return fail(GPBO_EINVAL, "weighted_products_host: bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    int rc = weighted_products(c, s, "weighted_products_host", sqrtw, G, n, lhs, d, rhs);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_lhs, c->wp_olhs.p, (size_t)G * n * d * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(out_rhs, c->wp_orhs.p, (size_t)G * n * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

int gpbo_posterior_grid_host(gpbo_ctx* c, const double* sqrtw, int G, int n, const double* lhs, int d, const double* rhs,
                             const double* regs, int nreg, double* means, double* chol, double* gram, double* proj,
                             int* status) {
    if (!c || !lhs || !rhs || !regs || !means || !status || G <= 0 || n <= 0 || d <= 0 || nreg <= 0)
        return fail(GPBO_EINVAL, "posterior_grid_host: bad argument");
    if (d > POST_DMAX) return fail(GPBO_EINVAL, "posterior_grid_host: operator rows longer than 128 entries are not supported");
    for (int k = 0; k < nreg; ++k)
        if (!std::isfinite(regs[k])) return fail(GPBO_EINVAL, "posterior_grid_host: non-finite regularizer");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    int rc = weighted_products(c, s, "posterior_grid_host", sqrtw, G, n, lhs, d, rhs);
    if (rc) return rc;
    const size_t slots = (size_t)nreg * G;
    CUDA_TRY(c->pg_gram.ensure((size_t)G * d * d * 8));
    CUDA_TRY(c->pg_proj.ensure((size_t)G * d * 8));
    CUDA_TRY(c->pg_regs.ensure((size_t)nreg * 8));
    CUDA_TRY(c->pg_means.ensure(slots * d * 8));
    if (chol) CUDA_TRY(c->pg_chol.ensure(slots * d * d * 8));
    CUDA_TRY(c->pg_status.ensure(slots * 4));
    CUDA_TRY(c->pg_tmp.ensure(slots * n * 8));
    CUDA_TRY(cudaMemcpyAsync(c->pg_regs.p, regs, (size_t)nreg * 8, cudaMemcpyHostToDevice, s));
    const size_t smem = ((size_t)d * (d + 1) + 3 * (size_t)d + 8) * 8;
    if (int e = smem_opt_in(c, ridge_solve_kernel, smem)) return e;
    const int nt = (d + GRAM_T - 1) / GRAM_T;
    launch(c, C_SQRTW, s, [&] {
        gram_kernel<<<dim3(nt * nt, G), 256, 0, s>>>(c->wp_olhs.as<double>(), c->wp_orhs.as<double>(), n, d,
                                                      c->pg_gram.as<double>(), c->pg_proj.as<double>());
    });
    launch(c, C_SQRTW, s, [&] {
        ridge_solve_kernel<<<dim3(G, nreg), 256, smem, s>>>(c->wp_olhs.as<double>(), c->wp_orhs.as<double>(), n, d,
                                                            c->pg_gram.as<double>(), c->pg_proj.as<double>(),
                                                            c->pg_regs.as<double>(), c->pg_means.as<double>(),
                                                            chol ? c->pg_chol.as<double>() : nullptr,
                                                            c->pg_status.as<int>(), c->pg_tmp.as<double>());
    });
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(means, c->pg_means.p, slots * d * 8, cudaMemcpyDeviceToHost, s));
    if (chol) CUDA_TRY(cudaMemcpyAsync(chol, c->pg_chol.p, slots * d * d * 8, cudaMemcpyDeviceToHost, s));
    if (gram) CUDA_TRY(cudaMemcpyAsync(gram, c->pg_gram.p, (size_t)G * d * d * 8, cudaMemcpyDeviceToHost, s));
    if (proj) CUDA_TRY(cudaMemcpyAsync(proj, c->pg_proj.p, (size_t)G * d * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(status, c->pg_status.p, slots * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return GPBO_OK;
}

int gpbo_lstsq_moments(gpbo_ctx* c, const double* t, const double* y, int G, int m, const double* theta,
                       const double* t_est, long test_stride, int n_est, double* state, double* ddt, double* cov,
                       int* status, void* stream) {
    if (!c || !t || !y || !theta || !t_est || !state || !ddt || G <= 0 || m <= 0 || n_est <= 0)
        return fail(GPBO_EINVAL, "lstsq_moments: bad argument");
    return moments_device(c, static_cast<cudaStream_t>(stream), 1, t, y, G, m, theta, t_est, test_stride, n_est, state,
                          ddt, cov, nullptr, status);
}

// ---- FP64 tensor-pipe peak: back-to-back independent DMMA chains --------------------------
__global__ void __launch_bounds__(256) dmma_peak_kernel(int iters, double* out) {
    double acc[16][2];
#pragma unroll
    for (int i = 0; i < 16; ++i) { acc[i][0] = 0.0; acc[i][1] = 0.0; }
    const double a = 1e-3 * (threadIdx.x & 7), b = 1e-3 * (threadIdx.x & 3);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) dmma884(acc[i], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += acc[i][0] + acc[i][1];
    if (s == 12345.678) out[0] = s;
}

int gpbo_bench_dmma_peak(gpbo_ctx* c, int iters, double* tflops, double* ms) {
    if (!c || !tflops || iters <= 0) return fail(GPBO_EINVAL, "bench_dmma_peak: bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, c->device));
    const int grid = prop.multiProcessorCount * 4;
    CUDA_TRY(c->out1.ensure(64));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    dmma_peak_kernel<<<grid, 256, 0, c->stream>>>(iters / 8 + 1, c->out1.as<double>());
    CUDA_TRY(cudaEventRecord(e0, c->stream));
    dmma_peak_kernel<<<grid, 256, 0, c->stream>>>(iters, c->out1.as<double>());
    CUDA_TRY(cudaEventRecord(e1, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->launches += 2;
    float f = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&f, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    const double flops = (double)grid * 8.0 * (double)iters * 16.0 * 512.0;
    *tflops = flops / (f * 1e-3) / 1e12;
    if (ms) *ms = f;
    return GPBO_OK;
}

}  // extern "C"
