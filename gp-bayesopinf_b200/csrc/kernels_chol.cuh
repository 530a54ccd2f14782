// Batched blocked FP64 Cholesky / triangular inverse / fused K^-1-gradient kernels.
//
// One launch processes one algorithmic step for EVERY (GP, start) pair of a wave, so the
// hyper-parameter optimiser's whole batch advances in lock-step (BASELINE.json north_star (2),(3)).
// Reference arithmetic: sklearn _gpr.py:583-651 (Cholesky, alpha, LML, K^-1, gradient traces).
//
// Per pair the workspace holds one m_pad x m_pad row-major buffer:
//   lower triangle  : L  (K = L L^T), written block column by block column (left-looking)
//   upper triangle  : U = L^-T (= W^T, W = L^-1), written block row by block row
//   side buffers    : D_j = inv(L_jj) and DT_j = D_j^T for every 128x128 diagonal block
// K itself is never materialised: tiles of K(theta) are generated in the epilogue of the
// kernel that first needs them, and K^-1 = W^T W is consumed tile-by-tile by the gradient
// reductions (sum_ij (alpha_i alpha_j - K^-1_ij) dK_ij/dtheta) without being written.
#pragma once
#include "tile_engine.cuh"

namespace gpbo {

struct MatArgs {
    double* A;          // [cap][m_pad*lda]
    long mat_stride;    // doubles between consecutive pairs' matrices
    int lda;            // = m_pad
    int m;              // valid size
    int T;              // m_pad / 128
    double* D;          // [cap][T][128*128]
    double* DT;         // [cap][T][128*128]
    double* logdet;     // [cap][T]   sum_i log L_ii of each diagonal block
    int* status;        // [cap]      0 ok, 1 = not positive definite
    const PairParams* pp;   // [cap]
    const double* ts;   // [cap][m_pad] scaled abscissae t/ell (sklearn order) or raw t (rbf_eval order)
    int flags;          // bit 0: trtri rows launch their tiles longest-first (j-major) instead of pair-major
    // [cap][2 T] (lo, hi) of each 128-row block of ts over its real rows (prep_pairs_kernel), or nullptr: no profile
    // skipping.  Set for the RBF family in sklearn order only; the intervals live in the z buffer, which nothing
    // else uses before the factorisation and the inverse rows are done (see band_first).
    const double* band = nullptr;
};

// Whether the factorisation of pair p has already failed: chol_diag_kernel sets status[p] at the diagonal block with a
// non-positive pivot, and everything computed for the pair after that is discarded by finalize_kernel (-inf, zero
// gradient, as scikit-learn, _gpr.py:589-593).  The kernels of the LML / gradient path call this first and return
// for such a pair, so a pair that fails in block column 0 costs one diagonal block instead of a whole evaluation.
// Thread 0 reads the flag and __syncthreads_or hands the one answer to every thread: the whole CTA leaves, or none of it,
// before any mbarrier, cp.async or TMA is set up -- a CTA whose warps decided differently would wait forever at a
// barrier.  With the inverse rows on the side stream (eval_wave) trtri_row_kernel may read the flag while
// chol_diag_kernel writes it; a CTA that misses a just-written failure computes numbers that finalize_kernel discards.
__device__ __forceinline__ bool pair_failed(const int* status, int p) {
    return __syncthreads_or(threadIdx.x == 0 && status[p] != 0);
}

// ---- exactly-zero tiles of short-length-scale RBF kernel matrices -------------------------------------------------
// AsmSklearn computes an off-diagonal element as sig2 * gpbo_exp_neg(-0.5 * (d * d)), d = x_r - x_c, and gpbo_exp_neg
// returns exactly 0.0 once |argument| > 708 (the flush on the high word, fastmath.h).  Let the rows of block i have
// scaled abscissae in [lo_i, hi_i] and those of block k in [lo_k, hi_k].  If lo_i - hi_k > 38, every x_r - x_c >=
// lo_i - hi_k, and rounding is monotone, so fl(x_r - x_c) > 38, fl(d * d) >= 1444 and the argument is <= -722: every
// element of tile (i, k) is sig2 * 0.0 = 0.0, whatever the order of the abscissae.  The same holds with i and k swapped.
// The outer span bounds |d| from above: below 1e150, d * d is finite, so the gradient terms sig2 R_ij d^2 of
// lauum_grad_kernel are exactly 0 there too (and not 0 * inf).  NaN bounds compare false: no tile is skipped.
// tests/test_band_rule.py and tools/ab_bench.py read BAND_GAP / BAND_SPAN_MAX from this file; the test checks the rule
// element by element on the CPU against the host gpbo_exp_neg.
constexpr double BAND_GAP = 38.0;
constexpr double BAND_SPAN_MAX = 1e150;
__device__ __forceinline__ bool tile_zero(double lo_i, double hi_i, double lo_k, double hi_k) {
    return (lo_i - hi_k > BAND_GAP || lo_k - hi_i > BAND_GAP) && fmax(hi_i - lo_k, hi_k - lo_i) < BAND_SPAN_MAX;
}

// The profile of the factor: f(r) = the first block column k <= r whose K tile (r, k) is not certainly zero (0 without
// a.band).  By induction over the left-looking recurrence, L_rk is exactly zero for k < f(r): S_rk = K_rk - sum_{k' < k}
// L_rk' L_kk'^T has only zero terms, and a sum of products with an exactly-zero operand stays +0.  So the k-loops
// of the factorisation and the inverse may start at the profile without changing a bit of any accumulator.
// Returns (f(i), f(j)) to every thread: warp 0 scans row i, warp 1 row j, 32 block columns per ballot.  Every thread
// of the CTA calls it, once per kernel (after pair_failed, before any mbarrier, cp.async or TMA set-up).
__device__ __forceinline__ int2 band_first(const MatArgs& a, int p, int i, int j) {
    __shared__ int first[2];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (w < 2) {
        const int r = w == 0 ? i : j;
        int f = 0;
        if (a.band) {
            const double* bp = a.band + (long)p * a.lda;
            const double lo = bp[2 * r], hi = bp[2 * r + 1];
            f = r;
            for (int k0 = 0; k0 < r; k0 += 32) {
                const int k = k0 + lane;
                const unsigned live = __ballot_sync(0xffffffffu, k < r && !tile_zero(lo, hi, bp[2 * k], bp[2 * k + 1]));
                if (live) { f = k0 + __ffs(live) - 1; break; }
            }
        }
        if (lane == 0) first[w] = f;
    }
    __syncthreads();
    return make_int2(first[0], first[1]);
}

// Whether K tile (I, J), I != J, is certainly zero, from the tile's own rows of ts (lauum_grad_kernel runs after
// z_from_inverse_kernel has overwritten the intervals of a.band).  Every thread of the CTA calls it.
__device__ __forceinline__ bool tile_zero_from_ts(const MatArgs& a, int p, int I, int J) {
    static_assert(NTHR == 2 * TB, "one thread per row of the two blocks: warps 0-3 take block I, warps 4-7 block J");
    __shared__ double ext[2][NTHR / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = (tid < TB ? I : J) * TB + (tid & (TB - 1));        // warps 0-3: block I, warps 4-7: block J
    double lo = INFINITY, hi = -INFINITY;
    if (r < a.m) {
        const double x = a.ts[(long)p * a.lda + r];
        lo = x == x ? x : -INFINITY;
        hi = x == x ? x : INFINITY;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) { ext[0][warp] = lo; ext[1][warp] = hi; }
    __syncthreads();
    bool zero = false;
    if (tid == 0) {
        const double li = fmin(fmin(ext[0][0], ext[0][1]), fmin(ext[0][2], ext[0][3]));
        const double hi_ = fmax(fmax(ext[1][0], ext[1][1]), fmax(ext[1][2], ext[1][3]));
        const double lj = fmin(fmin(ext[0][4], ext[0][5]), fmin(ext[0][6], ext[0][7]));
        const double hj = fmax(fmax(ext[1][4], ext[1][5]), fmax(ext[1][6], ext[1][7]));
        zero = tile_zero(li, hi_, lj, hj);
    }
    return __syncthreads_or(zero);
}

// A 128 x 128 tile of one value (row stride ld), coalesced: the tiles that the profile makes exactly zero.
__device__ __forceinline__ void store_const_tile(double* dst, long ld, double v) {
    for (int q = threadIdx.x; q < TB * TB / 2; q += NTHR)
        *reinterpret_cast<double2*>(dst + (long)(q / (TB / 2)) * ld + 2 * (q % (TB / 2))) = make_double2(v, v);
}

// ---- element generators ("assemblers") ---------------------------------------------------
// sklearn order (kernels.py:1559-1565, 1279-1292, 1407-1414): x = t/ell, R = exp(-0.5 (xi-xj)^2),
// diagonal exactly sigma^2 + chi.
struct AsmSklearn {
    double sig2, chi;
    int m;
    __device__ __forceinline__ double operator()(int r, int c, double xr, double xc) const {
        if (r >= m || c >= m) return r == c ? 1.0 : 0.0;
        if (r == c) return sig2 + chi;
        const double d = xr - xc;
        return sig2 * gpbo_exp_neg(-0.5 * (d * d));
    }
};
// rbf_eval order (gpkernels.py:608-609, 639): kappa = sigma^2 exp(-(ti-tj)^2 / (2 ell^2)), + chi on the diagonal.
struct AsmRbfEval {
    double sig2, chi, two_ell2, r_two_ell2;
    int m;
    __device__ __forceinline__ double operator()(int r, int c, double tr, double tcn) const {
        if (r >= m || c >= m) return r == c ? 1.0 : 0.0;
        if (r == c) return sig2 + chi;
        const double d = tr - tcn;
        return sig2 * gpbo_exp_neg(-gpbo_div(d * d, two_ell2, r_two_ell2));
    }
};

// Matern nu = FAM / 2 (FAM = 3 or 5), scikit-learn order (kernels.py:1601-1790: dists = |xi - xj| with x = t / ell,
// K = dists * sqrt(2 nu), then (1 + K) exp(-K) resp. (1 + K + K^2 / 3) exp(-K)).  Extension: the reference is RBF-only.
template <int FAM>
__device__ __forceinline__ double matern_value(double sig2, double dx) {
    const double K = fabs(dx) * (FAM == 3 ? 1.7320508075688772 : 2.23606797749979);
    const double e = gpbo_exp_neg(-K);
    return sig2 * ((FAM == 3) ? (1.0 + K) * e : (1.0 + K + K * K / 3.0) * e);
}
template <int FAM>
struct AsmMatern {
    double sig2, chi;
    int m;
    __device__ __forceinline__ double operator()(int r, int c, double xr, double xc) const {
        if (r >= m || c >= m) return r == c ? 1.0 : 0.0;
        if (r == c) return sig2 + chi;
        return matern_value<FAM>(sig2, xr - xc);
    }
};

// ORDER: 0 RBF sklearn order, 1 RBF rbf_eval order, 2 Matern-3/2, 3 Matern-5/2 (both sklearn order, scaled abscissae)
template <int ORDER>
struct AsmSelect;
template <>
struct AsmSelect<0> {
    using type = AsmSklearn;
    static __device__ __forceinline__ type make(const PairParams& q, int m) { return {q.sig2, q.chi, m}; }
};
template <>
struct AsmSelect<1> {
    using type = AsmRbfEval;
    static __device__ __forceinline__ type make(const PairParams& q, int m) {
        return {q.sig2, q.chi, 2 * (q.ell * q.ell), 0.5 * q.inv_ell2, m};
    }
};

template <>
struct AsmSelect<2> {
    using type = AsmMatern<3>;
    static __device__ __forceinline__ type make(const PairParams& q, int m) { return {q.sig2, q.chi, m}; }
};
template <>
struct AsmSelect<3> {
    using type = AsmMatern<5>;
    static __device__ __forceinline__ type make(const PairParams& q, int m) { return {q.sig2, q.chi, m}; }
};

// ---- prep: natural-unit hyper-parameters and scaled abscissae ------------------------------
// ORDER 0: ts = t / ell (sklearn divides X by length_scale before pdist, kernels.py:1559);
// ORDER 1: ts = t.
// band (order 0 only, may be nullptr): [pair][2 T] the (lo, hi) of each block of ts over its real rows, computed from the
// same quotients, for the profile of the factor (MatArgs::band).  A NaN abscissa widens its block to (-inf, inf).
__global__ void prep_pairs_kernel(const double* __restrict__ theta, const int* __restrict__ gp_of,
                                  const double* __restrict__ t, int m, int m_pad, int order,
                                  PairParams* __restrict__ pp, double* __restrict__ ts, int* __restrict__ status,
                                  double* __restrict__ band) {
    const int p = blockIdx.x;
    const double sig2 = exp(theta[3 * p + 0]);
    const double ell = exp(theta[3 * p + 1]);
    const double chi = exp(theta[3 * p + 2]);
    const int gp = gp_of ? gp_of[p] : p;
    if (threadIdx.x == 0) {
        PairParams q;
        q.sig2 = sig2; q.ell = ell; q.chi = chi; q.inv_ell2 = 1.0 / (ell * ell); q.gp = gp; q.pad = 0;
        pp[p] = q;
        status[p] = 0;
    }
    const double* tg = t + (long)gp * m;
    for (int i = threadIdx.x; i < m_pad; i += blockDim.x)
        ts[(long)p * m_pad + i] = i < m ? (order == 0 ? tg[i] / ell : tg[i]) : 0.0;
    if (band) {
        const int lane = threadIdx.x & 31;
        for (int b = threadIdx.x >> 5; b < m_pad / TB; b += blockDim.x >> 5) {
            double lo = INFINITY, hi = -INFINITY;
            for (int i = b * TB + lane; i < min(m, (b + 1) * TB); i += 32) {
                const double x = tg[i] / ell;
                lo = x == x ? fmin(lo, x) : -INFINITY;
                hi = x == x ? fmax(hi, x) : INFINITY;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
                hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
            }
            if (lane == 0) {
                band[(long)p * m_pad + 2 * b] = lo;
                band[(long)p * m_pad + 2 * b + 1] = hi;
            }
        }
    }
}

// ---- in-shared factorisation of one 128x128 diagonal block -------------------------------
// P (stride LDP) holds the symmetric block S on entry (lower part used).  On exit the lower part
// holds L (S = L L^T), the strict upper part holds inv(L)^T, dinv[i] = 1 / L_ii.
// Returns (to every thread) whether a non-positive pivot was met; *logsum gets sum_i log L_ii.
//
// Blocked right-looking algorithm with 32-wide panels:
//   per panel  (1) chol32_block: the 32x32 diagonal block is factored by one warp in registers (warp_chol32:
//                  shuffles, no barrier);
//              (2) panel X L_kk^T = A by forward substitution, one thread per row with the row in registers;
//              (3) all warps: trailing A22 -= X X^T (register tiles);
//   then the four 32x32 diagonal blocks are inverted concurrently (2 lanes per column), and the off-diagonal
//   blocks of inv(L) follow by block rows: W_ij = -W_ii * sum_k L_ik W_kj.
// `scratch` needs PB + 1 doubles during the factorisation and PB*(3*PB+1) during the inversion (re-used).
constexpr int PB = 32;            // panel width
constexpr int LDG = 3 * PB + 1;   // stride of the G scratch of the inversion
constexpr int POTF_SCRATCH = PB * LDG;

// Reciprocal from the hardware approximation plus two Newton steps (<= 1 ulp): the one long-latency operation on the
// critical path of a pivot step.
__device__ __forceinline__ double fast_rcp(double d) {
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
    double e = fma(-d, x, 1.0);
    x = fma(x, e, x);
    e = fma(-d, x, 1.0);
    return fma(x, e, x);
}

// ONE WARP factors a 32 x 32 symmetric positive definite block in place: lane r takes row r into registers
// (a[c] = A[r][c], c <= r).  Right-looking with unscaled columns; per pivot step: the pivot comes by shuffle from
// lane j (so its reciprocal starts at once), the lanes publish their column-j entries in a double-buffered 32-double
// shared array and read the multipliers a_cj back as broadcasts, rank-1 update in registers -- warp-synchronous, one
// __syncwarp per step, no CTA-wide barrier (the all-threads version this replaces spent ~21 000 cycles per block on
// its 32 barriers).  The 32 square roots are taken once at the end.
// rowp: this lane's row (first of the block's 32 columns); dinv_lane receives 1 / L_rr.  Returns (warp-uniformly)
// whether a pivot was <= 0 (the pivot is then replaced by 1).  nv: number of leading rows that are not identity padding.
// Not inlined: its 32-double register row must not
// inflate the register allocation of the DMMA kernels that call it.
#ifndef GPBO_CHOL32_INLINE
#define GPBO_CHOL32_ATTR __noinline__
#else
#define GPBO_CHOL32_ATTR __forceinline__
#endif
__device__ GPBO_CHOL32_ATTR bool warp_chol32(double* rowp, double* dinv_lane, int nv) {
    __shared__ __align__(16) double colbuf[2][32];
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    // Nothing below is predicated on (c <= lane): the registers a[c], c > lane, hold whatever lies right of the
    // diagonal (finite or not) and are updated like the rest, but never read by another lane (col[c] is only read for
    // rows c > j, from lane c's VALID entry a[j], j < c) and never written back.  32 x 31 / 2 unpredicated DFMAs and 16-byte
    // broadcast loads instead of 4700 instructions of predicate bookkeeping.
    double a[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) a[c] = rowp[c];
    double my_d = 1.0;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        // rows / columns >= nv are identity padding (the reference's sizes m = 10 ... 200 rarely fill the last block):
        // their pivots are 1 and their multipliers 0, so the remaining steps change nothing (warp-uniform exit)
        if (j >= nv) break;
        double d = __shfl_sync(FULL, a[j], j);
        double* col = colbuf[j & 1];
        col[lane] = a[j];
        __syncwarp();
        if (!(d > 0.0)) { bad = true; d = 1.0; }
        if (lane == j) my_d = d;
        const double w = -(a[j] * fast_rcp(d));
        if ((j + 1) & 1) {                               // odd first column: one scalar step, then aligned pairs
            if (j + 1 < 32) a[j + 1] = fma(w, col[j + 1], a[j + 1]);
        }
#pragma unroll
        for (int c = (j + 2) & ~1; c < 32; c += 2) {
            const double2 cc = *reinterpret_cast<const double2*>(col + c);
            a[c] = fma(w, cc.x, a[c]);
            a[c + 1] = fma(w, cc.y, a[c + 1]);
        }
        // no second barrier: step j + 1 writes the other buffer, and nobody reaches step j + 2's write before every
        // lane has passed step j + 1's __syncwarp, i.e. finished reading this one
    }
    const double rs = rsqrt(my_d);
#pragma unroll
    for (int c = 0; c < 32; ++c) {
        const double rsc = __shfl_sync(FULL, rs, c);
        if (c <= lane) rowp[c] = (c == lane ? my_d : a[c]) * rsc;
    }
    *dinv_lane = rs;
    __syncwarp();
    return bad;
}

#ifndef GPBO_CHOL32_ALLTHREADS
// Cholesky of the 32x32 block at P[o..o+32)^2 (lower part, in place, row stride LDP) by warp 0; dinv[o+i] = 1 / L_ii.
// `flag` = one double of scratch.  Ends with __syncthreads(); returns (uniformly) whether a pivot was <= 0.
__device__ __forceinline__ bool chol32_block(double* P, int o, double* dinv, double* flag, int nv = 32) {
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        const bool bad = warp_chol32(P + (o + lane) * LDP + o, dinv + o + lane, nv);
        if (lane == 0) *flag = bad ? 1.0 : 0.0;
    }
    __syncthreads();
    return *flag != 0.0;
}

#else
// Variant kept for A/B measurements (-DGPBO_CHOL32_ALLTHREADS): all 256 threads, one CTA barrier per pivot step.
__device__ __forceinline__ bool chol32_block(double* P, int o, double* dinv, double* rsv, int /*nv*/ = 32) {
    const int tid = threadIdx.x;
    const int r = tid >> 3, c8 = tid & 7;                 // row of the block, column class
    double* Pr = P + (o + r) * LDP + o;
    bool bad = false;
    for (int j = 0; j < PB - 1; ++j) {
        double d = P[(o + j) * LDP + o + j];
        if (!(d > 0.0)) { bad = true; d = 1.0; }
        const double inv_d = __drcp_rn(d);
        if (tid == 0) rsv[j] = d;
        if (r > j) {
            const double w = Pr[j] * inv_d;
#pragma unroll
            for (int q = 0; q < PB / 8; ++q) {
                const int c = c8 + 8 * q;
                if (c > j && c <= r) Pr[c] = fma(-w, P[(o + c) * LDP + o + j], Pr[c]);
            }
        }
        __syncthreads();
    }
    {
        double d = P[(o + PB - 1) * LDP + o + PB - 1];
        if (!(d > 0.0)) { bad = true; d = 1.0; }
        if (tid == 0) rsv[PB - 1] = d;
    }
    __syncthreads();
    if (tid < PB) rsv[tid] = rsqrt(rsv[tid]);
    __syncthreads();
#pragma unroll
    for (int q = 0; q < PB / 8; ++q) {
        const int c = c8 + 8 * q;
        if (c <= r) {
            const double v = Pr[c];
            Pr[c] = (c == r && !(v > 0.0)) ? 1.0 : v * rsv[c];
        }
    }
    if (tid < PB) dinv[o + tid] = rsv[tid];
    __syncthreads();
    return bad;
}
#endif

// nv = number of valid (non-padding) rows of the block: rows >= nv are identity rows (the reference's sizes
// m = 10 ... 200 leave most of a 128-tile as padding), so only the first ceil(nv / 32) panels are factored and
// inverted; the identity part gets L = W = I directly.
__device__ __forceinline__ bool potf2_trtri_smem(double* P, double* scratch, double* dinv, double* logsum_out, int nv) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    bool bad = false;
    double* rsv = scratch;
    const int nvb = (nv + PB - 1) / PB;          // panels that hold valid rows (1..4)
    const int nact = nvb * PB;                   // rows / columns that take part in the factorisation
    __syncthreads();   // P was just filled by all threads
    if (nact < TB) {
        // identity part: 1 / L_ii = 1, and W[r][c] = 0 for r >= nact, c < r (stored transposed at P[c][r])
        for (int q = tid; q < TB * (TB - nact); q += NTHR) {
            const int c = q / (TB - nact), r = nact + q % (TB - nact);
            if (c < r) P[c * LDP + r] = 0.0;
        }
        if (tid >= nact && tid < TB) dinv[tid] = 1.0;
    }
    for (int kb = 0; kb < nvb; ++kb) {
        const int o = kb * PB;
        bad |= chol32_block(P, o, dinv, rsv, min(PB, nv - o));
        const int R0 = o + PB, n = nact - R0;
        if (n <= 0) break;
        // (2) panel by forward substitution, one thread per row:  X L_kk^T = A  (row in registers, L_kk broadcast)
        if (tid < n) {
            double* Ar = P + (R0 + tid) * LDP + o;
            const double* Lk = P + o * LDP + o;
            double x[PB];
#pragma unroll
            for (int c = 0; c < PB; ++c) x[c] = Ar[c];
#pragma unroll
            for (int c = 0; c < PB; ++c) {
                double s0 = x[c], s1 = 0.0;
#pragma unroll
                for (int k = 0; k + 1 < c; k += 2) {
                    s0 = fma(-x[k], Lk[c * LDP + k], s0);
                    s1 = fma(-x[k + 1], Lk[c * LDP + k + 1], s1);
                }
                if (c & 1) s0 = fma(-x[c - 1], Lk[c * LDP + c - 1], s0);
                x[c] = (s0 + s1) * dinv[o + c];
            }
#pragma unroll
            for (int c = 0; c < PB; ++c) Ar[c] = x[c];
        }
        __syncthreads();
        // (3) trailing update of the lower triangle: A[r][c] -= sum_k X[r][k] X[c][k]
        {
            const int ty = tid >> 4, tx = tid & 15;
            const int nt = n >> 4;                 // 6, 4, 2
            double acc[6][6];
#pragma unroll
            for (int ii = 0; ii < 6; ++ii)
#pragma unroll
                for (int jj = 0; jj < 6; ++jj) acc[ii][jj] = 0.0;
            const double* Xr = P + (R0 + ty) * LDP + o;
            const double* Xc = P + (R0 + tx) * LDP + o;
#pragma unroll 4
            for (int k = 0; k < PB; ++k) {
                double xr[6], xc[6];
#pragma unroll
                for (int ii = 0; ii < 6; ++ii) {
                    xr[ii] = ii < nt ? Xr[ii * 16 * LDP + k] : 0.0;
                    xc[ii] = ii < nt ? Xc[ii * 16 * LDP + k] : 0.0;
                }
#pragma unroll
                for (int ii = 0; ii < 6; ++ii)
#pragma unroll
                    for (int jj = 0; jj <= ii; ++jj) acc[ii][jj] = fma(xr[ii], xc[jj], acc[ii][jj]);
            }
#pragma unroll
            for (int ii = 0; ii < 6; ++ii)
#pragma unroll
                for (int jj = 0; jj <= ii; ++jj) {
                    const int r = R0 + ty + 16 * ii, c = R0 + tx + 16 * jj;
                    if (ii < nt && c <= r) P[r * LDP + c] -= acc[ii][jj];
                }
        }
        __syncthreads();
    }
#ifndef GPBO_DIAGINV_TWOLANE
    // inverses of the 32x32 diagonal blocks, all at once: one warp per block, lane = column jc with the column in
    // registers (forward substitution over the rows, L_bb read as broadcasts); W is written transposed into the strict
    // upper part of P, where the column under construction is contiguous.
    if (warp < nvb) {
        const int o = warp * PB, jc = lane;
        double w[PB];
#pragma unroll
        for (int rr = 0; rr < PB; ++rr) {
            const double* Lr = P + (o + rr) * LDP + o;
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int k = 0; k + 1 < rr; k += 2) {
                s0 = fma(Lr[k], w[k], s0);            // w[k] = 0 for k < jc
                s1 = fma(Lr[k + 1], w[k + 1], s1);
            }
            if (rr & 1) s0 = fma(Lr[rr - 1], w[rr - 1], s0);
            const double di = dinv[o + rr];
            w[rr] = rr < jc ? 0.0 : (rr == jc ? di : -(s0 + s1) * di);
        }
        double* Wc = P + (o + jc) * LDP + o;           // Wc[k] = W[k][jc], k > jc
#pragma unroll
        for (int rr = 1; rr < PB; ++rr)
            if (rr > jc) Wc[rr] = w[rr];
    }
#else
    // Variant kept for A/B measurements (-DGPBO_DIAGINV_TWOLANE): 64 threads per block, 2 lanes per column.
    if ((tid >> 6) < nvb) {
        const int o = (tid >> 6) * PB, jc = (tid & 63) >> 1, h = tid & 1;
        double* Wc = P + (o + jc) * LDP + o;
        const double wjj = dinv[o + jc];
        for (int rr = 1; rr < PB; ++rr) {
            double s0 = 0.0, s1 = 0.0;
            if (rr > jc) {
                const double* Lr = P + (o + rr) * LDP + o;
                if (h == 0) s0 = Lr[jc] * wjj;
                int k = jc + 1 + h;
                for (; k + 2 < rr; k += 4) {
                    s0 = fma(Lr[k], Wc[k], s0);
                    s1 = fma(Lr[k + 2], Wc[k + 2], s1);
                }
                if (k < rr) s0 = fma(Lr[k], Wc[k], s0);
            }
            double sacc = s0 + s1;
            sacc += __shfl_xor_sync(0xffffffffu, sacc, 1);
            if (h == 0 && rr > jc) Wc[rr] = -sacc * dinv[o + rr];
            __syncwarp();
        }
    }
#endif
    __syncthreads();
    // off-diagonal blocks of W = inv(L), block row bi; W stored transposed in the strict upper part of P
    double* Gs = scratch;
    for (int bi = 1; bi < nvb; ++bi) {
        const int oi = bi * PB, ncol = oi;
        const int r = oi + lane;
        const double* Lr = P + r * LDP;
        for (int col = warp; col < ncol; col += NTHR / 32) {
            const double* Wc = P + col * LDP;            // Wc[k] = W[k][col] for k > col
            // four independent partial sums: the dot product is a dependent-FMA chain otherwise
            double g0 = Lr[col] * dinv[col], g1 = 0.0, g2 = 0.0, g3 = 0.0;
            int k = col + 1;
            for (; k + 3 < oi; k += 4) {
                g0 = fma(Lr[k], Wc[k], g0);
                g1 = fma(Lr[k + 1], Wc[k + 1], g1);
                g2 = fma(Lr[k + 2], Wc[k + 2], g2);
                g3 = fma(Lr[k + 3], Wc[k + 3], g3);
            }
            for (; k < oi; ++k) g0 = fma(Lr[k], Wc[k], g0);
            Gs[lane * LDG + col] = (g0 + g1) + (g2 + g3);
        }
        __syncthreads();
        for (int col = warp; col < ncol; col += NTHR / 32) {
            double a0 = dinv[r] * Gs[lane * LDG + col], a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
            for (int ap = 0; ap < PB; ap += 4) {
                // W_ii[lane][ap] for ap < lane is stored at P[oi+ap][oi+lane]
                if (ap < lane) a0 = fma(P[(oi + ap) * LDP + r], Gs[ap * LDG + col], a0);
                if (ap + 1 < lane) a1 = fma(P[(oi + ap + 1) * LDP + r], Gs[(ap + 1) * LDG + col], a1);
                if (ap + 2 < lane) a2 = fma(P[(oi + ap + 2) * LDP + r], Gs[(ap + 2) * LDG + col], a2);
                if (ap + 3 < lane) a3 = fma(P[(oi + ap + 3) * LDP + r], Gs[(ap + 3) * LDG + col], a3);
            }
            P[col * LDP + r] = -((a0 + a1) + (a2 + a3));
        }
        __syncthreads();
    }
    if (tid < 32) {
        double ls = 0.0;
        for (int c = tid; c < TB; c += 32) ls += log(P[c * LDP + c]);
        ls = warp_sum(ls);
        if (tid == 0) *logsum_out = ls;
    }
    __syncthreads();
    return bad;
}

// ---- split-K pre-accumulation for small batches --------------------------------------------
// With few pairs in flight the left-looking k-loops (up to T-1 blocks long) leave most SMs idle and put
// the whole loop on the critical path of every block column / row.  splitk_partial_kernel then computes the
// tile products in `nsplit` k-chunks on separate CTAs into a scratch buffer (accumulator layout, fixed order ->
// deterministic), and the consumer kernels (chol_diag / chol_panel / trtri_row) start from the summed tile
// instead of running their own loop.
struct PreAcc {
    const double* buf;   // [unit][nsplit][64][256] partial accumulators; nullptr: the kernel runs its own k-loop
    int nsplit;          // chunks per tile
    int chunk;           // k-slices per chunk
};

__device__ __forceinline__ void preacc_load(Acc& acc, const PreAcc& pre, long unit, int nk, int tid) {
    const int nsp = min(pre.nsplit, (nk + pre.chunk - 1) / pre.chunk);
    for (int sidx = 0; sidx < nsp; ++sidx) {
        const double* b = pre.buf + ((unit * pre.nsplit + sidx) * 64) * NTHR + tid;
#pragma unroll
        for (int mi = 0; mi < 8; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int e = 0; e < 2; ++e) acc.v[mi][ni][e] += b[((mi * 4 + ni) * 2 + e) * NTHR];
    }
}

// mode 0: Cholesky column idx=j : tile t of pair p is block row j + t (t = 0: diagonal tile), k-slices [0, 8 j)
// mode 1: trtri row idx=i       : tile t is column block t < i,                             k-slices [0, 8 (i - t))
// mode 2: prediction TRSM col j : tile t is row block t of X (rows = prediction points),     k-slices [0, 8 j)
// blockIdx.x = ((p * ntile) + t) * nsplit + chunk index.
__global__ void __launch_bounds__(NTHR, 1)
splitk_partial_kernel(MatArgs a, int mode, int idx, int ntile, int nsplit, int chunk, double* __restrict__ buf,
                      const double* __restrict__ X, long x_stride) {
    extern __shared__ __align__(16) double smem[];
    const ThreadCoord tc;
    const int unit = blockIdx.x / nsplit, sp = blockIdx.x % nsplit;
    const int p = unit / ntile, t = unit % ntile;
    const int nk = (mode == 1 ? idx - t : idx) * (TB / BK);
    const int k1 = min(nk, sp * chunk + chunk);
    int k0 = sp * chunk;
    if (k0 >= k1) return;
    if (mode != 2 && pair_failed(a.status, p)) return;   // mode 2 (prediction): a not-PD GP is an error there anyway
    // the profile (band_first): slices before it multiply exactly-zero blocks of L.  A tile that its consumer writes as
    // zero needs no partials; a chunk that lies wholly before the profile stores an exact zero in its place.
    if (mode == 0) {
        const int2 f = band_first(a, p, idx + t, idx);
        if (idx < f.x) return;
        k0 = max(k0, max(f.x, f.y) * (TB / BK));
    } else if (mode == 1) {
        const int fi = band_first(a, p, idx, idx).x;
        if (fi == idx) return;
        k0 = max(k0, (max(t, fi) - t) * (TB / BK));
    }
    const double* Ap = a.A + (long)p * a.mat_stride;
    __shared__ uint64_t bars[2 * NSTAGE];
    Ring ring;
    ring_init(ring, bars);
    Acc acc;
    acc_zero(acc);
    if (mode == 1) {
        const int i = idx, j = t;
        const double* Lrow = Ap + (long)i * TB * a.lda;
        const double* Urow = Ap + (long)j * TB * a.lda;
        const double* DTj = a.DT + ((long)p * a.T + j) * (TB * TB);
        gemm_nt_loop<false>(
            acc,
            [&](int kk) {
                const int kt = kk + k0;
                const double* ap = Lrow + j * TB + kt * BK;
                return kt < TB / BK ? SliceSrc{ap, a.lda, DTj + kt * BK, TB}
                                    : SliceSrc{ap, a.lda, Urow + j * TB + kt * BK, a.lda};
            },
            k1 - k0, smem, ring, tc);
    } else {
        const double* arows = (mode == 2 ? X + (long)p * x_stride + (long)t * TB * a.lda
                                         : Ap + (long)(idx + t) * TB * a.lda);
        const double* brows = Ap + (long)idx * TB * a.lda;
        gemm_nt_loop<false>(
            acc, [&](int kk) { return SliceSrc{arows + (kk + k0) * BK, a.lda, brows + (kk + k0) * BK, a.lda}; },
            k1 - k0, smem, ring, tc);
    }
    double* b = buf + ((long)blockIdx.x * 64) * NTHR + tc.tid;
#pragma unroll
    for (int mi = 0; mi < 8; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int e = 0; e < 2; ++e) b[((mi * 4 + ni) * 2 + e) * NTHR] = acc.v[mi][ni][e];
}

// ---- Cholesky, diagonal tile of block column j ---------------------------------------------
// S_jj = K_jj - sum_{k<j} L_jk L_jk^T (DMMA);  L_jj = chol(S_jj);  D_j = inv(L_jj).
// TMA: the k-loop's operand slices come by cp.async.bulk.tensor through `tm` (gemm_nt_loop_tma) instead of LDGSTS.
template <int ORDER, bool TMA>
__global__ void __launch_bounds__(NTHR, 1)
chol_diag_kernel(MatArgs a, int j, PreAcc pre, const __grid_constant__ TmaMaps tm) {
    extern __shared__ __align__(16) double smem_raw[];
    double* smem = smem_align_1024(smem_raw);     // TMA's 128-byte swizzle atoms are 1024 bytes (launch: + SMEM_ALIGN_PAD)
    const ThreadCoord tc;
    const int p = blockIdx.x;
    if (j > 0 && pair_failed(a.status, p)) return;
    const int kb = ORDER == 0 && j > 0 ? band_first(a, p, j, j).x * (TB / BK) : 0;   // L_jk = 0 left of the profile
    double* Ap = a.A + (long)p * a.mat_stride;
    const double* rows = Ap + (long)j * TB * a.lda;
    __shared__ uint64_t bars[2 * NSTAGE];
    Ring ring;
    if (TMA) ring_init_tma(ring, bars); else ring_init(ring, bars);
    Acc acc;
    acc_zero(acc);
    if (pre.buf)
        preacc_load(acc, pre, (long)p * (a.T - j), j * (TB / BK), tc.tid);
    else if (TMA)
        gemm_nt_loop_tma<true>(
            acc, [&](int kt) { return TmaSlice{&tm.A, (kb + kt) * BK, p * a.lda + j * TB, nullptr, 0, 0}; },
            j * (TB / BK) - kb, smem, ring, tc);
    else
        gemm_nt_loop<true>(acc, [&](int kt) { return SliceSrc{rows + (kb + kt) * BK, a.lda, nullptr, 0}; },
                           j * (TB / BK) - kb, smem, ring, tc);
    __syncthreads();   // every warp is done with the ring: its memory becomes P

    double* P = smem;
    double* dinv = smem + TB * LDP;
    double* scratch = dinv + TB;
    __shared__ double logsum;
    {
        const PairParams q = a.pp[p];
        const auto el = AsmSelect<ORDER>::make(q, a.m);
        const double* tsp = a.ts + (long)p * a.lda + j * TB;
        double xr[8], xc[4][2];
#pragma unroll
        for (int mi = 0; mi < 8; ++mi) xr[mi] = tsp[tc.row(mi)];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) { xc[ni][0] = tsp[tc.col(ni, 0)]; xc[ni][1] = tsp[tc.col(ni, 1)]; }
#pragma unroll
        for (int mi = 0; mi < 8; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int r = tc.row(mi), c = tc.col(ni, e);
                    if (c <= r)
                        P[r * LDP + c] = el(j * TB + r, j * TB + c, xr[mi], xc[ni][e]) - acc.v[mi][ni][e];
                }
    }
    const bool bad = potf2_trtri_smem(P, scratch, dinv, &logsum, min(TB, a.m - j * TB));

    // write L_jj (lower), D_j = inv(L_jj) and DT_j = D_j^T
    double* Lout = Ap + (long)j * TB * a.lda + j * TB;
    double* Dj = a.D + ((long)p * a.T + j) * (TB * TB);
    double* DTj = a.DT + ((long)p * a.T + j) * (TB * TB);
    const int c = tc.tid & (TB - 1);
    for (int r = tc.tid >> 7; r < TB; r += 2) {
        if (c <= r) Lout[(long)r * a.lda + c] = P[r * LDP + c];
        Dj[r * TB + c] = c < r ? P[c * LDP + r] : (c == r ? dinv[r] : 0.0);
        DTj[r * TB + c] = c > r ? P[r * LDP + c] : (c == r ? dinv[r] : 0.0);
    }
    if (tc.tid == 0) {
        a.logdet[(long)p * a.T + j] = logsum;
        if (bad) a.status[p] = 1;
    }
}

// ---- element generators for rows that are NOT training points (prediction rows) -----------
// Rows are estimation points t'_a, columns training points t_j (gpkernels.py:630-641).
struct CrossArgs {
    const double* trow;   // [G][lrow] row abscissae (t_est, or t_est/ell in sklearn order), zero padded
    int nrow;             // valid rows (m')
    int lrow;             // padded rows
    int kind;             // 0: K(t*, t) sklearn order (predict, _gpr.py:446); 1: kappa_zy; 2: K_zy
    int fam;              // 0 RBF; 3 / 5 Matern (rows and columns are then always t / ell)
};

__device__ __forceinline__ double cross_element(int kind, int fam, const PairParams& q, int r, int c, int nrow, int m,
                                                double xr, double xc) {
    if (r >= nrow || c >= m) return 0.0;
    const double d = xr - xc;
    if (fam != 0) {
        // Matern: value for kinds 0 / 1, d kappa / d t' for kind 2 (tau = ell d, a^2 = 2 nu / ell^2)
        if (kind != 2) return fam == 3 ? matern_value<3>(q.sig2, d) : matern_value<5>(q.sig2, d);
        const double K = fabs(d) * (fam == 3 ? 1.7320508075688772 : 2.23606797749979);
        const double e = gpbo_exp_neg(-K);
        const double a2 = (fam == 3 ? 3.0 : 5.0) * q.inv_ell2;
        const double tau = d * q.ell;
        return fam == 3 ? -q.sig2 * a2 * tau * e : -q.sig2 * (a2 / 3.0) * tau * (1.0 + K) * e;
    }
    if (kind == 0) return q.sig2 * gpbo_exp_neg(-0.5 * (d * d));
    const double ell2 = q.ell * q.ell;
    const double kap = q.sig2 * gpbo_exp_neg(-gpbo_div(d * d, 2 * ell2, 0.5 * q.inv_ell2));
    if (kind == 1) return kap;
    return gpbo_div(-d * kap, ell2, q.inv_ell2);     // gpkernels.py:640
}

// ---- Cholesky panel / triangular solve with many right-hand sides -------------------------
// tile (i, j):  X_ij = (S_ij - sum_{k<j} X_ik L_jk^T) * inv(L_jj)^T
// CROSS == false: X = L itself (rows i > j of the factor), S = K(theta) tile.
// CROSS == true : X = V^T (rows = prediction points), S = cross-covariance tile; this is the
//                 TRSM  V = L^-1 K_zy^T  of gpkernels.py:491 / _gpr.py:460 done as a continuation
//                 of the Cholesky of the joint covariance.
template <int ORDER, bool CROSS, bool TMA>
__global__ void __launch_bounds__(NTHR, 1)
chol_panel_kernel(MatArgs a, int j, double* X, long x_stride, int xT, CrossArgs cr, PreAcc pre,
                  const __grid_constant__ TmaMaps tm) {
    static_assert(!(CROSS && TMA), "the prediction rows live in X, which has no tensor map");
    extern __shared__ __align__(16) double smem_raw[];
    double* smem = smem_align_1024(smem_raw);     // TMA's 128-byte swizzle atoms are 1024 bytes (launch: + SMEM_ALIGN_PAD)
    const ThreadCoord tc;
    int p, i;
    if (CROSS) { p = blockIdx.x / xT; i = blockIdx.x % xT; }
    else { const int per = a.T - 1 - j; p = blockIdx.x / per; i = j + 1 + blockIdx.x % per; }
    if (!CROSS && pair_failed(a.status, p)) return;      // CROSS (prediction): a not-PD GP is an error there anyway
    const double* Ap = a.A + (long)p * a.mat_stride;
    double* Xp = CROSS ? X + (long)p * x_stride : a.A + (long)p * a.mat_stride;
    int kb = 0;                                          // first k-slice right of the profiles of rows i and j
    if (!CROSS && ORDER == 0) {
        const int2 f = band_first(a, p, i, j);
        if (j < f.x) {                                   // left of row i's profile: L_ij is exactly zero
            store_const_tile(Xp + (long)i * TB * a.lda + j * TB, a.lda, 0.0);
            return;
        }
        kb = max(f.x, f.y) * (TB / BK);
    }
    const double* arows = Xp + (long)i * TB * a.lda;
    const double* brows = Ap + (long)j * TB * a.lda;
    __shared__ uint64_t bars[2 * NSTAGE], bars_tma[2 * NSTAGE];
    Ring ring;
    ring_init(ring, bars);                 // the epilogue product's cp.async ring (and the main loop's without TMA)
    Acc acc;
    acc_zero(acc);
    if (pre.buf)
        preacc_load(acc, pre, CROSS ? (long)p * xT + i : (long)p * (a.T - j) + (i - j), j * (TB / BK), tc.tid);
    else if (TMA) {
        Ring ring_m;
        ring_init_tma(ring_m, bars_tma);
        gemm_nt_loop_tma<false>(
            acc,
            [&](int kt) {
                return TmaSlice{&tm.A, (kb + kt) * BK, p * a.lda + i * TB, &tm.A, (kb + kt) * BK, p * a.lda + j * TB};
            },
            j * (TB / BK) - kb, smem, ring_m, tc);
    } else
        gemm_nt_loop<false>(
            acc, [&](int kt) { return SliceSrc{arows + (kb + kt) * BK, a.lda, brows + (kb + kt) * BK, a.lda}; },
            j * (TB / BK) - kb, smem, ring, tc);

    double* S = smem;
    double* stages = smem + TB * LDS;
    const double* Dj = a.D + ((long)p * a.T + j) * (TB * TB);
    __syncthreads();   // every warp is done with the main loop's ring: its memory becomes S + the epilogue's stages
    epi_prefill_D(Dj, stages, ring, tc);   // inv(L_jj) slices fly while the K tile is generated in registers
    {
        const PairParams q = a.pp[p];
        double xr[8], xc[4][2];
        const double* tcol = a.ts + (long)p * a.lda + j * TB;
        const double* trow = CROSS ? cr.trow + (long)p * cr.lrow + i * TB : a.ts + (long)p * a.lda + i * TB;
#pragma unroll
        for (int mi = 0; mi < 8; ++mi) xr[mi] = trow[tc.row(mi)];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) { xc[ni][0] = tcol[tc.col(ni, 0)]; xc[ni][1] = tcol[tc.col(ni, 1)]; }
        const auto el = AsmSelect<ORDER>::make(q, a.m);
#pragma unroll
        for (int mi = 0; mi < 8; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int r = i * TB + tc.row(mi), c = j * TB + tc.col(ni, e);
                    const double kv = CROSS ? cross_element(cr.kind, cr.fam, q, r, c, cr.nrow, a.m, xr[mi], xc[ni][e])
                                            : el(r, c, xr[mi], xc[ni][e]);
                    acc.v[mi][ni][e] = kv - acc.v[mi][ni][e];
                }
    }
    acc_to_smem<LDS>(acc, S, tc);
    __syncthreads();
    Acc out;
    acc_zero(out);
    epi_product_SxDt(out, S, Dj, stages, ring, tc, true);
    double* dst = Xp + (long)i * TB * a.lda + j * TB;
#pragma unroll
    for (int mi = 0; mi < 8; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
            double2 v = make_double2(out.v[mi][ni][0], out.v[mi][ni][1]);
            *reinterpret_cast<double2*>(dst + (long)tc.row(mi) * a.lda + tc.col(ni, 0)) = v;
        }
}

// ---- prediction TRSM as ONE persistent launch ("row sweep") ---------------------------------
// Row tile i of X = K_* L^-T depends only on itself and on L:  X_ij = (S_ij - sum_{k<j} X_ik L_jk^T) inv(L_jj)^T,
// so a CTA can sweep j = 0 .. T-1 for its 128 rows with no other CTA involved.  A unit = one (GP, row tile) sweep;
// all units cost the same, so with `units` not a multiple of the CTA count (8 GPs x 32 row tiles = 256 units on 148
// SMs) whole-unit scheduling loses up to half a round.  The sweeps are therefore cut ALONG j: the linear work order
// (unit-major, step-minor, step j costing 2 j + 2) is divided into gridDim.x equal cost ranges.  A range starts inside
// unit u0 at step j0 and ends inside unit u1 before step j1; the CTA does the head of u1 (steps [0, j1)) FIRST and
// publishes it, then its whole units, then the tail of u0 (steps [j0, T)) LAST, waiting for the head that the
// previous CTA published at the very beginning of its own range -- no circular wait, and the wait is over long before
// it is reached.  flags[u] (zeroed before the launch) = head of unit u complete.
__device__ __forceinline__ void sweep_locate(long b, int T, long C, int* u, int* j) {
    *u = (int)(b / C);
    const long rem = b - (long)*u * C;
    int jj = (int)((sqrt(4.0 * (double)rem + 1.0) - 1.0) * 0.5);
    while ((long)jj * (jj + 1) < rem) ++jj;
    while (jj > 0 && (long)(jj - 1) * jj >= rem) --jj;
    if (jj >= T) { jj = 0; *u += 1; }
    *j = jj;                                   // smallest j with j (j + 1) >= rem: steps >= j lie at or after b
}

__global__ void __launch_bounds__(NTHR, 1)
cross_sweep_kernel(MatArgs a, double* X, long x_stride, int xT, int units, CrossArgs cr, int* flags) {
    extern __shared__ __align__(16) double smem[];
    const ThreadCoord tc;
    __shared__ uint64_t bars[2 * NSTAGE];
    Ring ring;
    ring_init(ring, bars);
    const int T = a.T;
    const long C = (long)T * (T + 1), W = (long)units * C;
    int u0, j0, u1, j1;
    sweep_locate(W * blockIdx.x / gridDim.x, T, C, &u0, &j0);
    sweep_locate(W * (blockIdx.x + 1) / gridDim.x, T, C, &u1, &j1);

    auto steps = [&](int u, int ja, int jb) {
        const int p = u / xT, i = u % xT;
        const double* Ap = a.A + (long)p * a.mat_stride;
        double* Xp = X + (long)p * x_stride;
        const double* arows = Xp + (long)i * TB * a.lda;
        const PairParams q = a.pp[p];
        const double* trow = cr.trow + (long)p * cr.lrow + i * TB;
        for (int j = ja; j < jb; ++j) {
            const double* brows = Ap + (long)j * TB * a.lda;
            Acc acc;
            acc_zero(acc);
            gemm_nt_loop<false>(acc, [&](int kt) { return SliceSrc{arows + kt * BK, a.lda, brows + kt * BK, a.lda}; },
                                j * (TB / BK), smem, ring, tc);
            double* S = smem;
            double* stages = smem + TB * LDS;
            const double* Dj = a.D + ((long)p * a.T + j) * (TB * TB);
            __syncthreads();
            epi_prefill_D(Dj, stages, ring, tc);
            {
                const double* tcol = a.ts + (long)p * a.lda + j * TB;
                double xr[8];
#pragma unroll
                for (int mi = 0; mi < 8; ++mi) xr[mi] = trow[tc.row(mi)];
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) {
                    const double2 xc = *reinterpret_cast<const double2*>(tcol + tc.col(ni, 0));
#pragma unroll
                    for (int mi = 0; mi < 8; ++mi) {
                        const int r = i * TB + tc.row(mi), c = j * TB + tc.col(ni, 0);
                        acc.v[mi][ni][0] = cross_element(cr.kind, cr.fam, q, r, c, cr.nrow, a.m, xr[mi], xc.x) - acc.v[mi][ni][0];
                        acc.v[mi][ni][1] = cross_element(cr.kind, cr.fam, q, r, c + 1, cr.nrow, a.m, xr[mi], xc.y) - acc.v[mi][ni][1];
                    }
                }
            }
            acc_to_smem<LDS>(acc, S, tc);
            __syncthreads();
            Acc out;
            acc_zero(out);
            epi_product_SxDt(out, S, Dj, stages, ring, tc, true);
            double* dst = Xp + (long)i * TB * a.lda + j * TB;
#pragma unroll
            for (int mi = 0; mi < 8; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni)
                    *reinterpret_cast<double2*>(dst + (long)tc.row(mi) * a.lda + tc.col(ni, 0)) =
                        make_double2(out.v[mi][ni][0], out.v[mi][ni][1]);
            __syncthreads();   // X_ij is visible to the whole CTA (it is an operand of the next step); smem is free again
        }
    };

    // Segments of this CTA's range, in execution order: [head of u1] [whole units] [tail of u0].  ONE call site of
    // steps(): the body (main loop + epilogue with all their dispatch switches) is instantiated once.
    // The host launches at most one CTA per unit, so a range covers at least one whole sweep and a unit is shared by
    // at most two CTAs; a range strictly inside one unit (u0 == u1, j0 > 0) cannot occur and is not supported.
    const bool split_tail = j0 > 0;                                  // u0's head belongs to the previous CTA
    const bool split_head = j1 > 0 && u1 < units;                    // u1's tail belongs to the next CTA
    const int first_whole = split_tail ? u0 + 1 : u0;
    const int n_whole = u1 > first_whole ? u1 - first_whole : 0;
    const int nseg = (split_head ? 1 : 0) + n_whole + (split_tail ? 1 : 0);
    for (int sidx = 0; sidx < nseg; ++sidx) {
        const int w = sidx - (split_head ? 1 : 0);
        const bool is_head = split_head && sidx == 0;
        const bool is_tail = !is_head && w >= n_whole;
        const int u = is_head ? u1 : (is_tail ? u0 : first_whole + w);
        const int ja = is_tail ? j0 : 0, jb = is_head ? j1 : T;
        if (is_tail) {                                               // the head was published by the previous CTA
            if (tc.tid == 0) { while (atomicAdd(&flags[u], 0) == 0) __nanosleep(64); __threadfence(); }
            __syncthreads();
        }
        steps(u, ja, jb);
        if (is_head) {
            __threadfence();
            __syncthreads();
            if (tc.tid == 0) atomicExch(&flags[u], 1);
        }
    }
}

// ---- forward / backward substitution with the block factor ------------------------------
// The diagonal-block solves use the block inverses D_j = inv(L_jj) (a 128x128 GEMV each) like the panel
// TRSM does, instead of a 128-step sequential substitution.
// One CTA of 1024 threads per pair: the GEMV parts are latency bound on a single SM, so they run with 32 warps
// and four rows per warp in flight.
constexpr int TRSV_THR = 1024;
constexpr int TRSV_RPW = TB / (TRSV_THR / 32);   // rows per warp = 4

// z = L^-1 y (one CTA per pair).  _gpr.py:601 (cho_solve, first half).
__global__ void __launch_bounds__(TRSV_THR, 1) trsv_fwd_kernel(MatArgs a, const double* __restrict__ ypad, double* z) {
    __shared__ double xs[TB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int p = blockIdx.x;
    if (pair_failed(a.status, p)) return;
    const double* Ap = a.A + (long)p * a.mat_stride;
    const double* yp = ypad + (long)a.pp[p].gp * a.lda;
    double* zp = z + (long)p * a.lda;
    for (int jb = 0; jb < a.T; ++jb) {
        const double* rows = Ap + (long)jb * TB * a.lda;
        const int nk = jb * TB;
        // r = y_j - L[j, 0:nk] z[0:nk]; TRSV_RPW rows per warp at once (z loaded once for them), lanes across k
        {
            const int r0 = warp * TRSV_RPW;
            double sacc[TRSV_RPW];
#pragma unroll
            for (int q = 0; q < TRSV_RPW; ++q) sacc[q] = 0.0;
#pragma unroll 2
            for (int k = 2 * lane; k < nk; k += 64) {
                const double2 zz = *reinterpret_cast<const double2*>(zp + k);
#pragma unroll
                for (int q = 0; q < TRSV_RPW; ++q) {
                    const double2 l = *reinterpret_cast<const double2*>(rows + (long)(r0 + q) * a.lda + k);
                    sacc[q] += l.x * zz.x + l.y * zz.y;
                }
            }
#pragma unroll
            for (int q = 0; q < TRSV_RPW; ++q) {
                const double sv = warp_sum(sacc[q]);
                if (lane == 0) xs[r0 + q] = yp[jb * TB + r0 + q] - sv;
            }
        }
        __syncthreads();
        // z_j = D_j r  (D_j lower triangular)
        const double* Dj = a.D + ((long)p * a.T + jb) * (TB * TB);
#pragma unroll
        for (int q = 0; q < TRSV_RPW; ++q) {
            const int r = warp * TRSV_RPW + q;
            double sv = 0.0;
#pragma unroll
            for (int u = 0; u < TB / 32; ++u) {
                const int c = lane + 32 * u;
                if (c <= r) sv = fma(Dj[r * TB + c], xs[c], sv);
            }
            sv = warp_sum(sv);
            if (lane == 0) zp[jb * TB + r] = sv;
        }
        __syncthreads();
    }
}

// alpha = L^-T z (one CTA per pair).  _gpr.py:601 (cho_solve, second half).
__global__ void __launch_bounds__(TRSV_THR, 1) trsv_bwd_kernel(MatArgs a, const double* __restrict__ z, double* alpha) {
    __shared__ double xs[TB], ws[TB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int p = blockIdx.x;
    if (pair_failed(a.status, p)) return;
    const double* Ap = a.A + (long)p * a.mat_stride;
    const double* zp = z + (long)p * a.lda;
    double* wp = alpha + (long)p * a.lda;
    for (int k = tid; k < a.lda; k += TRSV_THR) wp[k] = zp[k];
    __syncthreads();
    for (int jb = a.T - 1; jb >= 0; --jb) {
        const double* rows = Ap + (long)jb * TB * a.lda;
        if (tid < TB) ws[tid] = wp[jb * TB + tid];
        __syncthreads();
        // alpha_j = inv(L_jj)^T w_j = DT_j w_j  (DT_j upper triangular, rows contiguous)
        const double* DTj = a.DT + ((long)p * a.T + jb) * (TB * TB);
#pragma unroll
        for (int q = 0; q < TRSV_RPW; ++q) {
            const int r = warp * TRSV_RPW + q;
            double sv = 0.0;
#pragma unroll
            for (int u = 0; u < TB / 32; ++u) {
                const int c = lane + 32 * u;
                if (c >= r) sv = fma(DTj[r * TB + c], ws[c], sv);
            }
            sv = warp_sum(sv);
            if (lane == 0) { xs[r] = sv; wp[jb * TB + r] = sv; }
        }
        __syncthreads();
        // w[0:nk] -= L[j, 0:nk]^T alpha_j ; threads across k (coalesced rows), 16 rows in flight per thread
        const int nk = jb * TB;
        for (int k = tid; k < nk; k += TRSV_THR) {
            double sv = 0.0;
#pragma unroll 16
            for (int r = 0; r < TB; ++r) sv += rows[(long)r * a.lda + k] * xs[r];
            wp[k] -= sv;
        }
        __syncthreads();
    }
}

// z = L^-1 y = W y from the inverse factor (same motivation as alpha_from_inverse_kernel below): one CTA per
// (pair, block k):  z_k = D_k y_k + sum_{I < k} U[I][k]^T y_I,  U[I][k] = W[k][I]^T stored in the upper triangle.
// Thread (h, c): column c of the block, rows r = h, h + 2, ... (coalesced 1 KB row segments), four partial sums.
__global__ void __launch_bounds__(NTHR) z_from_inverse_kernel(MatArgs a, const double* __restrict__ ypad,
                                                              double* __restrict__ z) {
    __shared__ double part[NTHR];
    const int p = blockIdx.x / a.T, kb = blockIdx.x % a.T;
    if (pair_failed(a.status, p)) return;
    const int c = threadIdx.x & (TB - 1), h = threadIdx.x >> 7;
    const double* Ap = a.A + (long)p * a.mat_stride;
    const double* yp = ypad + (long)a.pp[p].gp * a.lda;
    const double* Dk = a.D + ((long)p * a.T + kb) * (TB * TB);
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const int nrow = kb * TB;
    const double* col = Ap + kb * TB + c;
    int r = h;
    for (; r + 6 < nrow; r += 8) {
        s0 = fma(col[(long)r * a.lda], yp[r], s0);
        s1 = fma(col[(long)(r + 2) * a.lda], yp[r + 2], s1);
        s2 = fma(col[(long)(r + 4) * a.lda], yp[r + 4], s2);
        s3 = fma(col[(long)(r + 6) * a.lda], yp[r + 6], s3);
    }
    for (; r < nrow; r += 2) s0 = fma(col[(long)r * a.lda], yp[r], s0);
    // diagonal block: z_k[c] += sum_{q <= c} D_k[c][q] y_k[q]  (row c of D_k; half of the q range per h)
    for (int q = h; q <= c; q += 2) s1 = fma(Dk[c * TB + q], yp[kb * TB + q], s1);
    part[threadIdx.x] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (h == 0) z[(long)p * a.lda + kb * TB + c] = part[c] + part[TB + c];
}

// alpha = L^-T z = W^T z = U z once the inverse factor U = W^T is available (LML + gradient path, after
// trtri): unlike the backward substitution this has no sequential dependency over the block rows -- one CTA per
// (pair, block row I) streams U[I][I+1..T) once (coalesced) -- which matters when few pairs are in flight.
// alpha_I = DT_I z_I + sum_{k > I} U[I][k] z_k.  Accuracy: O(cond(L) eps) like the substitution (cond(L) = sqrt(cond K)).
__global__ void __launch_bounds__(NTHR) alpha_from_inverse_kernel(MatArgs a, const double* __restrict__ z,
                                                                  double* __restrict__ alpha) {
    const int p = blockIdx.x / a.T, I = blockIdx.x % a.T;
    if (pair_failed(a.status, p)) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double* Ap = a.A + (long)p * a.mat_stride;
    const double* zp = z + (long)p * a.lda;
    const double* DTI = a.DT + ((long)p * a.T + I) * (TB * TB);
    const int k0 = (I + 1) * TB;
    for (int rg = 0; rg < 4; ++rg) {                   // 16 rows per warp, four at a time (z loaded once for them)
        const int r0 = warp * 16 + rg * 4;
        double sacc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int u = 0; u < TB / 32; ++u) {            // diagonal block: DT_I is upper triangular
            const int c = lane + 32 * u;
            const double zc = zp[I * TB + c];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (c >= r0 + q) sacc[q] = fma(DTI[(r0 + q) * TB + c], zc, sacc[q]);
        }
#pragma unroll 2
        for (int k = k0 + 2 * lane; k < a.lda; k += 64) {
            const double2 zz = *reinterpret_cast<const double2*>(zp + k);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double2 u2 = *reinterpret_cast<const double2*>(Ap + (long)(I * TB + r0 + q) * a.lda + k);
                sacc[q] += u2.x * zz.x + u2.y * zz.y;
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double sv = warp_sum(sacc[q]);
            if (lane == 0) alpha[(long)p * a.lda + I * TB + r0 + q] = sv;
        }
    }
}

// ---- triangular inverse, block row i:  W_ij = -inv(L_ii) sum_{k=j}^{i-1} L_ik W_kj -----------
// stored transposed: U[j-block rows][i-block cols] = W_ij^T (upper triangle of the pair's buffer).
template <bool TMA>
__global__ void __launch_bounds__(NTHR, 1)
trtri_row_kernel(MatArgs a, int i, PreAcc pre, const __grid_constant__ TmaMaps tm) {
    extern __shared__ __align__(16) double smem_raw[];
    double* smem = smem_align_1024(smem_raw);     // TMA's 128-byte swizzle atoms are 1024 bytes (launch: + SMEM_ALIGN_PAD)
    const ThreadCoord tc;
    // tile (p, j) has a k-loop of i - j blocks.  Pair-major order keeps the i tiles of a pair (which share the L row
    // block) together; longest-first (flags bit 0) leaves only the short tiles for the tail of the launch.
    int p, j;
    if (a.flags & 1) { const int nb = gridDim.x / i; j = blockIdx.x / nb; p = blockIdx.x % nb; }
    else { p = blockIdx.x / i; j = blockIdx.x % i; }
    if (pair_failed(a.status, p)) return;
    double* Ap = a.A + (long)p * a.mat_stride;
    // L_ik = 0 left of row i's profile: the sum runs over k in [max(j, f(i)), i); an empty sum leaves W_ij = -(D_i 0)
    const int k0 = max(j, band_first(a, p, i, i).x);
    if (k0 == i) {
        store_const_tile(Ap + (long)j * TB * a.lda + i * TB, a.lda, -0.0);
        return;
    }
    const int kb = (k0 - j) * (TB / BK);                     // slices skipped; the loop's first block is dense if kb > 0
    const int tri = kb == 0 ? TB / BK : 0;
    const double* Lrow = Ap + (long)i * TB * a.lda;          // L[i-block rows][*]
    const double* Urow = Ap + (long)j * TB * a.lda;          // U[j-block rows][*]
    const double* DTj = a.DT + ((long)p * a.T + j) * (TB * TB);
    __shared__ uint64_t bars[2 * NSTAGE], bars_tma[2 * NSTAGE];
    Ring ring;
    ring_init(ring, bars);
    Acc acc;
    acc_zero(acc);
    // k-block j: B[n][k] = W_jj[k][n] = DT_j[n][k];  k-blocks j+1 .. i-1: B[n][k] = U[j*128+n][k]
    if (pre.buf)
        preacc_load(acc, pre, (long)p * i + j, (i - j) * (TB / BK), tc.tid);
    else if (TMA) {
        Ring ring_m;
        ring_init_tma(ring_m, bars_tma);
        gemm_nt_loop_tma<false, SKIP_B_UP>(
            acc,
            [&](int kt) {
                kt += kb;
                const int ka = j * TB + kt * BK, ra = p * a.lda + i * TB;
                return kt < TB / BK ? TmaSlice{&tm.A, ka, ra, &tm.DT, kt * BK, (p * a.T + j) * TB}
                                    : TmaSlice{&tm.A, ka, ra, &tm.A, ka, p * a.lda + j * TB};
            },
            (i - j) * (TB / BK) - kb, smem, ring_m, tc, tri);
    } else
        gemm_nt_loop<false, SKIP_B_UP>(
            acc,
            [&](int kt) {
                kt += kb;
                const double* ap = Lrow + j * TB + kt * BK;
                return kt < TB / BK ? SliceSrc{ap, a.lda, DTj + kt * BK, TB}
                                    : SliceSrc{ap, a.lda, Urow + j * TB + kt * BK, a.lda};
            },
            (i - j) * (TB / BK) - kb, smem, ring, tc, tri);
    double* G = smem;
    double* stages = smem + TB * LDS;
    const double* Di = a.D + ((long)p * a.T + i) * (TB * TB);
    __syncthreads();   // ring memory is re-used for G and the epilogue's stages
    epi_prefill_D(Di, stages, ring, tc);   // inv(L_ii) slices fly while the accumulators go to shared memory
    acc_to_smem<LDS>(acc, G, tc);      // G[k][n]
    __syncthreads();
    Acc out;
    acc_zero(out);
    epi_product_DxG(out, Di, G, stages, ring, tc, true);
    // transposed store: U[j*128 + col][i*128 + row] = -out[row][col]
    double* dst = Ap + (long)j * TB * a.lda + i * TB;
#pragma unroll
    for (int mi = 0; mi < 8; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int e = 0; e < 2; ++e) dst[(long)tc.col(ni, e) * a.lda + tc.row(mi)] = -out.v[mi][ni][e];
}

// ---- fused K^-1 tiles + gradient trace reductions -------------------------------------------
// tile (I, J), I >= J:  Kinv_IJ = sum_{k >= I} U[I][k] U[J][k]^T  (= (W^T W)_IJ), never stored.
// Reductions (sklearn _gpr.py:629-651 with kernels.py:1575-1577, 966-969, 1407-1414):
//   s0 = sum_ij (a_i a_j - Kinv_ij) sigma^2 R_ij
//   s1 = sum_ij (a_i a_j - Kinv_ij) sigma^2 R_ij (x_i - x_j)^2
//   s2 = sum_i  (a_i^2   - Kinv_ii)
// Off-diagonal tiles are counted twice (symmetry).  part[p][tile][4].
// FAM: 0 RBF (the reference), 3 / 5 Matern (dK/dlog ell from sklearn kernels.py: 3 D exp(-sqrt(3 D)) resp.
// 5/3 D (sqrt(5 D) + 1) exp(-sqrt(5 D)), D = squared scaled distance).
template <int FAM, bool TMA>
__global__ void __launch_bounds__(NTHR, 1)
lauum_grad_kernel(MatArgs a, const double* __restrict__ alpha, double* __restrict__ part, int ntiles,
                  const __grid_constant__ TmaMaps tm) {
    extern __shared__ __align__(16) double smem_raw[];
    double* smem = smem_align_1024(smem_raw);     // TMA's 128-byte swizzle atoms are 1024 bytes (launch: + SMEM_ALIGN_PAD)
    const ThreadCoord tc;
    const int p = blockIdx.x / ntiles, q = blockIdx.x % ntiles;
    if (pair_failed(a.status, p)) return;
    int I = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
    while ((I + 1) * (I + 2) / 2 <= q) ++I;
    while (I * (I + 1) / 2 > q) --I;
    const int J = q - I * (I + 1) / 2;
    // RBF: outside the band dK/dtheta is exactly 0 on the whole tile (tile_zero), so every term of the three sums is an
    // exact zero and the tile's partials are the +0 that the full computation would store
    if (FAM == 0 && I != J && tile_zero_from_ts(a, p, I, J)) {
        if (tc.tid < 4) part[((long)p * ntiles + q) * 4 + tc.tid] = 0.0;
        return;
    }
    const double* Ap = a.A + (long)p * a.mat_stride;
    const double* UI = Ap + (long)I * TB * a.lda;
    const double* UJ = Ap + (long)J * TB * a.lda;
    const double* DTI = a.DT + ((long)p * a.T + I) * (TB * TB);
    __shared__ uint64_t bars[2 * NSTAGE];
    Ring ring;
    if (TMA) ring_init_tma(ring, bars); else ring_init(ring, bars);
    Acc acc;
    acc_zero(acc);
    // k-block I comes from the diagonal-block inverse DT_I (row stride 128), k-blocks I+1.. from U (row stride lda)
    const int nk = (a.T - I) * (TB / BK);
    if (TMA) {
        const int rI = p * a.lda + I * TB, rJ = p * a.lda + J * TB, rD = (p * a.T + I) * TB;
        if (I == J)
            gemm_nt_loop_tma<true, SKIP_A_UP>(
                acc,
                [&](int kt) {
                    return kt < TB / BK ? TmaSlice{&tm.DT, kt * BK, rD, nullptr, 0, 0}
                                        : TmaSlice{&tm.A, I * TB + kt * BK, rI, nullptr, 0, 0};
                },
                nk, smem, ring, tc);
        else
            gemm_nt_loop_tma<false, SKIP_A_UP>(
                acc,
                [&](int kt) {
                    const int kb = I * TB + kt * BK;
                    return kt < TB / BK ? TmaSlice{&tm.DT, kt * BK, rD, &tm.A, kb, rJ} : TmaSlice{&tm.A, kb, rI, &tm.A, kb, rJ};
                },
                nk, smem, ring, tc);
    } else if (I == J) {
        gemm_nt_loop<true, SKIP_A_UP>(
            acc,
            [&](int kt) {
                return kt < TB / BK ? SliceSrc{DTI + kt * BK, TB, nullptr, 0}
                                    : SliceSrc{UI + I * TB + kt * BK, a.lda, nullptr, 0};
            },
            nk, smem, ring, tc);
    } else {
        gemm_nt_loop<false, SKIP_A_UP>(
            acc,
            [&](int kt) {
                const double* bp = UJ + I * TB + kt * BK;
                return kt < TB / BK ? SliceSrc{DTI + kt * BK, TB, bp, a.lda} : SliceSrc{UI + I * TB + kt * BK, a.lda, bp, a.lda};
            },
            nk, smem, ring, tc);
    }
    __syncthreads();   // ring memory is re-used by block_sum
    const PairParams pr = a.pp[p];
    const double* tsp = a.ts + (long)p * a.lda;
    const double* al = alpha + (long)p * a.lda;
    double xr[8], ar[8], xc[4][2], ac[4][2];
#pragma unroll
    for (int mi = 0; mi < 8; ++mi) { xr[mi] = tsp[I * TB + tc.row(mi)]; ar[mi] = al[I * TB + tc.row(mi)]; }
#pragma unroll
    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
        for (int e = 0; e < 2; ++e) { xc[ni][e] = tsp[J * TB + tc.col(ni, e)]; ac[ni][e] = al[J * TB + tc.col(ni, e)]; }
    // Off-diagonal tiles stand for (I,J) and (J,I): weight 2.  On a diagonal tile only the 8x8 blocks on or below
    // the diagonal were computed: blocks strictly below count twice, diagonal blocks hold both (r,c) and (c,r).
    double s[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int mi = 0; mi < 8; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
            const int gr = tc.rgroup(mi), gc = tc.cgroup(ni);
            if (I == J && gc > gr) continue;
            const double wgt = (I != J || gc < gr) ? 2.0 : 1.0;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int r = I * TB + tc.row(mi), c = J * TB + tc.col(ni, e);
                if (r < a.m && c < a.m) {
                    const double w = ar[mi] * ac[ni][e] - acc.v[mi][ni][e];
                    if (r == c) {
                        s[0] += w * pr.sig2;
                        s[2] += w;
                    } else {
                        const double d = xr[mi] - xc[ni][e];
                        const double d2 = d * d;
                        double kr, dkl;        // sigma^2 R_ij and dK_ij / dlog(ell)
                        if (FAM == 0) {
                            kr = pr.sig2 * gpbo_exp_neg(-0.5 * d2);
                            dkl = kr * d2;
                        } else {
                            const double K = fabs(d) * (FAM == 3 ? 1.7320508075688772 : 2.23606797749979);
                            const double ex = gpbo_exp_neg(-K);
                            kr = pr.sig2 * ((FAM == 3) ? (1.0 + K) * ex : (1.0 + K + K * K / 3.0) * ex);
                            dkl = pr.sig2 * ((FAM == 3) ? 3.0 * d2 * ex : 5.0 / 3.0 * d2 * (K + 1.0) * ex);
                        }
                        s[0] += wgt * (w * kr);
                        s[1] += wgt * (w * dkl);
                    }
                }
            }
        }
    double tot[3];
    block_sum<3>(s, smem, tot);
    if (tc.tid == 0) {
        double* o = part + ((long)p * ntiles + q) * 4;
        o[0] = tot[0]; o[1] = tot[1]; o[2] = tot[2]; o[3] = 0.0;
    }
}

// ---- finalize: LML and gradient from the partial sums (one CTA per pair) ---------------------
// LML = -1/2 y'alpha - sum log L_ii - m/2 log 2pi (_gpr.py:613-617); grad = 1/2 (s0, s1, chi s2).
__global__ void __launch_bounds__(NTHR, 1)
finalize_kernel(MatArgs a, const double* __restrict__ ypad, const double* __restrict__ alpha,
                const double* __restrict__ part, int ntiles, double* __restrict__ lml, double* __restrict__ grad,
                int* __restrict__ status_out, int with_grad) {
    __shared__ double red[32];
    const int p = blockIdx.x, tid = threadIdx.x;
    const PairParams pr = a.pp[p];
    const double* yp = ypad + (long)pr.gp * a.lda;
    const double* al = alpha + (long)p * a.lda;
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k = tid; k < a.m; k += NTHR) v[0] += yp[k] * al[k];
    if (with_grad)
        for (int q = tid; q < ntiles; q += NTHR) {
            const double* o = part + ((long)p * ntiles + q) * 4;
            v[1] += o[0]; v[2] += o[1]; v[3] += o[2];
        }
    double tot[4];
    block_sum<4>(v, red, tot);
    if (tid == 0) {
        double ld = 0.0;
        for (int j = 0; j < a.T; ++j) ld += a.logdet[(long)p * a.T + j];
        const int st = a.status[p];
        const double val = -0.5 * tot[0] - ld - 0.5 * a.m * 1.8378770664093453;  // log(2 pi)
        const bool ok = (st == 0) && isfinite(val);
        lml[p] = ok ? val : -INFINITY;
        if (with_grad) {
            grad[3 * p + 0] = ok ? 0.5 * tot[1] : 0.0;
            grad[3 * p + 1] = ok ? 0.5 * tot[2] : 0.0;
            grad[3 * p + 2] = ok ? 0.5 * pr.chi * tot[3] : 0.0;
        }
        if (status_out) status_out[p] = ok ? 0 : 1;
    }
}

__global__ void pad_rows_kernel(const double* __restrict__ src, int n, int n_pad, double* __restrict__ dst) {
    const int g = blockIdx.x;
    for (int i = threadIdx.x; i < n_pad; i += blockDim.x) dst[(long)g * n_pad + i] = i < n ? src[(long)g * n + i] : 0.0;
}

}  // namespace gpbo
