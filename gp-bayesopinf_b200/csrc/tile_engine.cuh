// FP64 DMMA tile engine: 128x128 output tile per CTA, 8 warps (2x4), 64x32 accumulator elements per warp,
// k-slices of 16 staged with cp.async into a 4-deep shared ring (see common.cuh).
//
// The 8x8 DMMA blocks of a warp are INTERLEAVED over the tile: warp (wm, wn) owns the 8-row groups
// GR = 2 mi + wm (mi = 0..7) and the 8-column groups GC = 4 ni + wn (ni = 0..3).  Every warp therefore sees the
// same share of any triangular / symmetric structure, and -- because the two warps of an SM sub-partition are
// (0, wn) and (1, wn) -- so does every sub-partition.  That is what makes skipping structurally-zero DMMA blocks
// pay: diagonal (symmetric) tiles issue only the blocks GC <= GR, products with a triangular block inverse
// (D / DT) skip the 8-row or 8-column groups that lie entirely in the zero part.  (With contiguous 64x32 warp
// tiles the skipped work piles up on some sub-partitions and the CTA is no faster.)
//
// Stage hand-over uses two mbarriers per stage instead of __syncthreads():
//   full[s]  (count 256): every thread issues its share of the slice with cp.async and then
//                         cp.async.mbarrier.arrive.noinc -> the phase completes when all copies landed;
//   empty[s] (count 8):   each warp arrives after its last DMMA that reads the stage.
// A warp refills the stage that was consumed one slice earlier in the MIDDLE of the current slice's
// DMMA block, so the wait on empty[] is practically never blocking and warps may drift by half a slice.
// Measured on B200 (tools/mma_sweep.cu, K^-1 tile product at m = 4096): 86.5 % of the DMMA issue peak with
// the __syncthreads ring, 95.9 % with this one (profiles/r01_mma_sweep.txt).
#pragma once
#include <type_traits>

#include <cuda.h>

#include "common.cuh"

namespace gpbo {

struct ThreadCoord {
    int tid, lane, warp, g, c, wm, wn;
    __device__ __forceinline__ ThreadCoord() {
        tid = threadIdx.x; lane = tid & 31; warp = tid >> 5;
        g = lane >> 2; c = lane & 3; wm = warp >> 2; wn = warp & 3;
    }
    // accumulator element (mi, ni, e) -> tile row / col
    __device__ __forceinline__ int rgroup(int mi) const { return 2 * mi + wm; }      // 8-row group index 0..15
    __device__ __forceinline__ int cgroup(int ni) const { return 4 * ni + wn; }      // 8-column group index 0..15
    __device__ __forceinline__ int row(int mi) const { return rgroup(mi) * 8 + g; }
    __device__ __forceinline__ int col(int ni, int e) const { return cgroup(ni) * 8 + 2 * c + e; }
};

// fragment geometry in a staged operand: first row of this lane, rows between consecutive mi / ni
constexpr int FRAG_A_STEP = 16;     // rows between the 8-row groups of one warp
constexpr int FRAG_B_STEP = 32;     // rows (= output columns) between the 8-column groups of one warp

// ---- the stage ring ---------------------------------------------------------------------------
// `count` = slices pushed through the ring so far by this CTA; it is carried across successive loops of
// one kernel so that barrier phase parities stay consistent without re-initialising the barriers.
struct Ring {
    uint64_t* full;
    uint64_t* empty;
    int count;
};

// bars: 2 * NSTAGE mbarriers in (static) shared memory.  Ends with __syncthreads().
__device__ __forceinline__ void ring_init(Ring& r, uint64_t* bars) {
    r.full = bars;
    r.empty = bars + NSTAGE;
    r.count = 0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&bars[s], NTHR);
            mbar_init(&bars[NSTAGE + s], NTHR / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::);
    }
    __syncthreads();
}

// Runs nk slices through the ring.  stage(st, kt): issue this thread's cp.async for slice kt into stage st.
// compute(st, kt, half): the DMMA work of slice kt (half = integral_constant 0 / 1: first / second BK/8 k-steps).
// `prefilled`: the first NSTAGE - 1 slices were already issued by ring_prefill (same nk, same stage functor).
template <class STAGE, class COMPUTE>
__device__ __forceinline__ void ring_pipeline(Ring& ring, int nk, STAGE stage, COMPUTE compute, bool prefilled = false) {
    if (nk <= 0) return;
    const int lane = threadIdx.x & 31;
    const int base = ring.count;
    auto push = [&](int kt) {
        const int gi = base + kt;
        const int st = gi % NSTAGE;
        if (gi >= NSTAGE) mbar_wait(&ring.empty[st], ((gi / NSTAGE) - 1) & 1);
        stage(st, kt);
        mbar_cp_arrive(&ring.full[st]);
    };
    if (!prefilled) {
#pragma unroll
        for (int s = 0; s < NSTAGE - 1; ++s)
            if (s < nk) push(s);
    }
    for (int kt = 0; kt < nk; ++kt) {
        const int gi = base + kt;
        const int cs = gi % NSTAGE;
        mbar_wait(&ring.full[cs], (gi / NSTAGE) & 1);
        compute(cs, kt, std::integral_constant<int, 0>{});
        const int nx = kt + NSTAGE - 1;
        if (nx < nk) push(nx);
        compute(cs, kt, std::integral_constant<int, 1>{});
        __syncwarp();
        if (lane == 0) mbar_arrive(&ring.empty[cs]);
    }
    ring.count = base + nk;
}

// Issue the first NSTAGE - 1 slices of a pipeline ahead of time (e.g. before an epilogue's register math), so that
// their global -> shared latency is hidden; the matching ring_pipeline call passes prefilled = true.
// Every warp must have finished reading the ring memory the stages are written to (__syncthreads() before).
template <class STAGE>
__device__ __forceinline__ void ring_prefill(Ring& ring, int nk, STAGE stage) {
    const int base = ring.count;
#pragma unroll
    for (int s = 0; s < NSTAGE - 1; ++s)
        if (s < nk) {
            const int gi = base + s;
            const int st = gi % NSTAGE;
            if (gi >= NSTAGE) mbar_wait(&ring.empty[st], ((gi / NSTAGE) - 1) & 1);
            stage(st, s);
            mbar_cp_arrive(&ring.full[st]);
        }
}

// Stage one 128 x 16 operand slice (rows `ld` apart in global memory) into padded shared rows.
__device__ __forceinline__ void stage_slice(double* s, const double* __restrict__ g, long ld, int tid) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = tid + i * NTHR;
        const int r = q >> 3, cc = q & 7;
        cp_async16(s + r * LDT + cc * 2, g + (long)r * ld + cc * 2);
    }
}

// structural-zero skipping.  A predicated-off DMMA still occupies the tensor pipe (measured, tools/dmma_pred.cu:
// 16 of 32 DMMAs predicated off or individually branched over -> same time; one branch around the 16 -> half), so
// skipping is done by dispatching -- switch on the warp or on the slice index -- to bodies that simply do not
// contain the dead DMMAs.
constexpr int SKIP_SYM = 1;         // symmetric output tile: only blocks GC <= GR            (switch on the warp)
constexpr int SKIP_A_UP = 2;        // A[r][k] != 0 only for k >= r  (DT as the row operand)    (switch on kt)
constexpr int SKIP_A_LO = 4;        // A[r][k] != 0 only for k <= r  (D as the row operand)
constexpr int SKIP_B_UP = 8;        // B[n][k] != 0 only for k >= n  (DT as the column operand)
constexpr int SKIP_B_LO = 16;       // B[n][k] != 0 only for k <= n  (D as the column operand)

// Where the four lanes c of a DMMA k-step ks read their k element inside a staged row (doubles from the row start).
//   KoffPadded : padded cp.async rows, natural order       k = 4 ks + c           (c is folded into the base pointer)
//   KoffSwz    : dense 128-byte TMA rows under the 128-byte swizzle, PERMUTED k  k = 8 (c >> 1) + 2 ks + (c & 1), i.e.
//                16-byte chunk 4 (c >> 1) + ks, which the swizzle stores at chunk (4 (c >> 1) + ks) ^ (row & 7).  Both
//                operands use the same permutation, so the contraction is unchanged; the 16 lanes of a half warp
//                (row & 7 = g in 0..3 or 4..7, c = 0..3) hit 16 distinct 8-byte bank pairs -- conflict free without
//                padding (tools/mma_tma.cu).
struct KoffPadded {
    __device__ __forceinline__ int operator()(int ks) const { return ks * 4; }
};
struct KoffSwz {
    int o[BK / 4];
    __device__ __forceinline__ KoffSwz(int g, int c) {
#pragma unroll
        for (int ks = 0; ks < BK / 4; ++ks) o[ks] = ((((c >> 1) * 4 + ks) ^ g) << 1) + (c & 1);
    }
    __device__ __forceinline__ int operator()(int ks) const { return o[ks]; }
};

// Two of the four k-steps (HALF = 0: ks 0,1; HALF = 1: ks 2,3) of DMMA on one staged pair of slices, restricted
// to the accumulator blocks mi in [MI0, MI1), ni in [NI0, NI1).
// sa/sb already point at this thread's first fragment element: s?[(w? * 8 + g) * stride + c] (padded rows) or
// s?[(w? * 8 + g) * stride] (swizzled rows).
template <int SA_STRIDE, int SB_STRIDE, int HALF, int MI0 = 0, int MI1 = 8, int NI0 = 0, int NI1 = 4, class KOFF = KoffPadded>
__device__ __forceinline__ void mma_half(Acc& acc, const double* sa, const double* sb, const KOFF& ko = KOFF()) {
#pragma unroll
    for (int ks = HALF * (BK / 8); ks < (HALF + 1) * (BK / 8); ++ks) {
        double a[8], b[4];
#pragma unroll
        for (int mi = MI0; mi < MI1; ++mi) a[mi] = sa[mi * FRAG_A_STEP * SA_STRIDE + ko(ks)];
#pragma unroll
        for (int ni = NI0; ni < NI1; ++ni) b[ni] = sb[ni * FRAG_B_STEP * SB_STRIDE + ko(ks)];
#pragma unroll
        for (int mi = MI0; mi < MI1; ++mi)
#pragma unroll
            for (int ni = NI0; ni < NI1; ++ni) dmma884(acc.v[mi][ni], a[mi], b[ni]);
    }
}

// Same for a symmetric (diagonal) tile: warp (WM, WN) computes only its blocks with 4 ni + WN <= 2 mi + WM.
template <int SA_STRIDE, int SB_STRIDE, int HALF, int WM, int WN, class KOFF>
__device__ __forceinline__ void mma_half_sym(Acc& acc, const double* sa, const double* sb, const KOFF& ko) {
#pragma unroll
    for (int ks = HALF * (BK / 8); ks < (HALF + 1) * (BK / 8); ++ks) {
        double a[8], b[4];
#pragma unroll
        for (int mi = 0; mi < 8; ++mi)
            if (WN <= 2 * mi + WM) a[mi] = sa[mi * FRAG_A_STEP * SA_STRIDE + ko(ks)];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
            if (4 * ni + WN <= 14 + WM) b[ni] = sb[ni * FRAG_B_STEP * SB_STRIDE + ko(ks)];
#pragma unroll
        for (int mi = 0; mi < 8; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
                if (4 * ni + WN <= 2 * mi + WM) dmma884(acc.v[mi][ni], a[mi], b[ni]);
    }
}

template <int SA_STRIDE, int SB_STRIDE, int HALF, class KOFF = KoffPadded>
__device__ __forceinline__ void mma_half_sym_dispatch(Acc& acc, const double* sa, const double* sb, int warp,
                                                      const KOFF& ko = KOFF()) {
    switch (warp) {   // warp = wm * 4 + wn
        case 0: mma_half_sym<SA_STRIDE, SB_STRIDE, HALF, 0, 0>(acc, sa, sb, ko); break;
        case 1: mma_half_sym<SA_STRIDE, SB_STRIDE, HALF, 0, 1>(acc, sa, sb, ko); break;
        case 2: mma_half_sym<SA_STRIDE, SB_STRIDE, HALF, 0, 2>(acc, sa, sb, ko); break;
        case 3: mma_half_sym<SA_STRIDE, SB_STRIDE, HALF, 0, 3>(acc, sa, sb, ko); break;
        case 4: mma_half_sym<SA_STRIDE, SB_STRIDE, HALF, 1, 0>(acc, sa, sb, ko); break;
        case 5: mma_half_sym<SA_STRIDE, SB_STRIDE, HALF, 1, 1>(acc, sa, sb, ko); break;
        case 6: mma_half_sym<SA_STRIDE, SB_STRIDE, HALF, 1, 2>(acc, sa, sb, ko); break;
        default: mma_half_sym<SA_STRIDE, SB_STRIDE, HALF, 1, 3>(acc, sa, sb, ko); break;
    }
}

// One slice (kt = 0..7) of a k-block in which an operand is a triangular block inverse: the 8-row (8-column)
// groups that lie entirely in its zero part are left out.  With the interleaved layout the live set is the
// same for every warp:  A_UP: mi <= kt;   A_LO: mi >= kt;   B_UP: ni <= (2 kt + 1) / 4;   B_LO: ni >= ceil((2 kt - 3) / 4).
// (The k permutation of KoffSwz stays inside the 16-wide slice, so the slice-level zero structure is the same.)
template <int SA_STRIDE, int SB_STRIDE, int HALF, int KIND, int KT, class KOFF>
__device__ __forceinline__ void mma_half_tri_case(Acc& acc, const double* sa, const double* sb, const KOFF& ko) {
    constexpr int MI0 = (KIND == SKIP_A_LO) ? KT : 0;
    constexpr int MI1 = (KIND == SKIP_A_UP) ? KT + 1 : 8;
    constexpr int NI0 = (KIND == SKIP_B_LO) ? (2 * KT - 3 > 0 ? (2 * KT - 3 + 3) / 4 : 0) : 0;
    constexpr int NI1 = (KIND == SKIP_B_UP) ? (2 * KT + 1) / 4 + 1 : 4;
    mma_half<SA_STRIDE, SB_STRIDE, HALF, MI0, MI1, NI0, NI1, KOFF>(acc, sa, sb, ko);
}

template <int SA_STRIDE, int SB_STRIDE, int HALF, int KIND, class KOFF = KoffPadded>
__device__ __forceinline__ void mma_half_tri_dispatch(Acc& acc, const double* sa, const double* sb, int kt,
                                                      const KOFF& ko = KOFF()) {
    switch (kt) {
        case 0: mma_half_tri_case<SA_STRIDE, SB_STRIDE, HALF, KIND, 0>(acc, sa, sb, ko); break;
        case 1: mma_half_tri_case<SA_STRIDE, SB_STRIDE, HALF, KIND, 1>(acc, sa, sb, ko); break;
        case 2: mma_half_tri_case<SA_STRIDE, SB_STRIDE, HALF, KIND, 2>(acc, sa, sb, ko); break;
        case 3: mma_half_tri_case<SA_STRIDE, SB_STRIDE, HALF, KIND, 3>(acc, sa, sb, ko); break;
        case 4: mma_half_tri_case<SA_STRIDE, SB_STRIDE, HALF, KIND, 4>(acc, sa, sb, ko); break;
        case 5: mma_half_tri_case<SA_STRIDE, SB_STRIDE, HALF, KIND, 5>(acc, sa, sb, ko); break;
        case 6: mma_half_tri_case<SA_STRIDE, SB_STRIDE, HALF, KIND, 6>(acc, sa, sb, ko); break;
        default: mma_half_tri_case<SA_STRIDE, SB_STRIDE, HALF, KIND, 7>(acc, sa, sb, ko); break;
    }
}

// Where slice kt of the two operands lives in global memory: 128 rows each, `ld*` doubles apart,
// 16 contiguous doubles per row starting at a / b.
struct SliceSrc {
    const double* a;
    long lda;
    const double* b;
    long ldb;
};

// acc += A * B^T over nk k-slices; src(kt) -> SliceSrc.  SAME: both operands are the same rows
// (diagonal tiles) -> staged once (src.b ignored) and only the blocks on or below the diagonal are computed
// (the rest of acc stays zero).  TRI1: one SKIP_* kind that holds for the first tri_nk slices (by default the first
// k-block, slices 0..7), e.g. SKIP_A_UP when the row operand of that block is a transposed block inverse (ignored on
// SAME tiles); tri_nk = 0 when the loop starts past that block.  On return every warp has finished its
// DMMAs but other warps may still be reading the ring: callers __syncthreads() before re-using `smem`.
template <bool SAME, int TRI1 = 0, class SRC>
__device__ __forceinline__ void gemm_nt_loop(Acc& acc, SRC src, int nk, double* smem, Ring& ring,
                                             const ThreadCoord& tc, int tri_nk = TB / BK) {
    double* sA = smem;
    double* sB = smem + NSTAGE * STAGE_DBL;
    const int oa = (tc.wm * 8 + tc.g) * LDT + tc.c;
    const int ob = (tc.wn * 8 + tc.g) * LDT + tc.c;
    ring_pipeline(
        ring, nk,
        [&](int st, int kt) {
            const SliceSrc s = src(kt);
            stage_slice(sA + st * STAGE_DBL, s.a, s.lda, tc.tid);
            if (!SAME) stage_slice(sB + st * STAGE_DBL, s.b, s.ldb, tc.tid);
        },
        [&](int st, int kt, auto half) {
            const double* sa = sA + st * STAGE_DBL + oa;
            const double* sb = (SAME ? sA : sB) + st * STAGE_DBL + ob;
            constexpr int H = decltype(half)::value;
            if (SAME)
                mma_half_sym_dispatch<LDT, LDT, H>(acc, sa, sb, tc.warp);
            else if (TRI1 != 0 && kt < tri_nk)
                mma_half_tri_dispatch<LDT, LDT, H, TRI1>(acc, sa, sb, kt);
            else
                mma_half<LDT, LDT, H>(acc, sa, sb);
        });
}

// ---- the same main loop with TMA staging ---------------------------------------------------------------------
// Operand slices are fetched by cp.async.bulk.tensor (SASS UTMALDG) issued by ONE thread: a 16 x 128 box of a 2-D
// tensor map (inner dimension = k, 128-byte swizzle) lands as 128 dense 128-byte rows; the mbarrier of the stage gets
// the byte count with arrive.expect_tx and completes when the data has landed.  The 255 other threads do nothing but
// wait, load fragments and issue DMMAs: 97.9 % of the DMMA issue peak on the K^-1 tile product against 95.9 % for the
// LDGSTS ring (tools/mma_tma.cu, profiles/r02b_mma_tma.txt); three stages do as well as four.
struct TmaMaps {
    CUtensorMap A;    // [cap * m_pad rows][m_pad]   the pairs' factor / inverse buffers
    CUtensorMap D;    // [cap * T * 128 rows][128]   inv(L_jj)
    CUtensorMap DT;   // [cap * T * 128 rows][128]   inv(L_jj)^T
};

// Slice kt of the two operands as tensor-map coordinates: {k, row} of the box origin.
struct TmaSlice {
    const CUtensorMap* ma;
    int ka, ra;
    const CUtensorMap* mb;
    int kb, rb;
};

// The dynamic shared window starts right after the kernel's static shared variables, at whatever offset that is:
// kernels that stage with TMA round their base up to 1024 bytes themselves and are launched with SMEM_ALIGN_PAD extra.
constexpr int SMEM_ALIGN_PAD = 1024;
__device__ __forceinline__ double* smem_align_1024(double* raw) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(raw);
    return reinterpret_cast<double*>(reinterpret_cast<char*>(raw) + ((1024u - (a & 1023u)) & 1023u));
}

constexpr int TMA_STAGE_DBL = TB * BK;                                 // dense rows: 16 KB per operand per stage
constexpr int TMA_MAIN_SMEM = NSTAGE * 2 * TMA_STAGE_DBL * 8;          // 131072 B

__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
    uint32_t a = (uint32_t)__cvta_generic_to_shared(b);
    asm volatile("{ .reg .b64 t; mbarrier.arrive.expect_tx.shared.b64 t, [%0], %1; }\n" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    uint32_t d = (uint32_t)__cvta_generic_to_shared(dst), b = (uint32_t)__cvta_generic_to_shared(bar);
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n"
        ::"r"(d), "l"(map), "r"(c0), "r"(c1), "r"(b) : "memory");
}

// bars: 2 * NSTAGE mbarriers; full: one arrival (the producer's expect_tx) + the transaction bytes, empty: one per warp.
__device__ __forceinline__ void ring_init_tma(Ring& r, uint64_t* bars) {
    r.full = bars;
    r.empty = bars + NSTAGE;
    r.count = 0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&bars[s], 1);
            mbar_init(&bars[NSTAGE + s], NTHR / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::);
    }
    __syncthreads();
}

// acc += A * B^T over nk k-slices, src(kt) -> TmaSlice; SAME / TRI1 as in gemm_nt_loop.  smem must be 1024-byte aligned
// (swizzle atom) and must not have been written through the generic proxy since the last TMA use without a
// fence.proxy.async (it is not, in the kernels that use this: the loop runs once, first thing).
template <bool SAME, int TRI1 = 0, class SRC>
__device__ __forceinline__ void gemm_nt_loop_tma(Acc& acc, SRC src, int nk, double* smem, Ring& ring,
                                                 const ThreadCoord& tc, int tri_nk = TB / BK) {
    if (nk <= 0) return;
    double* sA = smem;
    double* sB = smem + NSTAGE * TMA_STAGE_DBL;
    const KoffSwz ko(tc.g, tc.c);
    const int oa = (tc.wm * 8 + tc.g) * BK;
    const int ob = (tc.wn * 8 + tc.g) * BK;
    const int base = ring.count;
    auto push = [&](int kt) {
        const int gi = base + kt;
        const int st = gi % NSTAGE;
        if (gi >= NSTAGE) mbar_wait(&ring.empty[st], ((gi / NSTAGE) - 1) & 1);
        const TmaSlice t = src(kt);
        mbar_expect_tx(&ring.full[st], (SAME ? 1 : 2) * TMA_STAGE_DBL * 8);
        tma_load_2d(sA + st * TMA_STAGE_DBL, t.ma, t.ka, t.ra, &ring.full[st]);
        if (!SAME) tma_load_2d(sB + st * TMA_STAGE_DBL, t.mb, t.kb, t.rb, &ring.full[st]);
    };
    if (tc.tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE - 1; ++s)
            if (s < nk) push(s);
    }
    for (int kt = 0; kt < nk; ++kt) {
        const int gi = base + kt;
        const int cs = gi % NSTAGE;
        const int nx = kt + NSTAGE - 1;
        if (tc.tid == 0 && nx < nk) push(nx);        // refill of the stage consumed one slice ago, before this slice's DMMAs
        mbar_wait(&ring.full[cs], (gi / NSTAGE) & 1);
        const double* sa = sA + cs * TMA_STAGE_DBL + oa;
        const double* sb = (SAME ? sA : sB) + cs * TMA_STAGE_DBL + ob;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (SAME) {
                if (h == 0) mma_half_sym_dispatch<BK, BK, 0>(acc, sa, sb, tc.warp, ko);
                else mma_half_sym_dispatch<BK, BK, 1>(acc, sa, sb, tc.warp, ko);
            } else if (TRI1 != 0 && kt < tri_nk) {
                if (h == 0) mma_half_tri_dispatch<BK, BK, 0, TRI1>(acc, sa, sb, kt, ko);
                else mma_half_tri_dispatch<BK, BK, 1, TRI1>(acc, sa, sb, kt, ko);
            } else {
                if (h == 0) mma_half<BK, BK, 0, 0, 8, 0, 4>(acc, sa, sb, ko);
                else mma_half<BK, BK, 1, 0, 8, 0, 4>(acc, sa, sb, ko);
            }
        }
        __syncwarp();
        if (tc.lane == 0) mbar_arrive(&ring.empty[cs]);
    }
    ring.count = base + nk;
}

// Store the accumulator tile into a shared 128x128 tile with row stride LD.
template <int LD>
__device__ __forceinline__ void acc_to_smem(const Acc& acc, double* S, const ThreadCoord& tc) {
#pragma unroll
    for (int mi = 0; mi < 8; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
            double* p = S + tc.row(mi) * LD + tc.col(ni, 0);
            p[0] = acc.v[mi][ni][0];
            p[1] = acc.v[mi][ni][1];
        }
}

// out += S * Dm^T : S is a shared 128x128 tile [r][k] (stride LDS), complete and visible to the CTA;
// Dm is a LOWER-TRIANGULAR 128x128 global block (a block inverse D, row stride 128) whose rows [n][k] are streamed
// through `stages`; column groups that lie entirely above the diagonal of Dm are skipped.
// The slices of a 128 x 128 block inverse Dm for the epilogue products below, issued early.
__device__ __forceinline__ void epi_prefill_D(const double* __restrict__ Dm, double* stages, Ring& ring,
                                              const ThreadCoord& tc) {
    ring_prefill(ring, TB / BK, [&](int st, int kt) { stage_slice(stages + st * STAGE_DBL, Dm + kt * BK, TB, tc.tid); });
}

__device__ __forceinline__ void epi_product_SxDt(Acc& out, const double* S, const double* __restrict__ Dm,
                                                 double* stages, Ring& ring, const ThreadCoord& tc,
                                                 bool prefilled = false) {
    const double* sa0 = S + (tc.wm * 8 + tc.g) * LDS + tc.c;
    const int ob = (tc.wn * 8 + tc.g) * LDT + tc.c;
    ring_pipeline(
        ring, TB / BK, [&](int st, int kt) { stage_slice(stages + st * STAGE_DBL, Dm + kt * BK, TB, tc.tid); },
        [&](int st, int kt, auto half) {
            mma_half_tri_dispatch<LDS, LDT, decltype(half)::value, SKIP_B_LO>(out, sa0 + kt * BK,
                                                                              stages + st * STAGE_DBL + ob, kt);
        },
        prefilled);
}

// out += Dm * G : Dm is a LOWER-TRIANGULAR 128x128 global block [r][k] (a block inverse D) streamed through
// `stages`; G is a shared 128x128 tile stored [k][n] (stride LDS), complete and visible to the CTA.
__device__ __forceinline__ void epi_product_DxG(Acc& out, const double* __restrict__ Dm, const double* G,
                                                double* stages, Ring& ring, const ThreadCoord& tc,
                                                bool prefilled = false) {
    const int oa = (tc.wm * 8 + tc.g) * LDT + tc.c;
    ring_pipeline(
        ring, TB / BK, [&](int st, int kt) { stage_slice(stages + st * STAGE_DBL, Dm + kt * BK, TB, tc.tid); },
        [&](int st, int kt, auto half) {
            constexpr int H = decltype(half)::value;
            const double* sa = stages + st * STAGE_DBL + oa;
            // B fragment: element (k = kt*16 + ks*4 + c, n = cgroup(ni)*8 + g) of G[k][n]
            const double* sb = G + (kt * BK + tc.c) * LDS + tc.wn * 8 + tc.g;
            auto body = [&](auto mi0) {     // rows of Dm with k <= r only: row groups mi >= kt
                constexpr int MI0 = decltype(mi0)::value;
#pragma unroll
                for (int ks = H * (BK / 8); ks < (H + 1) * (BK / 8); ++ks) {
                    double a[8], b[4];
#pragma unroll
                    for (int mi = MI0; mi < 8; ++mi) a[mi] = sa[mi * FRAG_A_STEP * LDT + ks * 4];
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) b[ni] = sb[ks * 4 * LDS + ni * FRAG_B_STEP];
#pragma unroll
                    for (int mi = MI0; mi < 8; ++mi)
#pragma unroll
                        for (int ni = 0; ni < 4; ++ni) dmma884(out.v[mi][ni], a[mi], b[ni]);
                }
            };
            switch (kt) {
                case 0: body(std::integral_constant<int, 0>{}); break;
                case 1: body(std::integral_constant<int, 1>{}); break;
                case 2: body(std::integral_constant<int, 2>{}); break;
                case 3: body(std::integral_constant<int, 3>{}); break;
                case 4: body(std::integral_constant<int, 4>{}); break;
                case 5: body(std::integral_constant<int, 5>{}); break;
                case 6: body(std::integral_constant<int, 6>{}); break;
                default: body(std::integral_constant<int, 7>{}); break;
            }
        },
        prefilled);
}

}  // namespace gpbo
