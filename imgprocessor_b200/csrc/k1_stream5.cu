// K1, streaming variant for the 5x5 window (medianThreshold(size=5), filters/medianThreshold.py:7-30): the same
// warp-specialised TMA pipeline as k1_stream.cu with a 5-row register window.
//
//   * work unit = (frame, 112-column strip, segment of rows); CTA = 4 consumer warps + 1 producer warp; the producer's
//     elected lane streams 8-row boxes of raw / dark / flat through a 4-stage shared-memory ring (full / empty mbarriers).
//   * each consumer lane owns one image column of its warp's 28-column slice (+2 halo lanes on each side; halo and
//     out-of-frame lanes read the mirrored column = scipy 'reflect').  Per row: pointwise value in float64 registers,
//     the four horizontal neighbours by warp shuffle, a 9-comparator sort of the horizontal quintuple — shared by the
//     five windows that row takes part in —, and the generated 57-comparator selection network (median25_net.inc)
//     over this quintuple and the four previous rows' quintuples held in registers.  The window holds order-preserving
//     integer keys: a compare-exchange is one VIMNMX plus max = a + b - min as two IMADs (FMA pipe), because two
//     FMNMX per exchange saturate the half-rate ALU pipe.
//   * vertical 'reflect': rows -1, -2 are rows 0, 1 (the window is primed with Q1, Q0, Q0, Q1), rows H, H+1 are rows
//     H-1, H-2 (two more emits after the last row).
//
// Same arithmetic as the tile kernels (imgcorr_core.cuh): results are bit-identical (tests/test_gpu_parity.py).
#include "imgcorr_kernels.cuh"
#include "imgcorr_tma.cuh"

namespace imgcorr {

__constant__ int k5_one = 1, k5_minus_one = -1;   // run-time values for ptxas: keeps the two IMADs from folding into IADD3
template <> __device__ __forceinline__ void cswap<OrdKey>(OrdKey& a, OrdKey& b) {
    const int lo = a.k < b.k ? a.k : b.k;
    int hi;
    asm("{\n\t.reg .s32 t;\n\tmad.lo.s32 t, %1, %4, %2;\n\tmad.lo.s32 %0, %3, %5, t;\n\t}"
        : "=r"(hi) : "r"(a.k), "r"(b.k), "r"(lo), "r"(k5_one), "r"(k5_minus_one));
    b.k = hi;
    a.k = lo;
}

namespace {

constexpr int K5_HW = 2;                    // halo width
constexpr int K5_CW = 4;                    // consumer warps per CTA
constexpr int K5_SW = 32 - 2 * K5_HW;       // 28 output columns per consumer warp
constexpr int K5_TW = K5_CW * K5_SW;        // 112 output columns per strip
#ifndef K5_MINB_V
#define K5_MINB_V 3
#endif
#ifndef K5_R_V
#define K5_R_V 8
#endif
#ifndef K5_NSTAGE_V
#define K5_NSTAGE_V 4
#endif
constexpr int K5_R = K5_R_V;                // rows per pipeline stage
constexpr int K5_NSTAGE = K5_NSTAGE_V;
constexpr int K5_MAPW = 128;                // float32 box: tx0-4 .. tx0+123
constexpr int K5_MAPX = 4;
constexpr int K5_THREADS = (K5_CW + 1) * 32;

template <typename RawT> struct Box5 {
    static constexpr int XOFF = 16 / (int)sizeof(RawT);                        // u8 16, u16 8, f32 4
    static constexpr int GRAN = 16 / (int)sizeof(RawT);
    // the box starts at the 16-byte boundary at or left of tx0, minus XOFF: columns tx0-2 .. tx0+113 are inside
    static constexpr int BOXW = ((K5_TW + 2 * XOFF + GRAN - 1) / GRAN) * GRAN;  // u8 144, u16 128, f32 120
    static constexpr size_t raw_bytes = (size_t)K5_R * BOXW * sizeof(RawT);     // multiples of 128
    static constexpr size_t map_bytes = (size_t)K5_R * K5_MAPW * sizeof(float);
    static constexpr size_t stage_bytes = raw_bytes + 2 * map_bytes;
    static constexpr size_t bar_off = K5_NSTAGE * stage_bytes;
    static constexpr size_t total = bar_off + 2 * K5_NSTAGE * sizeof(uint64_t) + 64;
};

template <typename T> struct Raw5;
template <> struct Raw5<uint8_t>  { static __device__ __forceinline__ void ld(uint8_t v, double& d, float& a)  { d = (double)(int)v; a = 0.0f; } };
template <> struct Raw5<uint16_t> { static __device__ __forceinline__ void ld(uint16_t v, double& d, float& a) { d = (double)(int)v; a = 0.0f; } };
template <> struct Raw5<float>    { static __device__ __forceinline__ void ld(float v, double& d, float& a)    { d = (double)v; a = fabsf(v); } };

template <typename OutT> __device__ __forceinline__ OutT out5(const K1Args& a, float v);
template <> __device__ __forceinline__ float    out5<float>(const K1Args&, float v)      { return v; }
template <> __device__ __forceinline__ uint16_t out5<uint16_t>(const K1Args& a, float v) { return quantise<uint16_t>(v, a.q); }
template <> __device__ __forceinline__ uint8_t  out5<uint8_t>(const K1Args& a, float v)  { return quantise<uint8_t>(v, a.q); }

__device__ __noinline__ bool exact5(float x, float b, double thr, int cond) {
    PredicateConst pc;
    pc.thr = thr; pc.cond = cond; pc.lo = 0.f; pc.hi = 0.f; pc.fast_ok = 0;
    return predicate_exact((double)x, (double)b, pc);
}

typedef OrdKey K5T;                         // the window holds order-preserving integer keys (see imgcorr_core.cuh)
__device__ __forceinline__ K5T k5_in(float x) { return to_key(x); }
__device__ __forceinline__ float k5_out(K5T q) { return from_key(q); }
__device__ __forceinline__ K5T k5_shfl_up(K5T c, int d) { K5T r; r.k = __shfl_up_sync(0xffffffffu, c.k, d); return r; }
__device__ __forceinline__ K5T k5_shfl_down(K5T c, int d) { K5T r; r.k = __shfl_down_sync(0xffffffffu, c.k, d); return r; }
struct Q5 { K5T v[5]; };                    // sorted horizontal quintuple of one row

// Row-pair scheme (median25_pair_net.inc, tools/gen_median25_pair.py): two vertically adjacent windows share four of their
// five rows.  Net A reduces the four shared sorted quintuples to the six values of rank 7..12 (the only ones of the 20
// that can be a median of 25), once per PAIR of output rows; net B picks rank 5 of those six plus the window's own fifth
// row, once per output row.  38 + 14/2 exchanges per pair and 3 + 10/2 per row instead of 57 per row.
#include "median25_pair_net.inc"
struct Band6 { K5T v[6]; };
__device__ __forceinline__ Band6 band_of_four(const Q5& r0, const Q5& r1, const Q5& r2, const Q5& r3) {
    K5T v[20];
#pragma unroll
    for (int k = 0; k < 5; ++k) { v[k] = r0.v[k]; v[5 + k] = r1.v[k]; v[10 + k] = r2.v[k]; v[15 + k] = r3.v[k]; }
#define M25_CE(a, b) cswap(v[a], v[b]);
#define M25_LO(a, b) v[a] = vmin(v[a], v[b]);
#define M25_HI(a, b) v[b] = vmax(v[a], v[b]);
    M25A_NET
    Band6 b;
    b.v[0] = v[M25A_BAND0]; b.v[1] = v[M25A_BAND1]; b.v[2] = v[M25A_BAND2];
    b.v[3] = v[M25A_BAND3]; b.v[4] = v[M25A_BAND4]; b.v[5] = v[M25A_BAND5];
    return b;
}
__device__ __forceinline__ K5T median_band_row(const Band6& b, const Q5& own) {
    K5T v[11];
#pragma unroll
    for (int k = 0; k < 6; ++k) v[k] = b.v[k];
#pragma unroll
    for (int k = 0; k < 5; ++k) v[6 + k] = own.v[k];
    M25B_NET
#undef M25_CE
#undef M25_LO
#undef M25_HI
    return v[M25B_RESULT];
}

struct Unit5 {
    int frame, tx0, ys, ye, yl0, n_in, nchunk;
};
__device__ __forceinline__ Unit5 unit5(int unit, int strips, int seg_rows, int H, int n_frames) {
    // frame index fastest: dark / flat rows of one (strip, segment) are read from DRAM once per launch
    Unit5 u;
    u.frame = unit % n_frames;
    int t = unit / n_frames;
    const int strip = t % strips;
    const int seg = t / strips;
    u.tx0 = strip * K5_TW;
    u.ys = seg * seg_rows;
    u.ye = u.ys + seg_rows < H ? u.ys + seg_rows : H;
    u.yl0 = u.ys > 0 ? u.ys - K5_HW : 0;
    const int yl1 = u.ye + K5_HW - 1 < H - 1 ? u.ye + K5_HW - 1 : H - 1;
    u.n_in = yl1 - u.yl0 + 1;
    u.nchunk = (u.n_in + K5_R - 1) / K5_R;
    return u;
}

enum : int { K5_DARK = 1, K5_FLAT = 2, K5_N2N = 4, K5_MASK = 8, K5_CHECK = 16, K5_NZ = 64 };

template <typename RawT, typename OutT, int CFG>
__global__ void __launch_bounds__(K5_THREADS, K5_MINB_V)
k1_stream5_kernel(const __grid_constant__ CUtensorMap tm_raw, const __grid_constant__ CUtensorMap tm_dark,
                  const __grid_constant__ CUtensorMap tm_flat, K1Args a, int strips, int seg_rows, int total_units) {
    using B = Box5<RawT>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* full = (uint64_t*)(smem + B::bar_off);
    uint64_t* empty = full + K5_NSTAGE;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool has_dark = CFG >= 0 ? (CFG & K5_DARK) != 0 : a.dark != nullptr;
    const bool has_flat = CFG >= 0 ? (CFG & K5_FLAT) != 0 : a.flat != nullptr;
    const bool has_mask = CFG >= 0 ? (CFG & K5_MASK) != 0 : a.mask != nullptr;
    const bool check = CFG >= 0 ? (CFG & K5_CHECK) != 0 : true;
    const bool swap = CFG >= 0 ? false : a.raw_swap != 0;
    const int flags = CFG >= 0 ? ((CFG & K5_DARK ? FLAG_DARK : 0) | (CFG & K5_FLAT ? FLAG_FLAT : 0) | (CFG & K5_N2N ? FLAG_NAN_TO_NUM : 0))
                               : a.pw.flags;
    const int H = a.H, W = a.W;

    float* sconst = (float*)(smem + B::bar_off + 2 * K5_NSTAGE * sizeof(uint64_t));      // lo, hi, thr (double)
    if (threadIdx.x == 0) {
        for (int s = 0; s < K5_NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], K5_CW); }
        sconst[0] = a.pred.lo; sconst[1] = a.pred.hi; *(double*)(sconst + 2) = a.pred.thr;
        mbar_init_fence();
    }
    __syncthreads();

    if (warp == K5_CW) {
        // ------------------------------------------------------------------ producer
        if (lane != 0) return;
        const uint32_t tx_bytes = (uint32_t)(B::raw_bytes + (has_dark ? B::map_bytes : 0) + (has_flat ? B::map_bytes : 0));
        uint32_t g = 0;
        for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
            const Unit5 u = unit5(unit, strips, seg_rows, H, a.n_frames);
            for (int k = 0; k < u.nchunk; ++k, ++g) {
                const int stage = g % K5_NSTAGE;
                mbar_wait(&empty[stage], ((g / K5_NSTAGE) & 1) ^ 1);
                uint8_t* base = smem + (size_t)stage * B::stage_bytes;
                const int y = u.yl0 + k * K5_R;
                mbar_expect_tx(&full[stage], tx_bytes);
                // L2 priorities as in k1_stream.cu: raw samples pass once, the calibration maps are read again by every frame / launch
                tma_load_3d_hint(base, &tm_raw, &full[stage], (u.tx0 / B::GRAN) * B::GRAN - B::XOFF, y, u.frame, L2_EVICT_FIRST);
                if (has_dark) tma_load_2d_hint(base + B::raw_bytes, &tm_dark, &full[stage], u.tx0 - K5_MAPX, y, L2_EVICT_LAST);
                if (has_flat) tma_load_2d_hint(base + B::raw_bytes + B::map_bytes, &tm_flat, &full[stage], u.tx0 - K5_MAPX, y, L2_EVICT_LAST);
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    const PointwiseConst pw = a.pw;
    PredicateConst pred = a.pred;
    pred.lo = sconst[0]; pred.hi = sconst[1]; pred.thr = *(const double*)(sconst + 2);
    const int lc = warp * K5_SW - K5_HW + lane;        // strip-local column of this lane: -2 .. 113
    uint32_t g = 0;

    for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
        const Unit5 u = unit5(unit, strips, seg_rows, H, a.n_frames);
        const int gc = u.tx0 + lc;
        const int rc = reflect_index(gc, W);             // scipy 'reflect' in x
        int mcol = rc - (u.tx0 - K5_MAPX);
        mcol = mcol < 0 ? 0 : (mcol > K5_MAPW - 1 ? K5_MAPW - 1 : mcol);
        int rcol = rc - ((u.tx0 / B::GRAN) * B::GRAN - B::XOFF);
        rcol = rcol < 0 ? 0 : (rcol > B::BOXW - 1 ? B::BOXW - 1 : rcol);
        const bool valid = lane >= K5_HW && lane < K5_HW + K5_SW && gc < W;
        const int i_first = u.ys == 0 ? K5_HW : 2 * K5_HW;          // first input row index whose step emits an output row
        const ptrdiff_t o0 = ((ptrdiff_t)u.frame * H + u.yl0 - K5_HW) * W + gc;      // row (yl0 + i - 2) at step i
        OutT* outp = (OutT*)a.out + o0;
        uint8_t* maskp = has_mask ? a.mask + o0 : nullptr;

        Q5 w0, w1, w2, w3;                               // the four previous rows' quintuples, oldest first
        float c1 = 0.f, c2 = 0.f;                        // centre values one / two rows back
        int i = 0;

        auto pixel = [&](const uint8_t* base, int j) -> float {
            RawT rv = ((const RawT*)base)[j * B::BOXW + rcol];
            if (sizeof(RawT) == 2 && swap) rv = (RawT)__byte_perm((unsigned)rv, 0u, 0x0001);
            const float d = has_dark ? ((const float*)(base + B::raw_bytes))[j * K5_MAPW + mcol] : 0.0f;
            const float f = has_flat ? ((const float*)(base + B::raw_bytes + B::map_bytes))[j * K5_MAPW + mcol] : 0.0f;
            double rd; float ra;
            Raw5<RawT>::ld(rv, rd, ra);
            bool ok;
            float x = (CFG >= 0 && (CFG & K5_NZ)) ? pointwise_fast_nz(flags, rd, ra, d, f, ok) : pointwise_fast(flags, rd, ra, d, f, ok);
            if (check) { if (!ok) x = pointwise<float>(pw, rd, d, 0.0f, f); }
            return x;
        };
        auto quint = [&](float x) -> Q5 {
            Q5 q;
            const K5T c = k5_in(x);                      // one conversion per pixel; the neighbours arrive as keys
            q.v[0] = k5_shfl_up(c, 2);
            q.v[1] = k5_shfl_up(c, 1);
            q.v[2] = c;
            q.v[3] = k5_shfl_down(c, 1);
            q.v[4] = k5_shfl_down(c, 2);
            sort5(q.v);
            return q;
        };
        auto median = [&](const Q5& q) -> float {
            K5T v[25];
#pragma unroll
            for (int k = 0; k < 5; ++k) { v[k] = w0.v[k]; v[5 + k] = w1.v[k]; v[10 + k] = w2.v[k]; v[15 + k] = w3.v[k]; v[20 + k] = q.v[k]; }
            return k5_out(median25_sorted_rows(v));
        };
        auto emit = [&](const Q5& q, bool on) {
            const float med = median(q);
            bool rep;
            const bool sure = predicate_certain(c2, med, pred, rep);
            if (on) {
                *outp = out5<OutT>(a, rep ? med : c2);
                if (has_mask) *maskp = rep ? 1 : 0;
            }
            if (__any_sync(0xffffffffu, !sure)) {
                if (!sure && on) {
                    const bool r2 = exact5(c2, med, pred.thr, pred.cond);
                    *outp = out5<OutT>(a, r2 ? med : c2);
                    if (has_mask) *maskp = r2 ? 1 : 0;
                }
            }
        };
        auto push = [&](const Q5& q, float x) {
            w0 = w1; w1 = w2; w2 = w3; w3 = q;
            c2 = c1; c1 = x;
        };
        auto row = [&](const uint8_t* base, int j) {
            const float x = pixel(base, j);
            const Q5 q = quint(x);
            if (i >= i_first) emit(q, valid);            // (warp-uniform: every lane takes part in the vote inside)
            push(q, x);
            if (u.ys == 0 && i == 1) { w0 = w3; w1 = w2; }   // top 'reflect': window (Q1, Q0, Q0, Q1) before row 2
            outp += W;
            if (has_mask) maskp += W;
            ++i;
        };

        for (int k = 0; k < u.nchunk; ++k, ++g) {
            const int stage = g % K5_NSTAGE;
            mbar_wait(&full[stage], (g / K5_NSTAGE) & 1);
            const uint8_t* base = smem + (size_t)stage * B::stage_bytes;
            const int rows = u.n_in - k * K5_R;
            if (k > 0 && rows >= K5_R) {
                // steady state: every row emits and stores are unconditional (lanes without an output pixel write to a
                // private scratch slot).  The ~1e-5 of pixels inside the guard band of the float32 predicate take the exact
                // float64 evaluation out of line; at ~140 instructions per pixel the per-row vote costs nothing (the 3x3
                // kernel defers it to the end of the chunk).
                OutT* op = valid ? outp : (OutT*)a.dump + (size_t)blockIdx.x * K5_THREADS + threadIdx.x;
                uint8_t* mp = has_mask ? (valid ? maskp : (uint8_t*)a.dump + (size_t)(gridDim.x + blockIdx.x) * K5_THREADS * sizeof(OutT) + threadIdx.x) : nullptr;
                const int ostride = valid ? W : 0;
                static_assert(K5_R % 2 == 0, "rows per stage must be even (outputs are produced in vertical pairs)");
#pragma unroll
                for (int j = 0; j < K5_R; j += 2) {
                    // two new rows -> two outputs: windows (w0 w1 w2 w3 qa) and (w1 w2 w3 qa qb) share w1 w2 w3 qa
                    const float xa = pixel(base, j), xb = pixel(base, j + 1);
                    const Q5 qa = quint(xa), qb = quint(xb);
                    const Band6 band = band_of_four(w1, w2, w3, qa);
                    const float med_a = k5_out(median_band_row(band, w0));
                    const float med_b = k5_out(median_band_row(band, qb));
                    bool rep_a, rep_b;
                    const bool sure_a = predicate_certain(c2, med_a, pred, rep_a);
                    const bool sure_b = predicate_certain(c1, med_b, pred, rep_b);
                    if (__any_sync(0xffffffffu, !(sure_a && sure_b))) {
                        if (!sure_a) rep_a = exact5(c2, med_a, pred.thr, pred.cond);
                        if (!sure_b) rep_b = exact5(c1, med_b, pred.thr, pred.cond);
                    }
                    op[0] = out5<OutT>(a, rep_a ? med_a : c2);
                    op[ostride] = out5<OutT>(a, rep_b ? med_b : c1);
                    if (has_mask) { mp[0] = rep_a ? 1 : 0; mp[ostride] = rep_b ? 1 : 0; mp += 2 * ostride; }
                    op += 2 * ostride;
                    push(qa, xa);
                    push(qb, xb);
                }
                outp += (size_t)K5_R * W;
                if (has_mask) maskp += (size_t)K5_R * W;
                i += K5_R;
            } else {
                const int n = rows < K5_R ? rows : K5_R;
                for (int j = 0; j < n; ++j) row(base, j);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
        }
        if (u.ye == H) {
            // bottom 'reflect': output row H-2 sees (H-4 .. H-1, H-1), output row H-1 sees (H-3, H-2, H-1, H-1, H-2)
            const Q5 last = w3, before = w2;
            emit(last, valid);
            push(last, c1);
            outp += W;
            if (has_mask) maskp += W;
            emit(before, valid);
        }
    }
}

template <typename RawT, typename OutT>
cudaError_t launch5_t(const K1Args& a_in, CUtensorMapDataType rdt, int sm_count, int seg_rows, cudaStream_t st) {
    using B = Box5<RawT>;
    K1Args a = a_in;
    const bool check = !a.maps_finite || sizeof(RawT) == 4;
    const int f = a.pw.flags;
    const bool chain = a.dark && a.flat && a.flat_nz && (f & FLAG_DARK) && (f & FLAG_FLAT) && (f & FLAG_NAN_TO_NUM) && !a.mask &&
                       a.pred.cond == COND_GT && !a.raw_swap;
    const bool plain = !(f & (FLAG_DARK | FLAG_FLAT | FLAG_NAN_TO_NUM)) && a.mask && a.pred.cond == COND_GT && !a.raw_swap;
    void (*kern)(const CUtensorMap, const CUtensorMap, const CUtensorMap, K1Args, int, int, int);
    int slot;
    if (chain) a.flat = a.flat_nz;          // zero-free copy: "divide where flat != 0" becomes an unconditional division
    if (chain && !check && a.no_overflow) { kern = k1_stream5_kernel<RawT, OutT, K5_DARK | K5_FLAT | K5_NZ>; slot = 0; }
    else if (chain && !check) { kern = k1_stream5_kernel<RawT, OutT, K5_DARK | K5_FLAT | K5_N2N | K5_NZ>; slot = 1; }
    else if (chain) { kern = k1_stream5_kernel<RawT, OutT, K5_DARK | K5_FLAT | K5_N2N | K5_NZ | K5_CHECK>; slot = 2; }
    else if (plain) { kern = k1_stream5_kernel<RawT, OutT, K5_MASK>; slot = 3; }
    else { kern = k1_stream5_kernel<RawT, OutT, -1>; slot = 4; }

    CUtensorMap tr, td, tf;
    if (!make_tensor_map(&tr, rdt, sizeof(RawT), a.raw, a.W, a.H, a.n_frames, B::BOXW, K5_R)) return cudaErrorInvalidValue;
    if (!make_tensor_map(&td, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.dark ? (const void*)a.dark : a.raw, a.W, a.H, 0, K5_MAPW, K5_R) && a.dark)
        return cudaErrorInvalidValue;
    if (!make_tensor_map(&tf, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.flat ? (const void*)a.flat : a.raw, a.W, a.H, 0, K5_MAPW, K5_R) && a.flat)
        return cudaErrorInvalidValue;
    cudaError_t e_attr = cudaSuccess;
    const int per_sm_k = blocks_per_sm_cached((const void*)kern, K5_THREADS, B::total, &e_attr);     // per (device, kernel)
    if (e_attr != cudaSuccess) return e_attr;
    (void)slot;
    const int strips = (a.W + K5_TW - 1) / K5_TW;
    const long long slots = (long long)sm_count * per_sm_k;
    if (seg_rows <= 0) {
        // equal-cost units: pick the segment height whose unit count fills whole waves of the resident CTAs best, counting
        // the four re-read halo rows per segment against it
        double best = -1.0;
        for (int waves = 1; waves <= 8; ++waves) {
            long long segs_try = slots * waves / ((long long)strips * a.n_frames);
            if (segs_try < 1) continue;
            int rows = (int)((a.H + segs_try - 1) / segs_try);
            if (rows < 2 * K5_R) rows = 2 * K5_R;
            const long long units = (long long)strips * ((a.H + rows - 1) / rows) * a.n_frames;
            const double util = (double)units / (double)(((units + slots - 1) / slots) * slots) * rows / (rows + 4.0);
            if (util > best) { best = util; seg_rows = rows; }
        }
        if (seg_rows <= 0) seg_rows = a.H;
    }
    if (seg_rows < 8) seg_rows = 8;
    // a 1-row last segment would leave its predecessor without the second halo row below it (row H does not exist and the
    // 'reflect' rows are only synthesised by the segment that ends at H)
    while (seg_rows < a.H && a.H % seg_rows == 1) ++seg_rows;
    const int segs = (a.H + seg_rows - 1) / seg_rows;
    const long long total = (long long)strips * segs * a.n_frames;
    if (total > 0x7fffffffLL) return cudaErrorInvalidValue;
    long long grid = slots;
    if (grid > total) grid = total;
    kern<<<(unsigned)grid, K5_THREADS, B::total, st>>>(tr, td, tf, a, strips, seg_rows, (int)total);
    return cudaGetLastError();
}

}  // namespace

bool k1_stream5_eligible(const K1Args& a, int raw_dtype, int out_dtype) {
    if (a.ksize != 5 || a.H < 8) return false;
    if (raw_dtype != DT_U8 && raw_dtype != DT_U16 && raw_dtype != DT_F32) return false;
    if (out_dtype != DT_F32 && out_dtype != DT_U16 && out_dtype != DT_U8) return false;
    if (a.pw.flags & FLAG_DARK_LINEAR) return false;
    if (a.raw_gap) return false;
    if (a.bg) return false;                              // per-frame backgrounds with 5x5: the generic tiles
    const size_t esz = dtype_size(raw_dtype);
    if (((size_t)a.W * esz) % 16 || ((size_t)a.W * 4) % 16) return false;
    if (((size_t)a.H * a.W * esz) % 16) return false;
    if (((uintptr_t)a.raw) % 16) return false;
    if (a.dark && ((uintptr_t)a.dark) % 16) return false;
    if (a.flat && ((uintptr_t)a.flat) % 16) return false;
    return tensor_map_encoder() != nullptr;
}

cudaError_t launch_k1_stream5(const K1Args& a, int raw_dtype, int out_dtype, int sm_count, int seg_rows, cudaStream_t st) {
    switch (raw_dtype) {
        case DT_U8:
            if (out_dtype == DT_F32) return launch5_t<uint8_t, float>(a, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, seg_rows, st);
            if (out_dtype == DT_U8) return launch5_t<uint8_t, uint8_t>(a, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, seg_rows, st);
            if (out_dtype == DT_U16) return launch5_t<uint8_t, uint16_t>(a, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, seg_rows, st);
            break;
        case DT_U16:
            if (out_dtype == DT_F32) return launch5_t<uint16_t, float>(a, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, seg_rows, st);
            if (out_dtype == DT_U16) return launch5_t<uint16_t, uint16_t>(a, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, seg_rows, st);
            if (out_dtype == DT_U8) return launch5_t<uint16_t, uint8_t>(a, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, seg_rows, st);
            break;
        case DT_F32:
            if (out_dtype == DT_F32) return launch5_t<float, float>(a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, seg_rows, st);
            if (out_dtype == DT_U16) return launch5_t<float, uint16_t>(a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, seg_rows, st);
            if (out_dtype == DT_U8) return launch5_t<float, uint8_t>(a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, seg_rows, st);
            break;
    }
    return cudaErrorInvalidValue;
}

}  // namespace imgcorr
