// K1 — fused dark-current subtraction / flat-field division / nan_to_num / NxN median-threshold.
//
// Replaces, for one frame, the reference's
//   image -= bg                              camera/CameraCalibration.py:502
//   image[flat != 0] /= flat[flat != 0]      camera/CameraCalibration.py:525-526
//   image = np.nan_to_num(image)             camera/CameraCalibration.py:561
//   medianThreshold(image, thr, size)        filters/medianThreshold.py:7-30
// with one pass over HBM: raw (2 or 4 B/px) + dark (4) + flat (4) in, corrected float32 (4) out.
//
// This file holds the tile kernels and the dispatcher (launch_k1).  The default paths are the streaming pipelines in
// k1_stream.cu (3x3, and threshold <= 0) and k1_stream5.cu (5x5); the tiles below serve the shapes / dtypes / options
// those do not take (odd widths, float64 frames, framed file images, the linear dark model outside the streaming
// configurations).
//
// Two staging variants share the same compute phases:
//   generic : coalesced ld.global.nc with reflect indexing (any W, any alignment, any dtype)
//   tma     : persistent CTAs, cp.async.bulk.tensor tiles (+halo) of raw/dark/flat into a
//             multi-stage shared-memory ring signalled by mbarriers; out-of-bounds halo
//             (TMA zero fill) is replaced by the mirrored in-tile sample (scipy 'reflect').
// Tile = 128 x TH outputs.  Phase A computes the pointwise value of every pixel of the tile + halo
// once into shared memory (4 pixels per thread-step, 128-bit shared accesses).  Phase B gives
// every thread a pair of adjacent columns and walks it down TH/4 rows: per row one sorted
// pair + two insertions yield the two sorted horizontal triples, each shared by the three
// vertically adjacent windows; three sorted triples combine to the median of 9 (FMNMX3).
// The kernel is instruction-issue bound, not DRAM bound (profiles/), so the structure is chosen to
// minimise issued instructions per pixel.
#include "imgcorr_kernels.cuh"
#include "imgcorr_tma.cuh"

namespace imgcorr {

constexpr int K1_THREADS = 256;
constexpr int K1_TW = 128;          // output columns per tile
constexpr int K1_BOXW = 136;        // staged float32 columns: tx0-4 .. tx0+131
constexpr int K1_XOFF = 4;          // column of tx0 inside the staged float32 box
constexpr int K1_GROUPS = K1_BOXW / 4;   // 34 groups of 4 columns per staged row
constexpr int K1_CPAIRS = K1_TW / 2;     // phase B: 64 column pairs ...
constexpr int K1_RGROUPS = K1_THREADS / K1_CPAIRS;   // ... x 4 row groups

// TMA needs the box to start on a 16-byte boundary of the row (coordinate * element size % 16 == 0) and
// to be a multiple of 16 bytes wide, so the raw tile of a 1- or 2-byte type starts 16 B left of tx0:
template <typename RawT> struct RawBox {
    static constexpr int XOFF = 16 / (int)sizeof(RawT);          // u8: 16, u16: 8, f32: 4
    static constexpr int BOXW = K1_TW + 2 * XOFF;                // u8: 160, u16: 144, f32: 136
};

template <typename T> struct RawIO;
template <> struct RawIO<uint8_t>  { using CT = float;  static __device__ __forceinline__ double ld(uint8_t v)  { return (double)(int)v; } };
template <> struct RawIO<uint16_t> { using CT = float;  static __device__ __forceinline__ double ld(uint16_t v) { return (double)(int)v; } };
template <> struct RawIO<float>    { using CT = float;  static __device__ __forceinline__ double ld(float v)    { return (double)v; } };
template <> struct RawIO<double>   { using CT = double; static __device__ __forceinline__ double ld(double v)   { return v; } };

// integer outputs go through the quantiser with the launch's scale (identity: saturate_cast, as sat_u16 / sat_u8)
template <typename OutT, typename CT> __device__ __forceinline__ OutT to_out(const K1Args& a, CT v);
template <> __device__ __forceinline__ float    to_out<float, float>(const K1Args&, float v)    { return v; }
template <> __device__ __forceinline__ double   to_out<double, float>(const K1Args&, float v)   { return (double)v; }
template <> __device__ __forceinline__ double   to_out<double, double>(const K1Args&, double v) { return v; }
template <> __device__ __forceinline__ uint16_t to_out<uint16_t, float>(const K1Args& a, float v) { return quantise<uint16_t>(v, a.q); }
template <> __device__ __forceinline__ uint8_t  to_out<uint8_t, float>(const K1Args& a, float v)  { return quantise<uint8_t>(v, a.q); }

template <typename T> struct alignas(2 * sizeof(T)) Pair { T x, y; };

// ingest formats (SURVEY §8 f2): big-endian uint16 samples (reader/RAW.py:19-20) and frames separated by small
// headers (reader/elbin.py:23-32) are consumed as stored — byte swap in the load, frame stride with a gap
template <typename RawT> __device__ __forceinline__ RawT raw_fix(RawT v, int) { return v; }
template <> __device__ __forceinline__ uint16_t raw_fix<uint16_t>(uint16_t v, int swap) {
    return swap ? (uint16_t)__byte_perm((unsigned)v, 0u, 0x0001) : v;
}
template <typename RawT> __device__ __forceinline__ const RawT* raw_frame(const K1Args& a, int frame) {
    return (const RawT*)((const char*)a.raw + (size_t)frame * ((size_t)a.H * a.W * sizeof(RawT) + (size_t)a.raw_gap));
}

// ------------------------------------------------------------------------------------------
// pointwise only (ksize == 0): pure streaming kernel; frames in grid.y, no per-pixel modulo
// ------------------------------------------------------------------------------------------
// per-frame background (K1Args::bg): sample i of the dense [n][H][W] block as the float32 dark value of its pixel.  The
// dtype is read at run time: the generic kernels are the fall-back of every allowed pair, and one instantiation serves
// all of them
__device__ __forceinline__ float bg_sample(const K1Args& a, size_t i) {
    if (a.bg_dtype == DT_U8) return (float)__ldg((const uint8_t*)a.bg + i);
    if (a.bg_dtype == DT_U16) return (float)__ldg((const uint16_t*)a.bg + i);
    return __ldg((const float*)a.bg + i);
}

// TT: per-frame exposure times (K1Args::exposures) for the line model: the frame's time replaces pw.exposure_time
template <typename RawT, typename OutT, bool BG, bool TT = false>
__device__ __forceinline__ void k1_pointwise_body(const K1Args& a) {
    using CT = typename RawIO<RawT>::CT;
    const size_t npx = (size_t)a.H * a.W;
    const RawT* raw = raw_frame<RawT>(a, blockIdx.y);
    OutT* out = (OutT*)a.out + (size_t)blockIdx.y * npx;
    PointwiseConst pw = a.pw;
    if (TT) pw.exposure_time = __ldg(a.exposures + blockIdx.y);
    const int swap = a.raw_swap;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npx; p += (size_t)gridDim.x * blockDim.x) {
        float d = BG ? bg_sample(a, (size_t)blockIdx.y * npx + p) : (a.dark ? __ldg(a.dark + p) : 0.0f);
        float s = a.ascent ? __ldg(a.ascent + p) : 0.0f;
        float f = a.flat ? __ldg(a.flat + p) : 0.0f;
        out[p] = to_out<OutT, CT>(a, pointwise<CT>(pw, RawIO<RawT>::ld(raw_fix<RawT>(__ldg(raw + p), swap)), d, s, f));
    }
}
template <typename RawT, typename OutT>
__global__ void __launch_bounds__(256) k1_pointwise_kernel(K1Args a) { k1_pointwise_body<RawT, OutT, false>(a); }
template <typename RawT, typename OutT>
__global__ void __launch_bounds__(256) k1_pointwise_bg_kernel(K1Args a) { k1_pointwise_body<RawT, OutT, true>(a); }
template <typename RawT, typename OutT>
__global__ void __launch_bounds__(256) k1_pointwise_tt_kernel(K1Args a) { k1_pointwise_body<RawT, OutT, false, true>(a); }

// ------------------------------------------------------------------------------------------
// phase B: median-threshold of one tile from the shared pointwise tile xs[TH+2h][K1_BOXW]
// ------------------------------------------------------------------------------------------
template <typename CT>
__device__ __forceinline__ void sorted_row_pair(const CT* p, Sorted3<CT>& A, Sorted3<CT>& B, CT& m0, CT& m1) {
    // p -> column of the first pixel; horizontal triples (p[-1],p[0],p[1]) and (p[0],p[1],p[2])
    const CT l = p[-1];
    const Pair<CT> mm = *reinterpret_cast<const Pair<CT>*>(p);
    const CT r = p[2];
    m0 = mm.x; m1 = mm.y;
    const CT lo = vmin(m0, m1), hi = vmax(m0, m1);
    CT t = vmax(l, lo);
    A.lo = vmin(l, lo); A.mid = vmin(t, hi); A.hi = vmax(t, hi);
    t = vmax(r, lo);
    B.lo = vmin(r, lo); B.mid = vmin(t, hi); B.hi = vmax(t, hi);
}

template <typename OutT, bool VEC>
__device__ __forceinline__ void store_pair(OutT* dst, OutT o0, OutT o1, bool two) {
    if (VEC) {
        Pair<OutT> v; v.x = o0; v.y = o1;
        *reinterpret_cast<Pair<OutT>*>(dst) = v;
    } else {
        dst[0] = o0;
        if (two) dst[1] = o1;
    }
}

template <typename CT, typename OutT, int KS, int TH, bool VEC>
__device__ __forceinline__ void median_phase(const CT* __restrict__ xs, const K1Args& a, const PredicateConst& pred,
                                             int frame, int tx0, int ty0) {
    constexpr int P = TH / K1_RGROUPS;                  // rows per thread
    const int cp = threadIdx.x % K1_CPAIRS;
    const int rg = threadIdx.x / K1_CPAIRS;
    const int c = 2 * cp;                               // first of the two output columns (tile-local)
    const int gx = tx0 + c;
    const int r0 = rg * P;
    int nrows = a.H - (ty0 + r0);
    if (gx >= a.W || nrows <= 0) return;
    if (nrows > P) nrows = P;
    const bool two = gx + 1 < a.W;
    const size_t o0 = ((size_t)frame * a.H + (ty0 + r0)) * a.W + gx;
    OutT* out = (OutT*)a.out + o0;
    uint8_t* mask = a.mask ? a.mask + o0 : nullptr;
    const int W = a.W;

    if (KS == 3) {
        // xs row (tile row r + HALO); window of output row r = xs rows r .. r+2
        const CT* p = xs + (size_t)r0 * K1_BOXW + (K1_XOFF + c);
        Sorted3<CT> a0, b0, a1, b1, a2, b2;
        CT c0, c1, n0, n1;
        sorted_row_pair(p, a0, b0, c0, c1);
        p += K1_BOXW;
        sorted_row_pair(p, a1, b1, c0, c1);
        auto step = [&](int j) {
            p += K1_BOXW;
            sorted_row_pair(p, a2, b2, n0, n1);
            const CT m0 = median9(a0, a1, a2), m1 = median9(b0, b1, b2);
            const bool rep0 = predicate(c0, m0, pred), rep1 = predicate(c1, m1, pred);
            store_pair<OutT, VEC>(out + (size_t)j * W, to_out<OutT, CT>(a, rep0 ? m0 : c0), to_out<OutT, CT>(a, rep1 ? m1 : c1), two);
            if (mask) store_pair<uint8_t, VEC>(mask + (size_t)j * W, (uint8_t)rep0, (uint8_t)rep1, two);
            a0 = a1; a1 = a2; b0 = b1; b1 = b2; c0 = n0; c1 = n1;
        };
        if (nrows == P) {
#pragma unroll
            for (int j = 0; j < P; ++j) step(j);
        } else {
            for (int j = 0; j < nrows; ++j) step(j);
        }
    } else {   // KS == 5
        // one column at a time: walk down the rows keeping the last five SORTED horizontal quintuples in registers
        // (each is sorted once and used by five windows); the loop is fully unrolled so the ring index is static.
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            if (cc == 1 && !two) break;
            const CT* p = xs + (size_t)r0 * K1_BOXW + (K1_XOFF + c + cc - 2);       // xs row r0 = window row 0 of output r0
            CT q[5][5];
            CT ctr[5];
#pragma unroll
            for (int j = 0; j < P + 4; ++j) {
                CT* row = q[j % 5];
#pragma unroll
                for (int dx = 0; dx < 5; ++dx) row[dx] = p[dx];
                ctr[j % 5] = row[2];
                sort5(row);
                p += K1_BOXW;
                if (j >= 4) {
                    const int o = j - 4;                                       // output row inside this thread's run
                    if (o < nrows) {
                        CT w[25];
#pragma unroll
                        for (int k = 0; k < 5; ++k)
#pragma unroll
                            for (int i = 0; i < 5; ++i) w[5 * k + i] = q[(j - 4 + k) % 5][i];
                        const CT med = median25_sorted_rows(w);
                        const CT centre = ctr[(j - 2) % 5];
                        const bool rep = predicate(centre, med, pred);
                        out[(size_t)o * W + cc] = to_out<OutT, CT>(a, rep ? med : centre);
                        if (mask) mask[(size_t)o * W + cc] = rep ? 1 : 0;
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// generic variant: one tile per CTA, reflect indexing on global loads
// ------------------------------------------------------------------------------------------
template <typename RawT, typename OutT, int KS, int TH, bool VEC, bool BG, bool TT = false>
__device__ __forceinline__ void k1_generic_body(const K1Args& a, int tiles_x, int tiles_y) {
    using CT = typename RawIO<RawT>::CT;
    constexpr int HALO = KS / 2;
    constexpr int LH = TH + 2 * HALO;
    constexpr int LW = K1_TW + 2 * HALO;
    __shared__ __align__(16) CT xs[LH * K1_BOXW];

    int t = blockIdx.x;
    const int txi = t % tiles_x; t /= tiles_x;
    const int tyi = t % tiles_y;
    const int frame = t / tiles_y;
    const int tx0 = txi * K1_TW, ty0 = tyi * TH;
    const RawT* raw = raw_frame<RawT>(a, frame);
    PointwiseConst pw = a.pw;
    if (TT) pw.exposure_time = __ldg(a.exposures + frame);
    const int swap = a.raw_swap;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    for (int ly = warp; ly < LH; ly += K1_THREADS / 32) {
        const size_t grow = (size_t)reflect_index(ty0 - HALO + ly, a.H) * a.W;
        CT* xrow = xs + ly * K1_BOXW + (K1_XOFF - HALO);
        for (int lx = lane; lx < LW; lx += 32) {
            const size_t g = grow + reflect_index(tx0 - HALO + lx, a.W);
            float d = BG ? bg_sample(a, (size_t)frame * a.H * a.W + g) : (a.dark ? __ldg(a.dark + g) : 0.0f);
            float s = a.ascent ? __ldg(a.ascent + g) : 0.0f;
            float f = a.flat ? __ldg(a.flat + g) : 0.0f;
            xrow[lx] = pointwise<CT>(pw, RawIO<RawT>::ld(raw_fix<RawT>(__ldg(raw + g), swap)), d, s, f);
        }
    }
    __syncthreads();
    const PredicateConst pred = a.pred;
    median_phase<CT, OutT, KS, TH, VEC>(xs, a, pred, frame, tx0, ty0);
}

template <typename RawT, typename OutT, int KS, int TH, bool VEC>
__global__ void __launch_bounds__(K1_THREADS) k1_generic_kernel(K1Args a, int tiles_x, int tiles_y) {
    k1_generic_body<RawT, OutT, KS, TH, VEC, false>(a, tiles_x, tiles_y);
}
// per-frame backgrounds: scalar stores only (any alignment), one instantiation per dtype pair and window size
template <typename RawT, typename OutT, int KS, int TH>
__global__ void __launch_bounds__(K1_THREADS) k1_generic_bg_kernel(K1Args a, int tiles_x, int tiles_y) {
    k1_generic_body<RawT, OutT, KS, TH, false, true>(a, tiles_x, tiles_y);
}
// per-frame exposure times of the line model (K1Args::exposures)
template <typename RawT, typename OutT, int KS, int TH, bool VEC>
__global__ void __launch_bounds__(K1_THREADS) k1_generic_tt_kernel(K1Args a, int tiles_x, int tiles_y) {
    k1_generic_body<RawT, OutT, KS, TH, VEC, false, true>(a, tiles_x, tiles_y);
}

// ------------------------------------------------------------------------------------------
// TMA variant
// ------------------------------------------------------------------------------------------
template <typename RawT, int KS, int TH, int NSTAGE>
struct K1TmaSmem {
    static constexpr int HALO = KS / 2;
    static constexpr int LH = TH + 2 * HALO;
    static constexpr size_t raw_bytes = (size_t)LH * RawBox<RawT>::BOXW * sizeof(RawT);
    static constexpr size_t map_bytes = (size_t)LH * K1_BOXW * sizeof(float);
    static constexpr size_t align128(size_t v) { return (v + 127) & ~(size_t)127; }
    static constexpr size_t stage_bytes = align128(raw_bytes) + 2 * align128(map_bytes);
    static constexpr size_t xs_off = NSTAGE * stage_bytes;
    static constexpr size_t bar_off = xs_off + align128(map_bytes);
    static constexpr size_t total = bar_off + 128;
};

// four consecutive raw samples starting at staged column 4*grp of the float32 box
template <typename RawT> __device__ __forceinline__ void load_raw4(const RawT* row, int grp, double v[4]);
template <> __device__ __forceinline__ void load_raw4<uint16_t>(const uint16_t* row, int grp, double v[4]) {
    const uint2 q = *reinterpret_cast<const uint2*>(row + (RawBox<uint16_t>::XOFF - K1_XOFF) + 4 * grp);
    v[0] = (double)(int)(q.x & 0xffffu); v[1] = (double)(int)(q.x >> 16);
    v[2] = (double)(int)(q.y & 0xffffu); v[3] = (double)(int)(q.y >> 16);
}
template <> __device__ __forceinline__ void load_raw4<uint8_t>(const uint8_t* row, int grp, double v[4]) {
    const uint32_t q = *reinterpret_cast<const uint32_t*>(row + (RawBox<uint8_t>::XOFF - K1_XOFF) + 4 * grp);
    v[0] = (double)(int)(q & 0xffu); v[1] = (double)(int)((q >> 8) & 0xffu);
    v[2] = (double)(int)((q >> 16) & 0xffu); v[3] = (double)(int)(q >> 24);
}
template <> __device__ __forceinline__ void load_raw4<float>(const float* row, int grp, double v[4]) {
    const float4 q = *reinterpret_cast<const float4*>(row + 4 * grp);
    v[0] = (double)q.x; v[1] = (double)q.y; v[2] = (double)q.z; v[3] = (double)q.w;
}

template <typename RawT, typename OutT, int KS, int TH, int NSTAGE>
__global__ void __launch_bounds__(K1_THREADS, KS == 5 ? 3 : 1)
k1_tma_kernel(const __grid_constant__ CUtensorMap tm_raw, const __grid_constant__ CUtensorMap tm_dark,
              const __grid_constant__ CUtensorMap tm_flat, K1Args a, int tiles_x, int tiles_y, int total_tiles) {
    using CT = float;
    using S = K1TmaSmem<RawT, KS, TH, NSTAGE>;
    constexpr int HALO = S::HALO;
    constexpr int LH = S::LH;
    constexpr int LW = K1_TW + 2 * HALO;
    extern __shared__ __align__(128) uint8_t smem[];
    CT* xs = (CT*)(smem + S::xs_off);
    uint64_t* full = (uint64_t*)(smem + S::bar_off);

    const bool has_dark = a.dark != nullptr, has_flat = a.flat != nullptr;
    const uint32_t tx_bytes = (uint32_t)(S::raw_bytes + (has_dark ? S::map_bytes : 0) + (has_flat ? S::map_bytes : 0));
    const PointwiseConst pw = a.pw;
    const PredicateConst pred = a.pred;

    auto issue = [&](int stage, int tile) {
        int t = tile;
        const int txi = t % tiles_x; t /= tiles_x;
        const int tyi = t % tiles_y;
        const int frame = t / tiles_y;
        const int y = tyi * TH - HALO;
        uint8_t* base = smem + (size_t)stage * S::stage_bytes;
        mbar_expect_tx(&full[stage], tx_bytes);
        tma_load_3d(base, &tm_raw, &full[stage], txi * K1_TW - RawBox<RawT>::XOFF, y, frame);
        if (has_dark) tma_load_2d(base + S::align128(S::raw_bytes), &tm_dark, &full[stage], txi * K1_TW - K1_XOFF, y);
        if (has_flat)
            tma_load_2d(base + S::align128(S::raw_bytes) + S::align128(S::map_bytes), &tm_flat, &full[stage],
                        txi * K1_TW - K1_XOFF, y);
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; ++s) mbar_init(&full[s], 1);
        mbar_init_fence();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; ++s) {
            int tile = blockIdx.x + s * gridDim.x;
            if (tile < total_tiles) issue(s, tile);
        }
    }

    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int stage = it % NSTAGE;
        const uint32_t parity = (it / NSTAGE) & 1;
        int t = tile;
        const int txi = t % tiles_x; t /= tiles_x;
        const int tyi = t % tiles_y;
        const int frame = t / tiles_y;
        const int tx0 = txi * K1_TW, ty0 = tyi * TH;

        mbar_wait(&full[stage], parity);
        const uint8_t* base = smem + (size_t)stage * S::stage_bytes;
        const RawT* sraw = (const RawT*)base;
        const float* sdark = (const float*)(base + S::align128(S::raw_bytes));
        const float* sflat = (const float*)(base + S::align128(S::raw_bytes) + S::align128(S::map_bytes));

        // phase A: pointwise value of every staged pixel, four columns per step
#pragma unroll 1
        for (int item = threadIdx.x; item < LH * K1_GROUPS; item += K1_THREADS) {
            const int ly = item / K1_GROUPS, grp = item - ly * K1_GROUPS;
            const int o = ly * K1_BOXW + 4 * grp;
            double v[4];
            load_raw4<RawT>(sraw + ly * RawBox<RawT>::BOXW, grp, v);
            float4 d = make_float4(0.f, 0.f, 0.f, 0.f), f = d;
            if (has_dark) d = *reinterpret_cast<const float4*>(sdark + o);
            if (has_flat) f = *reinterpret_cast<const float4*>(sflat + o);
            float4 x;
            x.x = pointwise<CT>(pw, v[0], d.x, 0.0f, f.x);
            x.y = pointwise<CT>(pw, v[1], d.y, 0.0f, f.y);
            x.z = pointwise<CT>(pw, v[2], d.z, 0.0f, f.z);
            x.w = pointwise<CT>(pw, v[3], d.w, 0.0f, f.w);
            *reinterpret_cast<float4*>(xs + o) = x;
        }
        __syncthreads();          // xs complete, stage fully consumed
        if (threadIdx.x == 0) {
            const int nxt = tile + NSTAGE * gridDim.x;
            if (nxt < total_tiles) issue(stage, nxt);
        }
        // scipy 'reflect' at the frame border: TMA zero-filled the out-of-frame part of the halo
        const bool border = (ty0 - HALO < 0) | (ty0 + TH + HALO > a.H) | (tx0 - HALO < 0) | (tx0 + K1_TW + HALO > a.W);
        if (border) {
            for (int idx = threadIdx.x; idx < LH * LW; idx += K1_THREADS) {
                const int ly = idx / LW, lx = idx - ly * LW;
                const int gy = ty0 - HALO + ly, gx = tx0 - HALO + lx;
                if ((unsigned)gy >= (unsigned)a.H || (unsigned)gx >= (unsigned)a.W) {
                    const int sy = reflect_index(gy, a.H) - (ty0 - HALO);
                    const int sx = reflect_index(gx, a.W) - (tx0 - HALO);
                    if ((unsigned)sy < (unsigned)LH && (unsigned)sx < (unsigned)LW)
                        xs[ly * K1_BOXW + (K1_XOFF - HALO) + lx] = xs[sy * K1_BOXW + (K1_XOFF - HALO) + sx];
                }
            }
            __syncthreads();
        }
        median_phase<CT, OutT, KS, TH, true>(xs, a, pred, frame, tx0, ty0);
        __syncthreads();          // xs is rewritten by the next tile's phase A
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
bool k1_tma_eligible(const K1Args& a, int raw_dtype, int out_dtype) {
    if (a.ksize != 3 && a.ksize != 5) return false;
    if (raw_dtype != DT_U8 && raw_dtype != DT_U16 && raw_dtype != DT_F32) return false;
    if (out_dtype != DT_F32 && out_dtype != DT_U16 && out_dtype != DT_U8) return false;
    if (a.ksize == 5 && out_dtype != DT_F32 && dtype_size(out_dtype) != dtype_size(raw_dtype)) return false;
    if (a.pw.flags & FLAG_DARK_LINEAR) return false;
    if (a.raw_swap || a.raw_gap) return false;
    if (a.bg) return false;                              // per-frame backgrounds: the streaming pipeline or the generic tiles
    const size_t esz = dtype_size(raw_dtype);
    if (((size_t)a.W * esz) % 16 || ((size_t)a.W * 4) % 16) return false;
    if (((size_t)a.H * a.W * esz) % 16) return false;
    if (((uintptr_t)a.raw) % 16 || ((uintptr_t)a.out) % 16) return false;
    if (a.mask && ((uintptr_t)a.mask) % 2) return false;
    if (a.dark && ((uintptr_t)a.dark) % 16) return false;
    if (a.flat && ((uintptr_t)a.flat) % 16) return false;
    return tensor_map_encoder() != nullptr;
}

template <typename RawT, typename OutT, int KS, int TH, int NSTAGE>
static cudaError_t launch_tma_t(const K1Args& a, CUtensorMapDataType rdt, int sm_count, cudaStream_t st) {
    using S = K1TmaSmem<RawT, KS, TH, NSTAGE>;
    CUtensorMap tr, td, tf;
    const int boxh = S::LH;
    if (!make_tensor_map(&tr, rdt, sizeof(RawT), a.raw, a.W, a.H, a.n_frames, RawBox<RawT>::BOXW, boxh)) return cudaErrorInvalidValue;
    // dark / flat maps: encode the raw pointer as a placeholder when absent (never dereferenced)
    if (!make_tensor_map(&td, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.dark ? (const void*)a.dark : a.raw, a.W, a.H, 0, K1_BOXW, boxh) && a.dark)
        return cudaErrorInvalidValue;
    if (!make_tensor_map(&tf, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.flat ? (const void*)a.flat : a.raw, a.W, a.H, 0, K1_BOXW, boxh) && a.flat)
        return cudaErrorInvalidValue;
    auto kern = k1_tma_kernel<RawT, OutT, KS, TH, NSTAGE>;
    cudaError_t e = cudaSuccess;
    const int per_sm = blocks_per_sm_cached((const void*)kern, K1_THREADS, S::total, &e);     // per (device, kernel)
    if (e != cudaSuccess) return e;
    const int tiles_x = (a.W + K1_TW - 1) / K1_TW, tiles_y = (a.H + TH - 1) / TH;
    const long long total = (long long)tiles_x * tiles_y * a.n_frames;
    long long grid = (long long)sm_count * per_sm;
    if (grid > total) grid = total;
    kern<<<(unsigned)grid, K1_THREADS, S::total, st>>>(tr, td, tf, a, tiles_x, tiles_y, (int)total);
    return cudaGetLastError();
}

template <typename RawT, typename OutT, int KS, int TH>
static cudaError_t launch_generic_t(const K1Args& a, cudaStream_t st) {
    const int tiles_x = (a.W + K1_TW - 1) / K1_TW, tiles_y = (a.H + TH - 1) / TH;
    const long long total = (long long)tiles_x * tiles_y * a.n_frames;
    if constexpr (sizeof(RawT) <= 4) {
        if (a.bg) {
            k1_generic_bg_kernel<RawT, OutT, KS, TH><<<(unsigned)total, K1_THREADS, 0, st>>>(a, tiles_x, tiles_y);
            return cudaGetLastError();
        }
    }
    const bool vec = (a.W % 2 == 0) && ((uintptr_t)a.out % (2 * sizeof(OutT)) == 0) && (!a.mask || (uintptr_t)a.mask % 2 == 0);
    if (a.exposures) {
        if (vec) k1_generic_tt_kernel<RawT, OutT, KS, TH, true><<<(unsigned)total, K1_THREADS, 0, st>>>(a, tiles_x, tiles_y);
        else k1_generic_tt_kernel<RawT, OutT, KS, TH, false><<<(unsigned)total, K1_THREADS, 0, st>>>(a, tiles_x, tiles_y);
        return cudaGetLastError();
    }
    if (vec) k1_generic_kernel<RawT, OutT, KS, TH, true><<<(unsigned)total, K1_THREADS, 0, st>>>(a, tiles_x, tiles_y);
    else k1_generic_kernel<RawT, OutT, KS, TH, false><<<(unsigned)total, K1_THREADS, 0, st>>>(a, tiles_x, tiles_y);
    return cudaGetLastError();
}

template <typename RawT, typename OutT>
static cudaError_t launch_pointwise_t(const K1Args& a, int sm_count, cudaStream_t st) {
    const size_t npx = (size_t)a.H * a.W;
    size_t bx = (npx + 255) / 256;
    const size_t cap = (size_t)sm_count * 16;
    if (bx > cap) bx = cap;
    for (int f0 = 0; f0 < a.n_frames; f0 += 65535) {
        K1Args b = a;
        const int nf = a.n_frames - f0 < 65535 ? a.n_frames - f0 : 65535;
        b.raw = (const char*)a.raw + (size_t)f0 * (npx * sizeof(RawT) + (size_t)a.raw_gap);
        b.out = (char*)a.out + (size_t)f0 * npx * sizeof(OutT);
        if constexpr (sizeof(RawT) <= 4) {
            if (a.bg) {
                b.bg = (const char*)a.bg + (size_t)f0 * npx * dtype_size(a.bg_dtype);
                k1_pointwise_bg_kernel<RawT, OutT><<<dim3((unsigned)bx, (unsigned)nf), 256, 0, st>>>(b);
                continue;
            }
        }
        if (a.exposures) {
            b.exposures = a.exposures + f0;
            k1_pointwise_tt_kernel<RawT, OutT><<<dim3((unsigned)bx, (unsigned)nf), 256, 0, st>>>(b);
            continue;
        }
        k1_pointwise_kernel<RawT, OutT><<<dim3((unsigned)bx, (unsigned)nf), 256, 0, st>>>(b);
    }
    return cudaGetLastError();
}

template <typename RawT, typename OutT>
static cudaError_t dispatch_ks(const K1Args& a, bool tma, CUtensorMapDataType rdt, int sm_count, cudaStream_t st) {
    if (a.ksize == 0) return launch_pointwise_t<RawT, OutT>(a, sm_count, st);
    if (a.ksize == 3) {
        if constexpr (sizeof(RawT) <= 4 && sizeof(OutT) <= 4)
            if (tma) {
                if constexpr (sizeof(RawT) <= 2) return launch_tma_t<RawT, OutT, 3, 32, 2>(a, rdt, sm_count, st);
                else return launch_tma_t<RawT, OutT, 3, 16, 2>(a, rdt, sm_count, st);
            }
        return launch_generic_t<RawT, OutT, 3, 32>(a, st);
    }
    if (a.ksize == 5) {
        // integer output of another width than the raw frames (the chain's quantised output) is not built for the 5x5
        // TMA tiles: those instantiations spill; they run the generic tiles (k1_tma_eligible says so)
        if constexpr (sizeof(RawT) <= 4 && sizeof(OutT) <= 4 && (sizeof(OutT) == 4 || sizeof(OutT) == sizeof(RawT)))
            if (tma) {
                return launch_tma_t<RawT, OutT, 5, 16, 2>(a, rdt, sm_count, st);      // 5x5 is register-heavy: small tiles, 3 CTAs / SM
            }
        return launch_generic_t<RawT, OutT, 5, 32>(a, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_k1(const K1Args& a, int raw_dtype, int out_dtype, int variant, int sm_count, int seg_rows,
                      cudaStream_t st, int* launches) {
    if (a.n_frames <= 0 || a.H <= 0 || a.W <= 0) return cudaSuccess;
    const bool stream_ok = (variant == 0 || variant == 3) && k1_stream_eligible(a, raw_dtype, out_dtype);
    const bool stream5_ok = (variant == 0 || variant == 3) && k1_stream5_eligible(a, raw_dtype, out_dtype);
    if (variant == 3 && !stream_ok && !stream5_ok) return cudaErrorNotSupported;
    if (stream_ok) {
        if (launches) ++*launches;
        return launch_k1_stream(a, raw_dtype, out_dtype, sm_count, seg_rows, st);
    }
    if (stream5_ok) {
        if (launches) ++*launches;
        return launch_k1_stream5(a, raw_dtype, out_dtype, sm_count, seg_rows, st);
    }
    bool tma = variant != 1 && k1_tma_eligible(a, raw_dtype, out_dtype);
    if (variant == 2 && !tma) return cudaErrorNotSupported;
    if (launches) ++*launches;
    switch (raw_dtype) {
        case DT_U8:
            if (out_dtype == DT_F32) return dispatch_ks<uint8_t, float>(a, tma, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, st);
            if (out_dtype == DT_U8) return dispatch_ks<uint8_t, uint8_t>(a, tma, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, st);
            if (out_dtype == DT_U16) return dispatch_ks<uint8_t, uint16_t>(a, tma, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, st);
            if (out_dtype == DT_F64) return dispatch_ks<uint8_t, double>(a, false, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, st);
            break;
        case DT_U16:
            if (out_dtype == DT_F32) return dispatch_ks<uint16_t, float>(a, tma, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, st);
            if (out_dtype == DT_U16) return dispatch_ks<uint16_t, uint16_t>(a, tma, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, st);
            if (out_dtype == DT_U8) return dispatch_ks<uint16_t, uint8_t>(a, tma, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, st);
            if (out_dtype == DT_F64) return dispatch_ks<uint16_t, double>(a, false, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, st);
            break;
        case DT_F32:
            if (out_dtype == DT_F32) return dispatch_ks<float, float>(a, tma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, st);
            if (out_dtype == DT_U16) return dispatch_ks<float, uint16_t>(a, tma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, st);
            if (out_dtype == DT_U8) return dispatch_ks<float, uint8_t>(a, tma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, st);
            if (out_dtype == DT_F64) return dispatch_ks<float, double>(a, false, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, st);
            break;
        case DT_F64:
            if (out_dtype == DT_F64) return dispatch_ks<double, double>(a, false, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, sm_count, st);
            break;
    }
    if (launches) --*launches;
    return cudaErrorInvalidValue;
}

}  // namespace imgcorr
