// k3_warp.cu — K3: perspective warp (SURVEY §8 row f3), sm_100a.
//
// Replaces cv2.warpPerspective in PerspectiveCorrection.correct (INTER_LANCZOS4,
// camera/PerspectiveCorrection.py:401-405) and .uncorrect (INTER_CUBIC | WARP_INVERSE_MAP, :374-378), and the
// tilt-factor division in front of it (:394-400).  Arithmetic: imgcorr_warp.cuh (bit-exact with OpenCV).
//
// One thread per output pixel x all frames of the launch: the float64 homography (a division and ~14 DP
// operations) and the 2 x N coefficient fetches are done once, then every frame gathers its N x N window.  N x N
// products + sums per pixel with OpenCV's rounding order cannot be separated into two 1-D passes, so the kernel
// is bound by load/FP32 issue (64 loads + 192 FP32 operations per Lanczos4 pixel), not by HBM; consecutive
// lanes read consecutive source columns, so the gathers are coalesced L1 hits for any sane homography.
#include <algorithm>
#include <type_traits>
#include "imgcorr_kernels.cuh"
#include "imgcorr_tma.cuh"
#include "imgcorr_warp.cuh"

namespace imgcorr {

namespace {

template <typename T> struct OutCast;
template <> struct OutCast<float> { static __device__ __forceinline__ float cast(float v) { return v; } };
template <> struct OutCast<double> { static __device__ __forceinline__ double cast(double v) { return v; } };
template <> struct OutCast<uint16_t> { static __device__ __forceinline__ uint16_t cast(float v) { return sat_u16(v); } };
// DT != T: a float32 source warped in float32 and stored through the quantiser (the batch chain's integer output)
template <typename T, typename DT, typename AT> __device__ __forceinline__ DT k3_out(AT v, const OutScale& q) {
    if constexpr (std::is_same<T, DT>::value) return OutCast<T>::cast(v);
    else return quantise<DT>(v, q);
}

template <typename T> __device__ __forceinline__ T ldg(const T* p) { return __ldg(p); }

template <typename T, typename AT, int N>
__device__ __noinline__ AT warp_border_ool(const T* S0, int H, int W, int sx, int sy, const float* wy, const float* wx, AT cv) {
    return warp_sum_border<T, AT, N>(S0, H, W, sx, sy, wy, wx, cv);
}

template <typename T> struct AccOf { typedef float type; };
template <> struct AccOf<double> { typedef double type; };

constexpr int K3_BX = 32, K3_BY = 8;

// PF: every frame has its own matrix (a.wcs), so the coordinate, the coefficients and the class of the pixel (interior /
// outside / border) are found per frame instead of once per launch
template <typename T, typename AT, int N, typename DT = T, bool PF = false>
__global__ void __launch_bounds__(K3_BX* K3_BY) k3_warp_kernel(const K3Args a) {
    __shared__ float tab[N][32];   // transposed: tab[tap][phase] -> lanes with different phases hit different banks
    for (int i = threadIdx.y * K3_BX + threadIdx.x; i < N * 32; i += K3_BX * K3_BY) tab[i % N][i / N] = a.tab[i];
    __syncthreads();
    const int x = blockIdx.x * K3_BX + threadIdx.x, y = blockIdx.y * K3_BY + threadIdx.y;
    if (x >= a.dw || y >= a.dh) return;
    if constexpr (PF) {
        constexpr int OFF = N / 2 - 1;
        const int w1 = max(a.W - (N - 1), 0), h1 = max(a.H - (N - 1), 0);
        const AT cv = (AT)a.border;
        const size_t spx = (size_t)a.H * a.W, dpx = (size_t)a.dh * a.dw;
        const T* S = (const T*)a.src;
        DT* D = (DT*)a.dst + (size_t)y * a.dw + x;
        for (int f = 0; f < a.n_frames; ++f, S += spx, D += dpx) {
            const FixedCoord c = warp_coord(a.wcs[f], x, y);
            const int sx = c.ix - OFF, sy = c.iy - OFF;
            float wy[N], wx[N];
#pragma unroll
            for (int i = 0; i < N; ++i) {
                wy[i] = tab[i][c.fy];
                wx[i] = tab[i][c.fx];
            }
            AT v;
            if ((unsigned)sx < (unsigned)w1 && (unsigned)sy < (unsigned)h1) {
                const T* P = S + ((long long)sy * a.W + sx);
                v = (AT)0;
#pragma unroll
                for (int r = 0; r < N; ++r) {
                    AT acc = wmul((AT)ldg(P), (AT)fmul(wy[r], wx[0]));
#pragma unroll
                    for (int k = 1; k < N; ++k) acc = wadd(acc, wmul((AT)ldg(P + k), (AT)fmul(wy[r], wx[k])));
                    v = wadd(v, acc);
                    P += a.W;
                }
            } else if (sx >= a.W || sx + N <= 0 || sy >= a.H || sy + N <= 0) {
                v = cv;
            } else {
                v = warp_border_ool<T, AT, N>(S, a.H, a.W, sx, sy, wy, wx, cv);
            }
            *D = k3_out<T, DT>(v, a.q);
        }
        return;
    }
    const FixedCoord c = warp_coord(a.wc, x, y);
    constexpr int OFF = N / 2 - 1;
    const int sx = c.ix - OFF, sy = c.iy - OFF;
    float wy[N], wx[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        wy[i] = tab[i][c.fy];
        wx[i] = tab[i][c.fx];
    }
    const int w1 = max(a.W - (N - 1), 0), h1 = max(a.H - (N - 1), 0);
    const bool interior = (unsigned)sx < (unsigned)w1 && (unsigned)sy < (unsigned)h1;
    const bool outside = sx >= a.W || sx + N <= 0 || sy >= a.H || sy + N <= 0;
    const AT cv = (AT)a.border;
    const size_t spx = (size_t)a.H * a.W, dpx = (size_t)a.dh * a.dw;
    const T* S = (const T*)a.src;
    DT* D = (DT*)a.dst + (size_t)y * a.dw + x;
    const long long o0 = (long long)sy * a.W + sx;
    for (int f = 0; f < a.n_frames; ++f, S += spx, D += dpx) {
        AT v;
        if (interior) {
            const T* P = S + o0;
            v = (AT)0;
#pragma unroll
            for (int r = 0; r < N; ++r) {
                T t[N];
#pragma unroll
                for (int k = 0; k < N; ++k) t[k] = ldg(P + k);
                AT acc = wmul((AT)t[0], (AT)fmul(wy[r], wx[0]));
#pragma unroll
                for (int k = 1; k < N; ++k) acc = wadd(acc, wmul((AT)t[k], (AT)fmul(wy[r], wx[k])));
                v = wadd(v, acc);
                P += a.W;
            }
        } else if (outside) {
            v = cv;
        } else {
            v = warp_border_ool<T, AT, N>(S, a.H, a.W, sx, sy, wy, wx, cv);
        }
        *D = k3_out<T, DT>(v, a.q);
    }
}


// ------------------------------------------------------------------------------------------------------------
// Tiled variant (uint16 / float32 sources whose rows are 16-byte multiples): the gathers above are bound by L1
// wavefronts (a warp's 32 consecutive, unaligned floats straddle two 128-byte lines, x 64 taps).  Here the source
// window of a 32x8 output tile is staged in shared memory by ONE TMA box per frame — 32 consecutive words are a
// single conflict-free wavefront at any alignment — and the frames of a launch are pipelined NBUF deep.
//   * box origin = (min sx rounded down to 16 bytes — TMA's rule —, min sy) over the tile's interior pixels, found
//     with REDUX + shared atomics; a tile whose window does not fit the fixed box (strong zoom-out / rotation) falls
//     back to the global gathers, so any homography stays correct;
//   * pixels whose window leaves the frame use OpenCV's border arithmetic from global memory, out of line.
#ifndef K3T_MINB_V
#define K3T_MINB_V 2
#endif
constexpr int K3T_TW = 32, K3T_TH = 8, K3T_THREADS = 256, K3T_BH = 24, K3T_NBUF = 4;
// The float32 window the taps are read from has a row pitch of 64 words: lanes of a warp that straddle two source rows
// (any tilt) then still hit 32 different banks.  uint16 boxes (56 columns: 16-byte origin granularity = 8 pixels) are
// converted to float32 once per staged element instead of once per tap (64 I2F per pixel would saturate the XU pipe).
constexpr int K3T_PITCH = 64;
template <typename T> struct K3Box;
template <> struct K3Box<float> { static constexpr int BW = 64, GRAN = 4; static constexpr CUtensorMapDataType DT = CU_TENSOR_MAP_DATA_TYPE_FLOAT32; };
template <> struct K3Box<uint16_t> { static constexpr int BW = 56, GRAN = 8; static constexpr CUtensorMapDataType DT = CU_TENSOR_MAP_DATA_TYPE_UINT16; };

template <typename T> constexpr int k3t_box_bytes() { return K3Box<T>::BW * K3T_BH * (int)sizeof(T); }
constexpr int K3T_CVT_BYTES = K3T_PITCH * K3T_BH * 4;
template <typename T> constexpr int k3t_smem() { return K3T_NBUF * k3t_box_bytes<T>() + (sizeof(T) == 4 ? 0 : 2 * K3T_CVT_BYTES) + 128; }

template <typename T, int N, typename DT = T>
__global__ void __launch_bounds__(K3T_THREADS, K3T_MINB_V) k3_tiled_kernel(const __grid_constant__ CUtensorMap tm_src, const K3Args a) {
    constexpr int BW = K3Box<T>::BW, BOX_BYTES = k3t_box_bytes<T>();
    constexpr bool CVT = sizeof(T) != 4;
    constexpr int RING = K3T_NBUF * BOX_BYTES + (CVT ? 2 * K3T_CVT_BYTES : 0);
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ float tab[N][32];
    uint64_t* full = (uint64_t*)(smem + RING);
    int* red = (int*)(smem + RING + 64);                       // min sx, max sx + N - 1, min sy, max sy + N - 1
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int b = 0; b < K3T_NBUF; ++b) mbar_init(&full[b], 1);
        red[0] = 0x7fffffff; red[1] = -1; red[2] = 0x7fffffff; red[3] = -1;
        mbar_init_fence();
    }
    for (int i = tid; i < N * 32; i += K3T_THREADS) tab[i % N][i / N] = a.tab[i];
    const int x = blockIdx.x * K3T_TW + (tid % K3T_TW), y = blockIdx.y * K3T_TH + (tid / K3T_TW);
    const bool live = x < a.dw && y < a.dh;
    const FixedCoord c = warp_coord(a.wc, live ? x : 0, live ? y : 0);
    constexpr int OFF = N / 2 - 1;
    const int sx = c.ix - OFF, sy = c.iy - OFF;
    const int H = a.H, W = a.W, nf = a.n_frames;
    const bool interior = live && (unsigned)sx < (unsigned)max(W - (N - 1), 0) && (unsigned)sy < (unsigned)max(H - (N - 1), 0);
    const bool outside = sx >= W || sx + N <= 0 || sy >= H || sy + N <= 0;
    int mnx = interior ? sx : 0x7fffffff, mxx = interior ? sx + N - 1 : -1;
    int mny = interior ? sy : 0x7fffffff, mxy = interior ? sy + N - 1 : -1;
    __syncthreads();                                   // red[], the barriers and the table are ready
    mnx = __reduce_min_sync(0xffffffffu, mnx); mxx = __reduce_max_sync(0xffffffffu, mxx);
    mny = __reduce_min_sync(0xffffffffu, mny); mxy = __reduce_max_sync(0xffffffffu, mxy);
    if ((tid & 31) == 0) { atomicMin(&red[0], mnx); atomicMax(&red[1], mxx); atomicMin(&red[2], mny); atomicMax(&red[3], mxy); }
    float wy[N], wx[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        wy[i] = tab[i][c.fy];
        wx[i] = tab[i][c.fx];
    }
    __syncthreads();
    const int bx = red[0] & ~(K3Box<T>::GRAN - 1), by = red[2];
    const bool any = red[1] >= 0;
    const bool fits = any && (red[1] + 1 - bx) <= BW && (red[3] + 1 - by) <= K3T_BH;

    typedef typename AccOf<T>::type AT;
    const size_t spx = (size_t)H * W, dpx = (size_t)a.dh * a.dw;
    DT* D = (DT*)a.dst + ((size_t)(live ? y : 0) * a.dw + (live ? x : 0));
    if (fits) {
        const int so = interior ? (sy - by) * K3T_PITCH + (sx - bx) : 0;
        auto issue = [&](int f) {
            uint64_t* bar = &full[f % K3T_NBUF];
            mbar_expect_tx(bar, BOX_BYTES);
            tma_load_3d(smem + (f % K3T_NBUF) * BOX_BYTES, &tm_src, bar, bx, by, f);
        };
        if (tid == 0) for (int f = 0; f < K3T_NBUF && f < nf; ++f) issue(f);
#pragma unroll 1
        for (int f = 0; f < nf; ++f) {
            mbar_wait(&full[f % K3T_NBUF], (f / K3T_NBUF) & 1);
            const float* P;
            if (CVT) {
                // widen the landed box into one of two float32 windows; the next frame widens into the other one, so one
                // barrier per frame orders both the reuse of the staging buffer and the reads of the window
                const T* raw = (const T*)(smem + (f % K3T_NBUF) * BOX_BYTES);
                float* win = (float*)(smem + K3T_NBUF * BOX_BYTES + (f & 1) * K3T_CVT_BYTES);
                for (int i = tid; i < BW * K3T_BH / 2; i += K3T_THREADS) {
                    const uint32_t two = ((const uint32_t*)raw)[i];
                    const int e = 2 * i, rr = e / BW, cc = e % BW;
                    *(float2*)(win + rr * K3T_PITCH + cc) = make_float2((float)(two & 0xffffu), (float)(two >> 16));
                }
                __syncthreads();
                if (tid == 0 && f + K3T_NBUF < nf) issue(f + K3T_NBUF);
                P = win + so;
            } else {
                P = (const float*)(smem + (f % K3T_NBUF) * BOX_BYTES) + so;
            }
            float v = 0.0f;
#pragma unroll
            for (int r = 0; r < N; ++r) {
                float acc = fmul(P[r * K3T_PITCH], fmul(wy[r], wx[0]));
#pragma unroll
                for (int k = 1; k < N; ++k) acc = fadd(acc, fmul(P[r * K3T_PITCH + k], fmul(wy[r], wx[k])));
                v = fadd(v, acc);
            }
            if (interior) D[f * dpx] = k3_out<T, DT>(v, a.q);
            if (!CVT) {
                __syncthreads();                       // everyone is done with this buffer
                if (tid == 0 && f + K3T_NBUF < nf) issue(f + K3T_NBUF);
            }
        }
    } else if (interior) {
        const T* S = (const T*)a.src + ((long long)sy * W + sx);
        for (int f = 0; f < nf; ++f, S += spx) {
            AT v = (AT)0;
#pragma unroll
            for (int r = 0; r < N; ++r) {
                const T* P = S + (size_t)r * W;
                AT acc = wmul((AT)ldg(P), (AT)fmul(wy[r], wx[0]));
#pragma unroll
                for (int k = 1; k < N; ++k) acc = wadd(acc, wmul((AT)ldg(P + k), (AT)fmul(wy[r], wx[k])));
                v = wadd(v, acc);
            }
            D[f * dpx] = k3_out<T, DT>(v, a.q);
        }
    }
    if (live && !interior) {
        const AT cv = (AT)a.border;
        const T* S = (const T*)a.src;
        for (int f = 0; f < nf; ++f, S += spx)
            D[f * dpx] = k3_out<T, DT>(outside ? cv : warp_border_ool<T, AT, N>(S, H, W, sx, sy, wy, wx, cv), a.q);
    }
}

template <typename T>
bool k3_tiled_eligible(const K3Args& a) {
    if (((size_t)a.W * sizeof(T)) % 16 || ((uintptr_t)a.src) % 16) return false;
    return tensor_map_encoder() != nullptr;
}

template <typename T, typename DT = T>
cudaError_t launch_tiled(const K3Args& a, int interp, cudaStream_t st) {
    CUtensorMap tm;
    if (!make_tensor_map(&tm, K3Box<T>::DT, sizeof(T), a.src, a.W, a.H, a.n_frames, K3Box<T>::BW, K3T_BH)) return cudaErrorInvalidValue;
    dim3 grid((a.dw + K3T_TW - 1) / K3T_TW, (a.dh + K3T_TH - 1) / K3T_TH);
    if (interp == WARP_LANCZOS4)
        k3_tiled_kernel<T, 8, DT><<<grid, K3T_THREADS, k3t_smem<T>(), st>>>(tm, a);
    else if constexpr (std::is_same<T, DT>::value)           // the chain warps with Lanczos4 only
        k3_tiled_kernel<T, 4><<<grid, K3T_THREADS, k3t_smem<T>(), st>>>(tm, a);
    else
        return cudaErrorNotSupported;
    return cudaGetLastError();
}

// uint8 images (OpenCV's int16 fixed-point weights): one thread per output pixel, the 2-D weight entry of the pixel's
// phase pair is fetched once from the (L2-resident) table and kept packed in registers for all frames of the launch.
template <int N>
__global__ void __launch_bounds__(K3_BX* K3_BY) k3_warp_u8_kernel(const K3Args a) {
    const int x = blockIdx.x * K3_BX + threadIdx.x, y = blockIdx.y * K3_BY + threadIdx.y;
    if (x >= a.dw || y >= a.dh) return;
    const FixedCoord c = warp_coord(a.wc, x, y);
    __align__(16) int16_t w[N * N];
    const int4* wp = reinterpret_cast<const int4*>(a.itab + ((size_t)c.fy * 32 + c.fx) * N * N);
#pragma unroll
    for (int i = 0; i < N * N / 8; ++i) reinterpret_cast<int4*>(w)[i] = __ldg(wp + i);
    const int cv = (int)a.border;
    const size_t spx = (size_t)a.H * a.W, dpx = (size_t)a.dh * a.dw;
    const uint8_t* S = (const uint8_t*)a.src;
    uint8_t* D = (uint8_t*)a.dst + (size_t)y * a.dw + x;
    for (int f = 0; f < a.n_frames; ++f, S += spx, D += dpx) *D = warp_pixel_u8<N>(S, a.H, a.W, c, w, cv);
}

// image / tiltFactor in float64 (PerspectiveCorrection.py:394-400: np.asfarray(img) / tf)
template <typename T>
__global__ void __launch_bounds__(256) k3_divide_kernel(const T* __restrict__ src, const double* __restrict__ div, double* __restrict__ dst,
                                                         size_t npx, int n_frames) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (size_t)gridDim.x * blockDim.x) {
        const double d = div[i];
        for (int f = 0; f < n_frames; ++f) dst[f * npx + i] = ddiv((double)src[f * npx + i], d);
    }
}

// the same division in place on float64 frames (src == dst): the chain divides its warp source this way.  No pointer
// is __restrict__, and each element is read and then written by the thread that owns it.
__global__ void __launch_bounds__(256) k3_divide_inplace_kernel(double* data, const double* __restrict__ div, size_t npx,
                                                                 int n_frames) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (size_t)gridDim.x * blockDim.x) {
        const double d = div[i];
        for (int f = 0; f < n_frames; ++f) data[f * npx + i] = ddiv(data[f * npx + i], d);
    }
}

template <typename T, typename AT, typename DT = T>
cudaError_t launch_typed(const K3Args& a, int interp, cudaStream_t st) {
    dim3 block(K3_BX, K3_BY), grid((a.dw + K3_BX - 1) / K3_BX, (a.dh + K3_BY - 1) / K3_BY);
    if (interp == WARP_LANCZOS4)
        k3_warp_kernel<T, AT, 8, DT><<<grid, block, 0, st>>>(a);
    else if constexpr (std::is_same<T, DT>::value)
        k3_warp_kernel<T, AT, 4><<<grid, block, 0, st>>>(a);
    else
        return cudaErrorNotSupported;
    return cudaGetLastError();
}

// one matrix per frame (a.wcs), Lanczos4 through L1: float to float / U16 / U8, or double to double
template <typename T, typename DT>
cudaError_t launch_frames(const K3Args& a, cudaStream_t st) {
    dim3 block(K3_BX, K3_BY), grid((a.dw + K3_BX - 1) / K3_BX, (a.dh + K3_BY - 1) / K3_BY);
    k3_warp_kernel<T, T, 8, DT, true><<<grid, block, 0, st>>>(a);
    return cudaGetLastError();
}

}  // namespace

// variant: 0 auto, 1 gathers through L1, 2 shared-memory staged tiles (uint16 / float32, one matrix per launch; fails if
// not eligible)
cudaError_t launch_k3(const K3Args& a, int dtype, int interp, int variant, cudaStream_t st, int* launches) {
    if (a.n_frames <= 0 || a.dw <= 0 || a.dh <= 0) return cudaSuccess;
    if (interp != WARP_LANCZOS4 && interp != WARP_CUBIC) return cudaErrorInvalidValue;
    cudaError_t e;
    if (a.wcs) {
        // the chain's per-frame table: float32 frames to float32 / U16 / U8, float64 frames to float64.  Measured (4096x3000,
        // B200) it is faster through L1 than through staged tiles (tools/perframe_warp.py, DESIGN §4 "Chain, host pipeline,
        // batches"), so it has no tiled kernel
        if (variant == 2) return cudaErrorNotSupported;
        if (interp != WARP_LANCZOS4) return cudaErrorInvalidValue;
        if (dtype == DT_F64 && a.dst_dtype == DT_F64) e = launch_frames<double, double>(a, st);
        else if (dtype == DT_F32 && a.dst_dtype == DT_F32) e = launch_frames<float, float>(a, st);
        else if (dtype == DT_F32 && a.dst_dtype == DT_U16) e = launch_frames<float, uint16_t>(a, st);
        else if (dtype == DT_F32 && a.dst_dtype == DT_U8) e = launch_frames<float, uint8_t>(a, st);
        else return cudaErrorInvalidValue;
        if (launches) ++*launches;
        return e;
    }
    // measured (4096x3000, B200): the staged tiles win for Lanczos4 once a launch carries a few frames (float32 138 vs
    // 160 us/frame, uint16 174 vs 224); a single frame and the 4x4 bicubic window are faster straight through L1
    const bool wanted = variant == 2 || (variant == 0 && interp == WARP_LANCZOS4 && a.n_frames >= 4);
    if (variant == 2 && dtype == DT_U8) return cudaErrorNotSupported;
    const bool tiled = wanted && ((dtype == DT_U16 && k3_tiled_eligible<uint16_t>(a)) || (dtype == DT_F32 && k3_tiled_eligible<float>(a)));
    if (variant == 2 && !tiled) return cudaErrorNotSupported;
    if (a.dst_dtype != dtype) {
        // float32 source, integer destination: the float32 warp of the F32 call, stored through the quantiser
        if (dtype != DT_F32 || (a.dst_dtype != DT_U16 && a.dst_dtype != DT_U8)) return cudaErrorInvalidValue;
        if (a.dst_dtype == DT_U16) e = tiled ? launch_tiled<float, uint16_t>(a, interp, st) : launch_typed<float, float, uint16_t>(a, interp, st);
        else e = tiled ? launch_tiled<float, uint8_t>(a, interp, st) : launch_typed<float, float, uint8_t>(a, interp, st);
        if (launches) ++*launches;
        return e;
    }
    switch (dtype) {
        case DT_U8: {
            if (!a.itab) return cudaErrorInvalidValue;
            dim3 block(K3_BX, K3_BY), grid((a.dw + K3_BX - 1) / K3_BX, (a.dh + K3_BY - 1) / K3_BY);
            if (interp == WARP_LANCZOS4) k3_warp_u8_kernel<8><<<grid, block, 0, st>>>(a);
            else k3_warp_u8_kernel<4><<<grid, block, 0, st>>>(a);
            e = cudaGetLastError();
            break;
        }
        case DT_U16: e = tiled ? launch_tiled<uint16_t>(a, interp, st) : launch_typed<uint16_t, float>(a, interp, st); break;
        case DT_F32: e = tiled ? launch_tiled<float>(a, interp, st) : launch_typed<float, float>(a, interp, st); break;
        case DT_F64: e = launch_typed<double, double>(a, interp, st); break;
        default: return cudaErrorInvalidValue;
    }
    if (launches) ++*launches;
    return e;
}

cudaError_t launch_k3_divide(const void* src, int dtype, const double* div, double* dst, size_t npx, int n_frames, int sm_count,
                             cudaStream_t st, int* launches) {
    if (npx == 0 || n_frames <= 0) return cudaSuccess;
    const int grid = (int)std::min<size_t>((npx + 255) / 256, (size_t)sm_count * 8);
    if (src == dst && dtype == DT_F64) {
        k3_divide_inplace_kernel<<<grid, 256, 0, st>>>(dst, div, npx, n_frames);
        if (launches) ++*launches;
        return cudaGetLastError();
    }
    switch (dtype) {
        case DT_U8: k3_divide_kernel<<<grid, 256, 0, st>>>((const uint8_t*)src, div, dst, npx, n_frames); break;
        case DT_U16: k3_divide_kernel<<<grid, 256, 0, st>>>((const uint16_t*)src, div, dst, npx, n_frames); break;
        case DT_F32: k3_divide_kernel<<<grid, 256, 0, st>>>((const float*)src, div, dst, npx, n_frames); break;
        case DT_F64: k3_divide_kernel<<<grid, 256, 0, st>>>((const double*)src, div, dst, npx, n_frames); break;
        default: return cudaErrorInvalidValue;
    }
    if (launches) ++*launches;
    return cudaGetLastError();
}

}  // namespace imgcorr
