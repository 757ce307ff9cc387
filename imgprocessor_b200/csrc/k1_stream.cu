// K1, streaming variant (3x3): the fused dark / flat / nan_to_num / median-threshold kernel as a
// warp-specialised TMA pipeline with the stencil window held in registers.
//
//   * work unit = (group of NF frames, 120-column strip, segment of rows).  A CTA is 4 consumer warps + 1 producer
//     warp and walks its units top to bottom in chunks of R rows.
//   * the producer warp (one elected lane) fills a shared-memory ring with cp.async.bulk.tensor boxes of
//     raw (one per frame of the group) / dark / flat rows (16-byte aligned, 16-byte multiple wide,
//     out-of-frame parts zero-filled by TMA), signalled through `full` mbarriers; consumers hand a
//     stage back through `empty` mbarriers.  There is no CTA-wide barrier in the steady state.
//   * each consumer lane owns one image column of its warp's 30-column slice (+1 halo lane on each
//     side; the halo / out-of-frame lanes read the mirrored column, which is scipy's 'reflect').
//     Per row it reads dark and flat once, turns the flat value into a float64 reciprocal once (MUFU seed + one Newton
//     step) and applies both to the raw sample of every frame of the group: float64 subtraction, reciprocal multiply,
//     residual correction (= the correctly rounded float64 quotient, imgcorr_core.cuh), one rounding to float32.  The
//     frame-independent half of the division is thereby shared by the NF frames (NF = 2 for batches).
//   * per frame: left / right neighbours with two warp shuffles, a 3-element sort of the horizontal triple, and — two
//     output rows at a time — the median of 9 from the sorted triples of four consecutive rows (the two middle rows'
//     contribution is computed once for both outputs); predicate + select + one coalesced store per row.
//   * vertical 'reflect' needs no halo rows: the first / last row's sorted triple is used twice.
//
// Same arithmetic as the tile kernels (imgcorr_core.cuh) — results are bit-identical.
#include <type_traits>
#include "imgcorr_kernels.cuh"
#include "imgcorr_tma.cuh"

namespace imgcorr {

constexpr int KS_CW = 4;                    // consumer warps per CTA
constexpr int KS_SW = 30;                   // output columns per consumer warp
constexpr int KS_TW = KS_CW * KS_SW;        // 120 output columns per strip
// Pipeline shape: rows per stage x stages x CTAs per SM the register allocation aims at x frames per work unit.
// Long straight-line chunks with many independent rows in flight per warp beat occupancy (round 1: 8 x 4 x 5 34.5 us per
// 4096x3000 frame, 32 x 2 x 2 30.6); with few frames per launch and for the integer-output instantiations the small shape
// wins, so both are built.  Batches of float32-output frames run two frames per unit (KsPair).
template <int R_, int NSTAGE_, int MINB_, int NF_> struct KsShape { static constexpr int R = R_, NSTAGE = NSTAGE_, MINB = MINB_, NF = NF_; };
#ifndef KS_NARROW_R
#define KS_NARROW_R 24
#define KS_NARROW_NSTAGE 3
#define KS_NARROW_MINB 2
#endif
typedef KsShape<KS_NARROW_R, KS_NARROW_NSTAGE, KS_NARROW_MINB, 1> KsNarrow;
#ifndef KS_WIDE_R
#define KS_WIDE_R 32
#define KS_WIDE_NSTAGE 2
#define KS_WIDE_MINB 3
#endif
typedef KsShape<KS_WIDE_R, KS_WIDE_NSTAGE, KS_WIDE_MINB, 1> KsWide;
#ifndef KS_PAIR_R
#define KS_PAIR_R 16
#define KS_PAIR_NSTAGE 3
#define KS_PAIR_MINB 3
#endif
typedef KsShape<KS_PAIR_R, KS_PAIR_NSTAGE, KS_PAIR_MINB, 2> KsPair;
// frame pairs with per-frame backgrounds: a background box per frame replaces the dark box.  Three stages of the pair
// shape would need 25.6 KB (uint16) / 40 KB (float32) each, just above what 3 (uint16) / 2 (float32) CTAs per SM can
// hold, so these shapes keep two stages.  Float32 frames fit 2 CTAs per SM (80 KB each) and get their registers:
// with the cap of 3 CTAs the checked arithmetic spills
#ifndef KS_PAIRBG_R
#define KS_PAIRBG_R 16
#define KS_PAIRBG_NSTAGE 2
#endif
typedef KsShape<KS_PAIRBG_R, KS_PAIRBG_NSTAGE, 3, 2> KsPairBg;         // uint16 frames, finite flat field
typedef KsShape<KS_PAIRBG_R, KS_PAIRBG_NSTAGE, 2, 2> KsPairBgF32;      // float32 frames
// the line model (KS_LIN): an offset box and an ascent box per stage in place of the dark box.  A 16-row uint16 pair stage
// is 33.3 KB (float32: 40 KB), a 24-row one-frame stage 42.4 KB (float32: 48 KB).  uint16 pairs take 3 stages x 2 CTAs per
// SM: at 2 stages x 3 CTAs the register cap makes the chain configurations spill (4 and 16 bytes)
#ifndef KS_PAIRLIN_NSTAGE
#define KS_PAIRLIN_NSTAGE 3
#define KS_PAIRLIN_MINB 2
#endif
typedef KsShape<16, KS_PAIRLIN_NSTAGE, KS_PAIRLIN_MINB, 2> KsPairLin;  // uint16 frames
typedef KsShape<16, 2, 2, 2> KsPairLinF32;                             // float32 frames
typedef KsShape<24, 2, 2, 1> KsNarrowLin;                              // one frame per unit
constexpr int KS_MAPW = 128;                // float32 box: tx0-4 .. tx0+123
constexpr int KS_MAPX = 4;
constexpr int KS_THREADS = (KS_CW + 1) * 32;

template <typename RawT, typename C, bool BG = false, bool LIN = false> struct StreamBox {
    static constexpr int XOFF = 16 / (int)sizeof(RawT);                        // u8 16, u16 8, f32 4
    static constexpr int GRAN = 16 / (int)sizeof(RawT);
    // the box starts at the 16-byte boundary at or left of tx0, minus XOFF: columns tx0-1 .. tx0+120 are inside
    static constexpr int BOXW = ((KS_TW + 2 * XOFF + GRAN - 1) / GRAN) * GRAN;  // u8 160, u16 136, f32 128
    static constexpr size_t raw_bytes = (size_t)C::R * BOXW * sizeof(RawT);     // multiples of 128
    static constexpr size_t map_bytes = (size_t)C::R * KS_MAPW * sizeof(float);
    // the dark box, a background box per frame, or the offset and ascent boxes of the line model
    static constexpr size_t dark_bytes = BG ? C::NF * raw_bytes : LIN ? 2 * map_bytes : map_bytes;
    static constexpr size_t stage_bytes = C::NF * raw_bytes + dark_bytes + map_bytes;    // raw[NF] | dark or bg[NF] | flat
    static_assert(raw_bytes % 128 == 0 && map_bytes % 128 == 0, "TMA destinations must be 128-byte aligned: rows per stage must be a multiple of 8");
    static constexpr size_t bar_off = C::NSTAGE * stage_bytes;
    static constexpr size_t total = bar_off + 2 * C::NSTAGE * sizeof(uint64_t) + 64;
};

template <typename T> struct StreamRaw;
template <> struct StreamRaw<uint8_t>  { static __device__ __forceinline__ void ld(uint8_t v, double& d, float& a)  { d = (double)(int)v; a = 0.0f; } };
template <> struct StreamRaw<uint16_t> { static __device__ __forceinline__ void ld(uint16_t v, double& d, float& a) { d = (double)(int)v; a = 0.0f; } };
template <> struct StreamRaw<float>    { static __device__ __forceinline__ void ld(float v, double& d, float& a)    { d = (double)v; a = fabsf(v); } };

template <typename OutT> __device__ __forceinline__ OutT ks_out(const K1Args& a, float v);
template <> __device__ __forceinline__ float    ks_out<float>(const K1Args&, float v)      { return v; }
template <> __device__ __forceinline__ uint16_t ks_out<uint16_t>(const K1Args& a, float v) { return quantise<uint16_t>(v, a.q); }
template <> __device__ __forceinline__ uint8_t  ks_out<uint8_t>(const K1Args& a, float v)  { return quantise<uint8_t>(v, a.q); }

// store with an L2 eviction-priority hint (float32 results of the straight-line chunks)
template <typename OutT> __device__ __forceinline__ void ks_store(OutT* p, OutT v, uint64_t) { *p = v; }
template <> __device__ __forceinline__ void ks_store<float>(float* p, float v, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(policy) : "memory");
}

__device__ __noinline__ bool ks_exact(float x, float b, double thr, int cond) {
    PredicateConst pc;
    pc.thr = thr; pc.cond = cond; pc.lo = 0.f; pc.hi = 0.f; pc.fast_ok = 0;
    return predicate_exact((double)x, (double)b, pc);
}

struct UnitGeom {
    int frame, tx0, ys, ye, yl0, n_in, nchunk;
};
template <int R, int NF>
__device__ __forceinline__ UnitGeom ks_unit(int unit, int strips, int seg_rows, int H, int n_groups) {
    // frame group fastest: the units that share the dark / flat rows of one (strip, segment) run back to back,
    // so those rows are read from DRAM once per launch and served from L2 for the other frames
    UnitGeom u;
    u.frame = (unit % n_groups) * NF;
    int t = unit / n_groups;
    const int strip = t % strips;
    const int seg = t / strips;
    u.tx0 = strip * KS_TW;
    u.ys = seg * seg_rows;
    u.ye = u.ys + seg_rows < H ? u.ys + seg_rows : H;
    u.yl0 = u.ys > 0 ? u.ys - 1 : 0;
    const int yl1 = u.ye < H ? u.ye : H - 1;
    u.n_in = yl1 - u.yl0 + 1;
    u.nchunk = (u.n_in + R - 1) / R;
    return u;
}

// CFG >= 0 bakes the per-launch switches into the instruction stream (the kernel is issue bound: every
// per-row flag test costs); CFG < 0 reads them from the arguments.
enum : int { KS_DARK = 1, KS_FLAT = 2, KS_N2N = 4, KS_MASK = 8, KS_CHECK = 16, KS_LT = 32, KS_NZ = 64, KS_SWAP = 128, KS_NOMED = 256,
             KS_BG = 512, KS_LIN = 1024 };
// KS_LIN: the line model (FLAG_DARK_LINEAR).  tm_dark maps the context's [2][H][W] offset / ascent block and the producer
// loads a box two maps deep (offset rows, then ascent rows) where the dark box was.  Consumers convert both values to
// float64 once per pixel position and, per frame, evaluate bg = offset + ascent * t (DMUL, DADD, the clip to max_value:
// dark_value()'s arithmetic) with the frame's time (K1Args::exposures, or pw.exposure_time); the flat value's float64
// reciprocal stays shared by the frames of the unit.  The checked arithmetic falls back to pointwise() where |bg| is above
// FLT_MAX or NaN
// KS_BG: per-frame backgrounds (K1Args::bg, of the raw dtype) in place of the dark map.  The producer loads one background
// box per frame next to the raw box (evict first: each is read once); the flat value's float64 reciprocal stays shared by
// the frames of the unit, and each frame subtracts float64(float32(its own background sample))
// KS_NOMED: ksize 0 (threshold <= 0, CameraCalibration.py:556-557 skips the artefact step): the pointwise value itself is
// stored, through the same pipeline (one row late, like the median's centre pixel)
// KS_SWAP: big-endian uint16 samples (reader/RAW.py default) — one PRMT per pixel after the shared-memory load
// KS_NZ: a.flat is the zero-free copy (zeros replaced by 1.0) -> unconditional division
// KS_CHECK: non-finite calibration values or float32 raw samples are possible -> test and fall back per pixel

// dark / flat of one pixel position, prepared once for all frames of the unit
struct RowMaps {
    float d, f, s;          // s: the ascent (KS_LIN)
    double dd, fd, y, sd;   // float64 copies and the refined reciprocal of the (zero-free) flat value
};

// medians of two vertically adjacent 3x3 windows from the sorted horizontal triples of four consecutive rows a, b, c, e:
// window 1 = rows (a, b, c), window 2 = rows (b, c, e).  The contribution of the shared rows b, c to the "median of the
// mids" is one ordered pair; max of the lows / min of the highs are single 3-input FMNMX3.  15 min/max per output pixel
// including the sort of the new row (16 with independent windows).
__device__ __forceinline__ void median9_pair(const Sorted3<float>& a, const Sorted3<float>& b, const Sorted3<float>& c,
                                             const Sorted3<float>& e, float& m1, float& m2) {
    const float mlo = vmin(b.mid, c.mid), mhi = vmax(b.mid, c.mid);
    const float mid1 = vmax(mlo, vmin(mhi, a.mid));
    const float mid2 = vmax(mlo, vmin(mhi, e.mid));
    const float lo1 = vmax(vmax(a.lo, b.lo), c.lo), hi1 = vmin(vmin(a.hi, b.hi), c.hi);
    const float lo2 = vmax(vmax(b.lo, c.lo), e.lo), hi2 = vmin(vmin(b.hi, c.hi), e.hi);
    m1 = med3(lo1, mid1, hi1);
    m2 = med3(lo2, mid2, hi2);
}

template <typename RawT, typename OutT, int CFG, typename C>
__global__ void __launch_bounds__(KS_THREADS, C::MINB)
k1_stream_kernel(const __grid_constant__ CUtensorMap tm_raw, const __grid_constant__ CUtensorMap tm_dark,
                 const __grid_constant__ CUtensorMap tm_flat, K1Args a, int strips, int seg_rows, int total_units) {
    constexpr bool BG = CFG >= 0 && (CFG & KS_BG);
    constexpr bool LIN = CFG >= 0 && (CFG & KS_LIN);
    using B = StreamBox<RawT, C, BG, LIN>;
    constexpr int KS_R = C::R, KS_NSTAGE = C::NSTAGE, NF = C::NF;
    static_assert(KS_R % 2 == 0, "rows per stage must be even (outputs are produced in vertical pairs)");
    static_assert(NF == 1 || (CFG >= 0 && !(CFG & KS_MASK)), "multi-frame units: specialised configurations without a mask only");
    // the frame-independent half of the division is hoisted whenever the flat value is known to be non-zero
    constexpr bool FASTDIV = CFG >= 0 && (CFG & KS_NZ) && (CFG & KS_DARK) && (CFG & KS_FLAT);
    static_assert(!BG || FASTDIV, "per-frame backgrounds: the specialised dark + zero-free flat configurations only");
    static_assert(!LIN || FASTDIV, "the line model: the specialised dark + zero-free flat configurations only");
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* full = (uint64_t*)(smem + B::bar_off);
    uint64_t* empty = full + KS_NSTAGE;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool has_dark = CFG >= 0 ? (CFG & KS_DARK) != 0 : a.dark != nullptr;
    const bool has_flat = CFG >= 0 ? (CFG & KS_FLAT) != 0 : a.flat != nullptr;
    const bool has_mask = CFG >= 0 ? (CFG & KS_MASK) != 0 : a.mask != nullptr;
    const bool check = CFG >= 0 ? (CFG & KS_CHECK) != 0 : true;
    const bool swap = CFG >= 0 ? (CFG & KS_SWAP) != 0 : a.raw_swap != 0;
    const bool nomed = CFG >= 0 ? (CFG & KS_NOMED) != 0 : a.ksize == 0;
    const int flags = CFG >= 0 ? ((CFG & KS_DARK ? FLAG_DARK : 0) | (CFG & KS_FLAT ? FLAG_FLAT : 0) | (CFG & KS_N2N ? FLAG_NAN_TO_NUM : 0))
                               : a.pw.flags;
    const int H = a.H, W = a.W;
    const int n_groups = a.n_frames / NF;

    float* sconst = (float*)(smem + B::bar_off + 2 * KS_NSTAGE * sizeof(uint64_t));      // lo, hi, thr (double)
    if (threadIdx.x == 0) {
        for (int s = 0; s < KS_NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], KS_CW); }
        sconst[0] = a.pred.lo; sconst[1] = a.pred.hi; *(double*)(sconst + 2) = a.pred.thr;
        mbar_init_fence();
    }
    __syncthreads();

    if (warp == KS_CW) {
        // ------------------------------------------------------------------ producer
        if (lane != 0) return;
        const uint32_t tx_bytes = (uint32_t)(NF * B::raw_bytes + (has_dark ? B::dark_bytes : 0) + (has_flat ? B::map_bytes : 0));
        uint32_t g = 0;
        for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
            const UnitGeom u = ks_unit<KS_R, NF>(unit, strips, seg_rows, H, n_groups);
            for (int k = 0; k < u.nchunk; ++k, ++g) {
                const int stage = g % KS_NSTAGE;
                mbar_wait(&empty[stage], ((g / KS_NSTAGE) & 1) ^ 1);
                uint8_t* base = smem + (size_t)stage * B::stage_bytes;
                const int y = u.yl0 + k * KS_R;
                mbar_expect_tx(&full[stage], tx_bytes);
                // L2 priorities: raw samples stream through once (evict first), the calibration maps are read again by every
                // frame of this launch and by the next launch (evict last): a one-frame launch then finds most of its 8 B/px of
                // dark / flat in L2 instead of DRAM
#pragma unroll
                for (int f = 0; f < NF; ++f)
                    tma_load_3d_hint(base + f * B::raw_bytes, &tm_raw, &full[stage], (u.tx0 / B::GRAN) * B::GRAN - B::XOFF, y, u.frame + f,
                                     L2_EVICT_FIRST);
                if (BG) {
                    // tm_dark holds the backgrounds [n][H][W]: the same box as the raw samples, streamed once as well
#pragma unroll
                    for (int f = 0; f < NF; ++f)
                        tma_load_3d_hint(base + (NF + f) * B::raw_bytes, &tm_dark, &full[stage], (u.tx0 / B::GRAN) * B::GRAN - B::XOFF, y,
                                         u.frame + f, L2_EVICT_FIRST);
                } else if (LIN) {
                    tma_load_3d_hint(base + NF * B::raw_bytes, &tm_dark, &full[stage], u.tx0 - KS_MAPX, y, 0, L2_EVICT_LAST);
                } else if (has_dark) {
                    tma_load_2d_hint(base + NF * B::raw_bytes, &tm_dark, &full[stage], u.tx0 - KS_MAPX, y, L2_EVICT_LAST);
                }
                if (has_flat) tma_load_2d_hint(base + NF * B::raw_bytes + B::dark_bytes, &tm_flat, &full[stage], u.tx0 - KS_MAPX, y,
                                               L2_EVICT_LAST);
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    const PointwiseConst pw = a.pw;
    // per-launch constants come from shared memory: ptxas would re-read kernel parameters at every use
    PredicateConst pred = a.pred;
    pred.lo = sconst[0]; pred.hi = sconst[1]; pred.thr = *(const double*)(sconst + 2);
    if (CFG >= 0) pred.cond = (CFG & KS_LT) ? COND_LT : COND_GT;
    const int lc = warp * KS_SW - 1 + lane;            // strip-local column of this lane: -1 .. 120
    // results that nobody reads back soon (a K1-only call) leave L2 first, so that the calibration maps stay; inside the
    // chain K2 reads them right away and they keep the normal priority
    const uint64_t out_policy = a.out_streaming ? L2_EVICT_FIRST : L2_EVICT_NORMAL;
    const ptrdiff_t frame_px = (ptrdiff_t)H * W;
    uint32_t g = 0;

    for (int unit = blockIdx.x; unit < total_units; unit += gridDim.x) {
        const UnitGeom u = ks_unit<KS_R, NF>(unit, strips, seg_rows, H, n_groups);
        const int gc = u.tx0 + lc;
        const int rc = reflect_index(gc, W);             // scipy 'reflect' in x: halo / outside lanes read the mirrored column
        int mcol = rc - (u.tx0 - KS_MAPX);
        mcol = mcol < 0 ? 0 : (mcol > KS_MAPW - 1 ? KS_MAPW - 1 : mcol);
        int rcol = rc - ((u.tx0 / B::GRAN) * B::GRAN - B::XOFF);
        rcol = rcol < 0 ? 0 : (rcol > B::BOXW - 1 ? B::BOXW - 1 : rcol);
        const bool valid = lane >= 1 && lane <= KS_SW && gc < W;
        const int i_first = u.ys == 0 ? 1 : 2;           // first input row index whose step emits an output row
        const ptrdiff_t o0 = ((ptrdiff_t)u.frame * H + u.yl0 - 1) * W + gc;          // row (yl0 + i - 1) at step i, first frame
        OutT* outp = (OutT*)a.out + o0;
        uint8_t* maskp = has_mask ? a.mask + o0 : nullptr;

        Sorted3<float> s0[NF], s1[NF];
        float c1[NF];
        int i = 0;
        double tf[NF];                                   // KS_LIN: the exposure time of each frame of the unit
        if constexpr (LIN) {
#pragma unroll
            for (int f = 0; f < NF; ++f) tf[f] = a.exposures ? __ldg(a.exposures + u.frame + f) : pw.exposure_time;
        }

        auto maps = [&](const uint8_t* base, int j, RowMaps& m) {
            m.d = has_dark && !BG ? ((const float*)(base + NF * B::raw_bytes))[j * KS_MAPW + mcol] : 0.0f;
            m.f = has_flat ? ((const float*)(base + NF * B::raw_bytes + B::dark_bytes))[j * KS_MAPW + mcol] : 0.0f;
            if (FASTDIV) {
                m.dd = (double)m.d;
                m.fd = (double)m.f;
                m.y = rcp_f32range(m.fd);
            }
            if constexpr (LIN) {
                m.s = ((const float*)(base + NF * B::raw_bytes + B::map_bytes))[j * KS_MAPW + mcol];
                m.sd = (double)m.s;
            }
        };
        auto pixel = [&](const uint8_t* base, int j, int f, const RowMaps& m) -> float {
            RawT rv = ((const RawT*)(base + f * B::raw_bytes))[j * B::BOXW + rcol];
            if (sizeof(RawT) == 2 && swap) rv = (RawT)__byte_perm((unsigned)rv, 0u, 0x0001);
            double rd; float ra;
            StreamRaw<RawT>::ld(rv, rd, ra);
            float d = m.d;
            double dd = m.dd;
            if constexpr (BG) {
                d = (float)((const RawT*)(base + (NF + f) * B::raw_bytes))[j * B::BOXW + rcol];      // exact for integer samples
                dd = (double)d;
            }
            if constexpr (LIN) {
                dd = dadd(m.dd, dmul(m.sd, tf[f]));
                dd = dd > pw.max_value ? pw.max_value : dd;     // NaN stays NaN
            }
            float x;
            bool ok;
            if (FASTDIV) {
                x = (float)ddiv_rcp(dsub(rd, dd), m.fd, m.y);
                if (flags & FLAG_NAN_TO_NUM) x = fminf(fmaxf(x, -FLT_MAX), FLT_MAX);
                if (check) ok = ((LIN ? (float)fabs(dd) : fabsf(d)) + fabsf(m.f) + ra) <= FLT_MAX;
            } else {
                x = (CFG >= 0 && (CFG & KS_NZ)) ? pointwise_fast_nz(flags, rd, ra, d, m.f, ok) : pointwise_fast(flags, rd, ra, d, m.f, ok);
            }
            if (check) {
                if (!ok) {
                    if constexpr (LIN) {
                        PointwiseConst pf = pw;
                        pf.exposure_time = tf[f];
                        x = pointwise<float>(pf, rd, m.d, m.s, m.f);
                    } else {
                        x = pointwise<float>(pw, rd, d, 0.0f, m.f);
                    }
                }
            }
            return x;
        };
        auto triple = [&](float x) -> Sorted3<float> {
            const float l = __shfl_up_sync(0xffffffffu, x, 1);
            const float r = __shfl_down_sync(0xffffffffu, x, 1);
            return sort3(l, x, r);
        };
        // slow path: one row of frame f, any row (first rows of a unit, short last chunk, guard-band redo)
        auto emit = [&](int f, const Sorted3<float>& t2, bool on) {
            OutT* op = outp + f * frame_px;
            if (nomed) {
                if (on) *op = ks_out<OutT>(a, c1[f]);
                return;
            }
            const float med = median9(s0[f], s1[f], t2);
            bool rep;
            const bool sure = predicate_certain(c1[f], med, pred, rep);
            if (on) {
                *op = ks_out<OutT>(a, rep ? med : c1[f]);
                if (has_mask) *maskp = rep ? 1 : 0;
            }
            // ~1e-5 of the pixels fall inside the guard band of the float32 test: those lanes evaluate the reference's
            // float64 expression out of line and overwrite their result (one warp-uniform branch in the common case)
            if (__any_sync(0xffffffffu, !sure)) {
                if (!sure && on) {
                    const bool r2 = ks_exact(c1[f], med, pred.thr, pred.cond);
                    *op = ks_out<OutT>(a, r2 ? med : c1[f]);
                    if (has_mask) *maskp = r2 ? 1 : 0;
                }
            }
        };
        auto row = [&](const uint8_t* base, int j) {
            RowMaps m;
            maps(base, j, m);
#pragma unroll
            for (int f = 0; f < NF; ++f) {
                const float x = pixel(base, j, f, m);
                const Sorted3<float> t2 = triple(x);
                emit(f, t2, valid && i >= i_first);
                s0[f] = s1[f]; s1[f] = t2; c1[f] = x;
            }
            outp += W;
            if (has_mask) maskp += W;
            ++i;
        };

        for (int k = 0; k < u.nchunk; ++k, ++g) {
            const int stage = g % KS_NSTAGE;
            mbar_wait(&full[stage], (g / KS_NSTAGE) & 1);
            const uint8_t* base = smem + (size_t)stage * B::stage_bytes;
            if (k == 0) {
                // vertical 'reflect' at the top (and a defined s0/s1 elsewhere): the first row's triple is used twice
                RowMaps m;
                maps(base, 0, m);
#pragma unroll
                for (int f = 0; f < NF; ++f) {
                    const float x = pixel(base, 0, f, m);
                    s1[f] = triple(x);
                    s0[f] = s1[f];
                    c1[f] = x;
                }
            }
            const int rows = u.n_in - k * KS_R;
            if (rows >= KS_R) {
                // straight-line chunk: every row emits; the store is unconditional (lanes without an output pixel write to
                // a private scratch slot) and the guard-band test is only accumulated — if any lane of the warp hit the
                // band in this chunk (rare), the chunk is redone below with the exact predicate.  A unit's FIRST chunk goes
                // through here as well: its first one or two steps belong to rows above the unit (the halo row, and the
                // priming step of the vertical 'reflect'), so only their stores are redirected to the scratch slot.
                Sorted3<float> k0[NF], k1[NF];
                float kc[NF];
                OutT* op[NF];
#pragma unroll
                for (int f = 0; f < NF; ++f) {
                    k0[f] = s0[f]; k1[f] = s1[f]; kc[f] = c1[f];
                    op[f] = valid ? outp + f * frame_px
                                  : (OutT*)a.dump + ((size_t)f * gridDim.x + blockIdx.x) * KS_THREADS + threadIdx.x;
                }
                uint8_t* const mdump = (uint8_t*)a.dump + (size_t)(gridDim.x + blockIdx.x) * KS_THREADS * sizeof(OutT) + threadIdx.x;
                uint8_t* mp = has_mask ? (valid ? maskp : mdump) : nullptr;
                const int ostride = valid ? W : 0;       // element index j * ostride stays below 2^31 (R * 32767)
                const bool skip0 = k == 0, skip1 = k == 0 && i_first == 2;      // steps of this chunk that emit nothing
                bool unsure = false;
#pragma unroll
                for (int j = 0; j < KS_R; j += 2) {
                    RowMaps ma, mb;
                    maps(base, j, ma);
                    maps(base, j + 1, mb);
#pragma unroll
                    for (int f = 0; f < NF; ++f) {
                        const float xa = pixel(base, j, f, ma);
                        const float xb = pixel(base, j + 1, f, mb);
                        OutT* d0 = op[f] + j * ostride;
                        OutT* d1 = op[f] + (j + 1) * ostride;
                        if (j == 0) {
                            OutT* const dumpp = (OutT*)a.dump + ((size_t)f * gridDim.x + blockIdx.x) * KS_THREADS + threadIdx.x;
                            d0 = skip0 ? dumpp : d0;
                            d1 = skip1 ? dumpp : d1;
                        }
                        if (nomed) {
                            ks_store<OutT>(d0, ks_out<OutT>(a, c1[f]), out_policy);
                            ks_store<OutT>(d1, ks_out<OutT>(a, xa), out_policy);
                            c1[f] = xb;
                            continue;
                        }
                        const Sorted3<float> ta = triple(xa), tb = triple(xb);
                        float m1, m2;
                        median9_pair(s0[f], s1[f], ta, tb, m1, m2);
                        bool r1, r2;
                        unsure |= !predicate_certain(c1[f], m1, pred, r1);
                        unsure |= !predicate_certain(xa, m2, pred, r2);
                        ks_store<OutT>(d0, ks_out<OutT>(a, r1 ? m1 : c1[f]), out_policy);
                        ks_store<OutT>(d1, ks_out<OutT>(a, r2 ? m2 : xa), out_policy);
                        if (has_mask) {
                            *((j == 0 && skip0) ? mdump : mp + j * ostride) = r1 ? 1 : 0;
                            *((j == 0 && skip1) ? mdump : mp + (j + 1) * ostride) = r2 ? 1 : 0;
                        }
                        s0[f] = ta; s1[f] = tb; c1[f] = xb;
                    }
                }
                if (__any_sync(0xffffffffu, unsure)) {
#pragma unroll
                    for (int f = 0; f < NF; ++f) { s0[f] = k0[f]; s1[f] = k1[f]; c1[f] = kc[f]; }
                    for (int j = 0; j < KS_R; ++j) row(base, j);
                } else {
                    outp += (size_t)KS_R * W;
                    if (has_mask) maskp += (size_t)KS_R * W;
                    i += KS_R;
                }
            } else {
                const int n = rows < KS_R ? rows : KS_R;
                for (int j = 0; j < n; ++j) row(base, j);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
        }
        if (u.ye == H) {
            // vertical 'reflect' at the bottom: output row H-1 sees (H-2, H-1, H-1)
#pragma unroll
            for (int f = 0; f < NF; ++f) {
                const Sorted3<float> t2 = s1[f];
                emit(f, t2, valid);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------ host
// per-frame backgrounds stream in these configurations only (the dtype pairs and options the instantiations below cover):
// a background of the raw dtype, uint16 or float32 frames, native byte order, the chain's dark + flat (+ nan_to_num) with
// the 3x3 median, or dark + flat alone with threshold <= 0.  Returns the configuration, or -1 (the generic tiles).
static int ks_bg_cfg(const K1Args& a, int raw_dtype) {
    if (!a.bg || a.bg_dtype != raw_dtype || (raw_dtype != DT_U16 && raw_dtype != DT_F32)) return -1;
    const int f = a.pw.flags;
    if (a.raw_swap || a.mask || a.dark || !a.flat || !a.flat_nz || !(f & FLAG_DARK) || !(f & FLAG_FLAT) || (f & FLAG_DARK_LINEAR))
        return -1;
    // float32 backgrounds can hold NaN / inf / FLT_MAX: the checked arithmetic, as for float32 frames
    const bool check = !a.maps_finite || raw_dtype == DT_F32;
    const int base = KS_BG | KS_DARK | KS_FLAT | KS_NZ;
    if (a.ksize == 3) {
        if (!(f & FLAG_NAN_TO_NUM) || a.pred.cond != COND_GT) return -1;
        return check ? base | KS_N2N | KS_CHECK : a.no_overflow ? base : base | KS_N2N;
    }
    if (a.ksize == 0 && a.H >= 4) {
        const int n2n = (f & FLAG_NAN_TO_NUM) && !a.no_overflow ? KS_N2N : 0;
        if (raw_dtype == DT_F32) return base | KS_NOMED | KS_CHECK | n2n;
        return check ? -1 : base | KS_NOMED | n2n;
    }
    return -1;
}

// the line model streams in the same configurations as per-frame backgrounds (uint16 and float32 frames, the chain's 3x3
// and threshold <= 0), with the context's [2][H][W] offset / ascent block.  Returns the configuration, or -1
static int ks_lin_cfg(const K1Args& a, int raw_dtype) {
    const int f = a.pw.flags;
    if (!(f & FLAG_DARK_LINEAR) || a.bg || (raw_dtype != DT_U16 && raw_dtype != DT_F32)) return -1;
    if (a.raw_swap || a.mask || !a.dark || a.ascent != a.dark + (size_t)a.H * a.W || !a.flat || !a.flat_nz || !(f & FLAG_DARK) ||
        !(f & FLAG_FLAT))
        return -1;
    const bool check = !a.maps_finite || raw_dtype == DT_F32;
    const int base = KS_LIN | KS_DARK | KS_FLAT | KS_NZ;
    if (a.ksize == 3) {
        if (!(f & FLAG_NAN_TO_NUM) || a.pred.cond != COND_GT) return -1;
        return check ? base | KS_N2N | KS_CHECK : a.no_overflow ? base : base | KS_N2N;
    }
    if (a.ksize == 0 && a.H >= 4) {
        const int n2n = (f & FLAG_NAN_TO_NUM) && !a.no_overflow ? KS_N2N : 0;
        if (raw_dtype == DT_F32) return base | KS_NOMED | KS_CHECK | n2n;
        return check ? -1 : base | KS_NOMED | n2n;
    }
    return -1;
}

bool k1_stream_eligible(const K1Args& a, int raw_dtype, int out_dtype) {
    if (a.ksize != 3 && a.ksize != 0) return false;
    if (a.ksize == 0 && a.H < 4) return false;
    if (raw_dtype != DT_U8 && raw_dtype != DT_U16 && raw_dtype != DT_F32) return false;
    if (out_dtype != DT_F32 && out_dtype != DT_U16 && out_dtype != DT_U8) return false;
    if ((a.pw.flags & FLAG_DARK_LINEAR) && ks_lin_cfg(a, raw_dtype) < 0) return false;
    if (a.raw_gap) return false;
    const size_t esz = dtype_size(raw_dtype);
    if (((size_t)a.W * esz) % 16 || ((size_t)a.W * 4) % 16) return false;
    if (((size_t)a.H * a.W * esz) % 16) return false;
    if (((uintptr_t)a.raw) % 16) return false;
    if (a.dark && ((uintptr_t)a.dark) % 16) return false;
    if (a.flat && ((uintptr_t)a.flat) % 16) return false;
    if (a.bg && (ks_bg_cfg(a, raw_dtype) < 0 || ((uintptr_t)a.bg) % 16)) return false;
    return tensor_map_encoder() != nullptr;
}

typedef void (*ks_kern_t)(const CUtensorMap, const CUtensorMap, const CUtensorMap, K1Args, int, int, int);

// the per-frame-background instantiations of one raw dtype (uint16: finite flat maps, with and without the overflow proof,
// and the checked chain; float32: checked only), or null
template <typename RawT, typename OutT, typename C>
static ks_kern_t ks_bg_kernel(int cfg) {
    constexpr int B0 = KS_BG | KS_DARK | KS_FLAT | KS_NZ;
    if constexpr (sizeof(RawT) == 2) {
        if (cfg == B0) return k1_stream_kernel<RawT, OutT, B0, C>;
        if (cfg == (B0 | KS_N2N)) return k1_stream_kernel<RawT, OutT, B0 | KS_N2N, C>;
        if constexpr (C::NF == 1) {
            if (cfg == (B0 | KS_N2N | KS_CHECK)) return k1_stream_kernel<RawT, OutT, B0 | KS_N2N | KS_CHECK, C>;
            if (cfg == (B0 | KS_NOMED)) return k1_stream_kernel<RawT, OutT, B0 | KS_NOMED, C>;
            if (cfg == (B0 | KS_NOMED | KS_N2N)) return k1_stream_kernel<RawT, OutT, B0 | KS_NOMED | KS_N2N, C>;
        }
    } else if constexpr (sizeof(RawT) == 4) {
        if (cfg == (B0 | KS_N2N | KS_CHECK)) return k1_stream_kernel<RawT, OutT, B0 | KS_N2N | KS_CHECK, C>;
        if constexpr (C::NF == 1) {
            if (cfg == (B0 | KS_NOMED | KS_CHECK)) return k1_stream_kernel<RawT, OutT, B0 | KS_NOMED | KS_CHECK, C>;
            if (cfg == (B0 | KS_NOMED | KS_CHECK | KS_N2N)) return k1_stream_kernel<RawT, OutT, B0 | KS_NOMED | KS_CHECK | KS_N2N, C>;
        }
    }
    return nullptr;
}

// the line-model instantiations, the same set as ks_bg_kernel's (uint16: finite maps with and without the overflow proof,
// and the checked chain; float32: checked only), or null
template <typename RawT, typename OutT, typename C>
static ks_kern_t ks_lin_kernel(int cfg) {
    constexpr int B0 = KS_LIN | KS_DARK | KS_FLAT | KS_NZ;
    if constexpr (sizeof(RawT) == 2) {
        if (cfg == B0) return k1_stream_kernel<RawT, OutT, B0, C>;
        if (cfg == (B0 | KS_N2N)) return k1_stream_kernel<RawT, OutT, B0 | KS_N2N, C>;
        if constexpr (C::NF == 1) {
            if (cfg == (B0 | KS_N2N | KS_CHECK)) return k1_stream_kernel<RawT, OutT, B0 | KS_N2N | KS_CHECK, C>;
            if (cfg == (B0 | KS_NOMED)) return k1_stream_kernel<RawT, OutT, B0 | KS_NOMED, C>;
            if (cfg == (B0 | KS_NOMED | KS_N2N)) return k1_stream_kernel<RawT, OutT, B0 | KS_NOMED | KS_N2N, C>;
        }
    } else if constexpr (sizeof(RawT) == 4) {
        if (cfg == (B0 | KS_N2N | KS_CHECK)) return k1_stream_kernel<RawT, OutT, B0 | KS_N2N | KS_CHECK, C>;
        if constexpr (C::NF == 1) {
            if (cfg == (B0 | KS_NOMED | KS_CHECK)) return k1_stream_kernel<RawT, OutT, B0 | KS_NOMED | KS_CHECK, C>;
            if (cfg == (B0 | KS_NOMED | KS_CHECK | KS_N2N)) return k1_stream_kernel<RawT, OutT, B0 | KS_NOMED | KS_CHECK | KS_N2N, C>;
        }
    }
    return nullptr;
}

// grid, segment height and launch of a streaming instantiation with stage layout B
template <typename B, typename C>
static cudaError_t ks_run(ks_kern_t kern, const K1Args& a, const CUtensorMap& tr, const CUtensorMap& td, const CUtensorMap& tf,
                          int sm_count, int seg_rows, cudaStream_t st) {
    constexpr int KS_R = C::R, NF = C::NF;
    cudaError_t e = cudaSuccess;
    const int per_sm = blocks_per_sm_cached((const void*)kern, KS_THREADS, B::total, &e);
    if (e != cudaSuccess) return e;
    const int strips = (a.W + KS_TW - 1) / KS_TW;
    const int n_groups = a.n_frames / NF;
    const long long slots = (long long)sm_count * per_sm;
    if (seg_rows <= 0) {
        // all units cost the same: pick the segment height whose unit count fills whole waves of the resident CTAs best,
        // counting the two re-read halo rows per segment against it.  (Searching beyond 8 waves finds better fills on
        // paper — 231-row segments for 32 frames — but measured slower, 36.1 vs 33.6 us/frame: every unit start refills
        // the pipeline and runs its first chunk row by row.)
        double best = -1.0;
        for (int waves = 1; waves <= 8; ++waves) {
            long long segs_try = slots * waves / ((long long)strips * n_groups);
            if (segs_try < 1) continue;
            int rows = (int)((a.H + segs_try - 1) / segs_try);
            if (rows < 2 * KS_R) rows = 2 * KS_R;
            const long long units = (long long)strips * ((a.H + rows - 1) / rows) * n_groups;
            const double util = (double)units / (double)(((units + slots - 1) / slots) * slots) * rows / (rows + 2.0);
            if (util > best) { best = util; seg_rows = rows; }
        }
        if (seg_rows <= 0) seg_rows = a.H;
    }
    if (seg_rows < 4) seg_rows = 4;
    const int segs = (a.H + seg_rows - 1) / seg_rows;
    const long long total = (long long)strips * segs * n_groups;
    if (total > 0x7fffffffLL) return cudaErrorInvalidValue;
    long long grid = slots;
    if (grid > total) grid = total;
    kern<<<(unsigned)grid, KS_THREADS, B::total, st>>>(tr, td, tf, a, strips, seg_rows, (int)total);
    return cudaGetLastError();
}

// per-frame backgrounds (ks_bg_cfg): the background block is a second 3-D map with the raw samples' box
template <typename RawT, typename OutT, typename C>
static cudaError_t launch_stream_bg(const K1Args& a_in, CUtensorMapDataType rdt, int sm_count, int seg_rows, cudaStream_t st) {
    using B = StreamBox<RawT, C, true>;
    constexpr int RDT = sizeof(RawT) == 1 ? DT_U8 : sizeof(RawT) == 2 ? DT_U16 : DT_F32;
    K1Args a = a_in;
    const int cfg = ks_bg_cfg(a, RDT);
    if (cfg < 0 || a.n_frames % C::NF) return cudaErrorInvalidValue;
    ks_kern_t kern = ks_bg_kernel<RawT, OutT, C>(cfg);
    if (!kern) return cudaErrorInvalidValue;
    a.flat = a.flat_nz;                                  // zero-free copy: an unconditional division
    CUtensorMap tr, tb, tf;
    if (!make_tensor_map(&tr, rdt, sizeof(RawT), a.raw, a.W, a.H, a.n_frames, B::BOXW, C::R)) return cudaErrorInvalidValue;
    if (!make_tensor_map(&tb, rdt, sizeof(RawT), a.bg, a.W, a.H, a.n_frames, B::BOXW, C::R)) return cudaErrorInvalidValue;
    if (!make_tensor_map(&tf, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.flat, a.W, a.H, 0, KS_MAPW, C::R)) return cudaErrorInvalidValue;
    return ks_run<B, C>(kern, a, tr, tb, tf, sm_count, seg_rows, st);
}

// the line model (ks_lin_cfg): the offset / ascent block is a 3-D map two deep, loaded as one box
template <typename RawT, typename OutT, typename C>
static cudaError_t launch_stream_lin(const K1Args& a_in, CUtensorMapDataType rdt, int sm_count, int seg_rows, cudaStream_t st) {
    using B = StreamBox<RawT, C, false, true>;
    constexpr int RDT = sizeof(RawT) == 1 ? DT_U8 : sizeof(RawT) == 2 ? DT_U16 : DT_F32;
    K1Args a = a_in;
    const int cfg = ks_lin_cfg(a, RDT);
    if (cfg < 0 || a.n_frames % C::NF) return cudaErrorInvalidValue;
    ks_kern_t kern = ks_lin_kernel<RawT, OutT, C>(cfg);
    if (!kern) return cudaErrorInvalidValue;
    a.flat = a.flat_nz;                                  // zero-free copy: an unconditional division
    CUtensorMap tr, td, tf;
    if (!make_tensor_map(&tr, rdt, sizeof(RawT), a.raw, a.W, a.H, a.n_frames, B::BOXW, C::R)) return cudaErrorInvalidValue;
    if (!make_tensor_map(&td, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.dark, a.W, a.H, 2, KS_MAPW, C::R, 2)) return cudaErrorInvalidValue;
    if (!make_tensor_map(&tf, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.flat, a.W, a.H, 0, KS_MAPW, C::R)) return cudaErrorInvalidValue;
    return ks_run<B, C>(kern, a, tr, td, tf, sm_count, seg_rows, st);
}

template <typename RawT, typename OutT, typename C>
static cudaError_t launch_stream_c(const K1Args& a_in, CUtensorMapDataType rdt, int sm_count, int seg_rows, cudaStream_t st) {
    using B = StreamBox<RawT, C>;
    constexpr int KS_R = C::R, NF = C::NF;
    K1Args a = a_in;
    // pick the instantiation: the hot configurations are fully specialised, the rest read their flags at run time
    const bool check = !a.maps_finite || sizeof(RawT) == 4;
    const int f = a.pw.flags;
    const bool chain = a.ksize == 3 && a.dark && a.flat && a.flat_nz && (f & FLAG_DARK) && (f & FLAG_FLAT) && (f & FLAG_NAN_TO_NUM) && !a.mask &&
                       a.pred.cond == COND_GT;
    const bool plain = a.ksize == 3 && !(f & (FLAG_DARK | FLAG_FLAT | FLAG_NAN_TO_NUM)) && a.mask && a.pred.cond == COND_GT;
    ks_kern_t kern = nullptr;
    // threshold <= 0: dark + flat only (nan_to_num is not applied then, CameraCalibration.py:556-561)
    const bool pw_only = a.ksize == 0 && a.dark && a.flat && a.flat_nz && (f & FLAG_DARK) && (f & FLAG_FLAT) && !a.raw_swap && !check;
    if (chain || pw_only) a.flat = a.flat_nz;          // zero-free copy: "divide where flat != 0" becomes an unconditional division
    if constexpr (NF > 1) {
        // frame-pair units: the chain configurations only (launch_stream_t sends nothing else here)
        if (!chain || a.raw_swap || a.n_frames % NF) return cudaErrorInvalidValue;
        if (!check && a.no_overflow) kern = k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_NZ, C>;
        else if (!check) kern = k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_N2N | KS_NZ, C>;
        else kern = k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_N2N | KS_NZ | KS_CHECK, C>;
    } else {
        if (pw_only) {
            kern = (f & FLAG_NAN_TO_NUM) && !a.no_overflow ? k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_N2N | KS_NZ | KS_NOMED, C>
                                                           : k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_NZ | KS_NOMED, C>;
        } else if (a.raw_swap && chain && !check && sizeof(RawT) == 2) {
            kern = a.no_overflow ? k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_NZ | KS_SWAP, C>
                                 : k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_N2N | KS_NZ | KS_SWAP, C>;
        } else if (a.raw_swap) { kern = k1_stream_kernel<RawT, OutT, -1, C>; if (chain) a.flat = a_in.flat; }
        else if (chain && !check && a.no_overflow) kern = k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_NZ, C>;
        else if (chain && !check) kern = k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_N2N | KS_NZ, C>;
        else if (chain) kern = k1_stream_kernel<RawT, OutT, KS_DARK | KS_FLAT | KS_N2N | KS_NZ | KS_CHECK, C>;
        else if (plain) kern = k1_stream_kernel<RawT, OutT, KS_MASK, C>;
        else kern = k1_stream_kernel<RawT, OutT, -1, C>;
    }
    CUtensorMap tr, td, tf;
    if (!make_tensor_map(&tr, rdt, sizeof(RawT), a.raw, a.W, a.H, a.n_frames, B::BOXW, KS_R)) return cudaErrorInvalidValue;
    if (!make_tensor_map(&td, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.dark ? (const void*)a.dark : a.raw, a.W, a.H, 0, KS_MAPW, KS_R) && a.dark)
        return cudaErrorInvalidValue;
    if (!make_tensor_map(&tf, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.flat ? (const void*)a.flat : a.raw, a.W, a.H, 0, KS_MAPW, KS_R) && a.flat)
        return cudaErrorInvalidValue;
    return ks_run<B, C>(kern, a, tr, td, tf, sm_count, seg_rows, st);
}

template <typename RawT, typename OutT>
static cudaError_t launch_stream_t(const K1Args& a, CUtensorMapDataType rdt, int sm_count, int seg_rows, cudaStream_t st) {
    if constexpr (sizeof(OutT) == 4) {
        const int f = a.pw.flags;
        const bool chain = a.ksize == 3 && (a.dark || a.bg) && a.flat && a.flat_nz && (f & FLAG_DARK) && (f & FLAG_FLAT) &&
                           (f & FLAG_NAN_TO_NUM) && !a.mask && a.pred.cond == COND_GT && !a.raw_swap;
        if (a.pw.flags & FLAG_DARK_LINEAR) {
            // the line model: frame pairs of the chain (uint16 frames with finite maps and a bounded |bg|, float32 frames),
            // everything else and an odd last frame one frame per unit
            using P = typename std::conditional<sizeof(RawT) == 4, KsPairLinF32, KsPairLin>::type;
            if (!chain || a.n_frames < 4 || (sizeof(RawT) != 4 && !a.maps_finite))
                return launch_stream_lin<RawT, OutT, KsNarrowLin>(a, rdt, sm_count, seg_rows, st);
            const int even = a.n_frames & ~1;
            K1Args b = a;
            b.n_frames = even;
            cudaError_t e = launch_stream_lin<RawT, OutT, P>(b, rdt, sm_count, seg_rows, st);
            if (e != cudaSuccess || even == a.n_frames) return e;
            b = a;
            b.n_frames = 1;
            b.raw = (const char*)a.raw + (size_t)even * a.H * a.W * sizeof(RawT);
            b.out = (char*)a.out + (size_t)even * a.H * a.W * sizeof(OutT);
            if (b.exposures) b.exposures += even;
            return launch_stream_lin<RawT, OutT, KsNarrowLin>(b, rdt, sm_count, seg_rows, st);
        }
        if (a.bg) {
            // per-frame backgrounds: frame pairs of the chain (uint16 frames with a finite flat field, float32 frames),
            // everything else and an odd last frame one frame per unit in the narrow shape
            using P = typename std::conditional<sizeof(RawT) == 4, KsPairBgF32, KsPairBg>::type;
            if (!chain || a.n_frames < 4 || (sizeof(RawT) != 4 && !a.maps_finite))
                return launch_stream_bg<RawT, OutT, KsNarrow>(a, rdt, sm_count, seg_rows, st);
            const int even = a.n_frames & ~1;
            K1Args b = a;
            b.n_frames = even;
            cudaError_t e = launch_stream_bg<RawT, OutT, P>(b, rdt, sm_count, seg_rows, st);
            if (e != cudaSuccess || even == a.n_frames) return e;
            b = a;
            b.n_frames = 1;
            b.raw = (const char*)a.raw + (size_t)even * a.H * a.W * sizeof(RawT);
            b.bg = (const char*)a.bg + (size_t)even * a.H * a.W * sizeof(RawT);
            b.out = (char*)a.out + (size_t)even * a.H * a.W * sizeof(OutT);
            return launch_stream_bg<RawT, OutT, KsNarrow>(b, rdt, sm_count, seg_rows, st);
        }
        // batches of the chain configuration: two frames per work unit share the dark / flat half of the arithmetic;
        // an odd last frame goes through the one-frame kernel
        if (chain && a.n_frames >= 4) {
            const int even = a.n_frames & ~1;
            K1Args b = a;
            b.n_frames = even;
            cudaError_t e = launch_stream_c<RawT, OutT, KsPair>(b, rdt, sm_count, seg_rows, st);
            if (e != cudaSuccess || even == a.n_frames) return e;
            b = a;
            b.n_frames = 1;
            b.raw = (const char*)a.raw + (size_t)even * a.H * a.W * sizeof(RawT);
            b.out = (char*)a.out + (size_t)even * a.H * a.W * sizeof(OutT);
            return launch_stream_c<RawT, OutT, KsNarrow>(b, rdt, sm_count, seg_rows, st);
        }
        // the wide shape pays with float32 output and a few frames per launch (see KsShape)
        if (a.n_frames >= 4) return launch_stream_c<RawT, OutT, KsWide>(a, rdt, sm_count, seg_rows, st);
    }
    if (a.pw.flags & FLAG_DARK_LINEAR) return launch_stream_lin<RawT, OutT, KsNarrowLin>(a, rdt, sm_count, seg_rows, st);
    if (a.bg) return launch_stream_bg<RawT, OutT, KsNarrow>(a, rdt, sm_count, seg_rows, st);
    return launch_stream_c<RawT, OutT, KsNarrow>(a, rdt, sm_count, seg_rows, st);
}

cudaError_t launch_k1_stream(const K1Args& a, int raw_dtype, int out_dtype, int sm_count, int seg_rows, cudaStream_t st) {
    switch (raw_dtype) {
        case DT_U8:
            if (out_dtype == DT_F32) return launch_stream_t<uint8_t, float>(a, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, seg_rows, st);
            if (out_dtype == DT_U8) return launch_stream_t<uint8_t, uint8_t>(a, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, seg_rows, st);
            if (out_dtype == DT_U16) return launch_stream_t<uint8_t, uint16_t>(a, CU_TENSOR_MAP_DATA_TYPE_UINT8, sm_count, seg_rows, st);
            break;
        case DT_U16:
            if (out_dtype == DT_F32) return launch_stream_t<uint16_t, float>(a, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, seg_rows, st);
            if (out_dtype == DT_U16) return launch_stream_t<uint16_t, uint16_t>(a, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, seg_rows, st);
            if (out_dtype == DT_U8) return launch_stream_t<uint16_t, uint8_t>(a, CU_TENSOR_MAP_DATA_TYPE_UINT16, sm_count, seg_rows, st);
            break;
        case DT_F32:
            if (out_dtype == DT_F32) return launch_stream_t<float, float>(a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, seg_rows, st);
            if (out_dtype == DT_U16) return launch_stream_t<float, uint16_t>(a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, seg_rows, st);
            if (out_dtype == DT_U8) return launch_stream_t<float, uint8_t>(a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sm_count, seg_rows, st);
            break;
    }
    return cudaErrorInvalidValue;
}

}  // namespace imgcorr
