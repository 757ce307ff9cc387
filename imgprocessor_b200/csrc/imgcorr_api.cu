// imgcorr_api.cu — the C ABI declared in include/imgcorr.h: context, calibration upload,
// kernel entry points, the device-resident chain and the host-buffer streaming pipeline.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <algorithm>
#include <memory>
#include <type_traits>
#include <vector>
#include <thread>

#include "../../include/imgcorr.h"
#include "imgcorr_kernels.cuh"

using namespace imgcorr;

static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
static int cuda_fail(cudaError_t e, const char* what) {
    return fail(IMGCORR_ERR_CUDA, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
}
#define CK(call)                                             \
    do {                                                     \
        cudaError_t e__ = (call);                            \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

// ---- owning handles: every CUDA resource the library keeps is released by its handle's destructor ---------------------
struct DevFree { void operator()(void* p) const { cudaFree(p); } };
struct HostFree { void operator()(void* p) const { cudaFreeHost(p); } };
struct EventFree { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
struct StreamFree { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
template <class T> using DevPtr = std::unique_ptr<T, DevFree>;
using PinnedPtr = std::unique_ptr<void, HostFree>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventFree>;
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamFree>;

// creation fills an empty handle and returns the CUDA error (nothing throws); on failure the handle stays empty
template <class H, class Create> static cudaError_t create(H& h, Create&& make) {
    typename H::pointer raw = nullptr;
    const cudaError_t e = make(&raw);
    h.reset(e == cudaSuccess ? raw : nullptr);
    return e;
}
template <class T> static cudaError_t dev_alloc(DevPtr<T>& p, size_t bytes) {
    return create(p, [&](T** raw) { return cudaMalloc((void**)raw, bytes); });
}
static cudaError_t host_alloc(PinnedPtr& p, size_t bytes) {
    return create(p, [&](void** raw) { return cudaHostAlloc(raw, bytes, cudaHostAllocDefault); });
}
static cudaError_t new_event(Event& ev, unsigned flags = cudaEventDisableTiming) {
    return create(ev, [&](cudaEvent_t* raw) { return cudaEventCreateWithFlags(raw, flags); });
}
static cudaError_t new_stream(Stream& s, int priority = 0) {      // non-blocking; 0 is the default priority
    return create(s, [&](cudaStream_t* raw) { return cudaStreamCreateWithPriority(raw, cudaStreamNonBlocking, priority); });
}

// 256 bytes, the alignment cudaMalloc gives: K1's TMA paths and K2's tiled path need 16-byte aligned frames and quietly
// take slower kernels otherwise, so every part of a split allocation starts on such a boundary
static size_t round256(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// Device memory that every call of one kind shares, one per context.  Calls may come on different streams: a call on
// another stream than the last user first waits until that user's launches are done with it.
struct SharedScratch {
    DevPtr<char> buf;
    size_t bytes = 0;
    Event last_use;                                 // recorded on the last user's stream after its last launch
    cudaStream_t last_st = nullptr;

    // at least `need` bytes, ordered on `st` after the last use
    cudaError_t acquire(size_t need, cudaStream_t st) {
        cudaError_t e;
        if (bytes < need) {
            // launches on other streams may still use the old buffer; it goes before the new one is allocated, so
            // peak memory stays one buffer, and a failed allocation leaves the scratch empty for the next call to retry
            if (buf && (e = cudaDeviceSynchronize()) != cudaSuccess) return e;
            buf.reset();
            bytes = 0;
            if ((e = dev_alloc(buf, need)) != cudaSuccess) return e;
            bytes = need;
        }
        if (!last_use) return new_event(last_use);
        return last_st == st ? cudaSuccess : cudaStreamWaitEvent(st, last_use.get(), 0);
    }
    void release(cudaStream_t st) { cudaEventRecord(last_use.get(), st); last_st = st; }
    struct Guard {                                  // releases on every exit path of the call that acquired the scratch
        SharedScratch& s;
        cudaStream_t st;
        ~Guard() { s.release(st); }
    };
};

struct HostSlot {
    DevPtr<void> d_raw, d_out;
    PinnedPtr h_raw, h_out;
    DevPtr<void> d_bg;                        // per-frame backgrounds of the slot's chunk (imgcorr_correct_host_bg only)
    PinnedPtr h_bg;                           // their staging for pageable input
    Event ev_in, ev_k, ev_out;
};

struct imgcorr_ctx {
    int device = 0, H = 0, W = 0, sm_count = 148;
    DevPtr<float> dark, flat;                 // dark: [H][W], or [2][H][W] = offset, ascent with the line model (`linear`)
    bool linear = false;
    double exposure = 0.0, maxval = 65535.0;
    DevPtr<double> exposures;                 // imgcorr_set_dark_exposures: one time per frame of a call, or empty
    int n_exposures = 0;
    double exposures_absmax = 0.0;            // max |t| over the table
    OutScale out_scale{0.0, 1.0};             // imgcorr_set_output_scale: read by chain calls with U16 / U8 output
    bool has_lens = false;
    LensConst lens{};
    LensExt lens_x{};                         // the lens' rational / thin-prism / tilt terms, used when lens_ext is set
    bool lens_ext = false;                    // some extra term is non-zero: K2 runs its EXT kernels
    double lens_in[33] = {0};                 // K, dist (14, zero-padded), P and the coefficient count as last given to
                                              // imgcorr_set_lens_model (an identical call is a no-op)
    DevPtr<double> lens_dev;
    DevPtr<float4> k2_wtab;                   // OpenCV's BilinearTab_f [32][32] (K2 tiles)
    struct GeomKey { int x0, y0, ow, oh, esz, g; };
    std::vector<GeomKey> k2_geom;             // staged-box geometry per output window (k2_pick_geometry), reset by set_lens
    // K2 coordinate cache: packed per-pixel source coordinates of the current lens for an output window (4 bytes per pixel),
    // written by the first tiled launch, read by the following ones; dropped by set_lens
    struct K2Cache { int x0, y0, ow, oh, g, esz; DevPtr<unsigned> pack; DevPtr<int2> hdr; Event ev; cudaStream_t st; unsigned long long stamp; };
    std::vector<K2Cache> k2_cache;
    int k2_cache_on = 1;
    unsigned long long k2_stamp = 0;
    DevPtr<void> dump;                        // scratch for stores of lanes that own no output pixel
    int raw_big_endian = 0;
    long long raw_gap = 0;
    int k1_variant = 0, k2_variant = 0, k3_variant = 0, host_slots = 4, k1_seg_rows = 0, profile = 0, chain_group = 16;
    long long chain_groups_seen = 0;
    double prof_frames[2] = {0.0, 0.0};
    std::vector<Event> prof_ev[2];            // [kernel] start/stop pairs (timing events)
    bool dark_finite = true, flat_finite = true, ascent_finite = true;
    DevPtr<float> flat_nz;                    // flat with zeros replaced by 1.0
    double dark_absmax = 0.0, ascent_absmax = 0.0, flat_absmin = 1.0;   // over finite entries (flat: non-zero entries)
    long long launches = 0;
    // the chain's K1 output (with a lens: two halves of `chain_group` float32 frames each), then the warp source of the
    // perspective stage (a group of chain frames in the output dtype)
    SharedScratch chain_scratch;
    // one matrix M (imgcorr_set_perspective), or a device table of one inverted matrix per frame (imgcorr_set_perspective_frames)
    struct Perspective {
        bool on = false; double M[9]; int dh = 0, dw = 0; double border = 0.0; DevPtr<double> tilt; int th = 0, tw = 0;
        DevPtr<WarpConst> table; int n_table = 0;
    };
    Perspective persp;                        // the chain's last stage
    int chain_overlap = 1;                    // K1 of group g+1 on the internal stream while K2 of group g runs: +2-3.5 % on batches
    struct ChainOverlap { Stream st; Event k1[2], k2[2], entry; };
    ChainOverlap ov;                          // high-priority stream of K1 in overlap mode and its hand-off events
    SharedScratch ste_scratch;                // K4: second running-average buffer, thresholds, counts
    DevPtr<int16_t> warp_itab[2];             // [bicubic, Lanczos4] fixed-point weights for uint8 images (K3)
    DevPtr<float> warp_tab;                   // [32][8] Lanczos4 then [32][4] bicubic coefficient tables (K3)
    // host pipeline
    Stream s_in, s_k, s_out;
    std::vector<HostSlot> slots;
    size_t slot_raw_bytes = 0, slot_out_bytes = 0, slot_bg_bytes = 0;
};

// The end of every launch: count the kernels the launch helper issued and map its error to a status.  K1, K2 and K3 name
// the errors they can explain: a requested variant that is not eligible, and a dtype pair no kernel implements (`pair`,
// formatted with the two dtypes).
static int launched(imgcorr_ctx* c, int l, cudaError_t e, const char* what, const char* ineligible = nullptr,
                    const char* pair = nullptr, int dt_in = 0, int dt_out = 0) {
    c->launches += l;
    if (e == cudaSuccess) return IMGCORR_OK;
    if (pair && e == cudaErrorInvalidValue && l == 0) return fail(IMGCORR_ERR_INVALID, pair, dt_in, dt_out);
    if (ineligible && e == cudaErrorNotSupported) return fail(IMGCORR_ERR_INVALID, "%s", ineligible);
    return cuda_fail(e, what);
}

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define GUARD(ctx)                                                           \
    if (!(ctx)) return fail(IMGCORR_ERR_INVALID, "null context");            \
    DeviceGuard guard__((ctx)->device);                                      \
    if (!guard__.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice")

extern "C" IMGCORR_API const char* imgcorr_last_error(void) { return g_err.c_str(); }
extern "C" IMGCORR_API int imgcorr_version(void) { return IMGCORR_VERSION; }

extern "C" IMGCORR_API int imgcorr_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
    return n;
}

extern "C" IMGCORR_API int imgcorr_ctx_create(int device, int height, int width, imgcorr_ctx** out_ctx) {
    if (!out_ctx) return fail(IMGCORR_ERR_INVALID, "out_ctx is null");
    *out_ctx = nullptr;
    if (height <= 0 || width <= 0) return fail(IMGCORR_ERR_INVALID, "bad frame shape %d x %d", height, width);
    int n = 0;
    CK(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(IMGCORR_ERR_INVALID, "device %d out of range (%d devices)", device, n);
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(IMGCORR_ERR_CUDA, "device %d is sm_%d%d; libimgcorr is built for sm_100a only", device, prop.major,
                    prop.minor);
    imgcorr_ctx* c = new (std::nothrow) imgcorr_ctx();
    if (!c) return fail(IMGCORR_ERR_NOMEM, "out of host memory");
    c->device = device;
    c->H = height;
    c->W = width;
    c->sm_count = prop.multiProcessorCount;
    *out_ctx = c;
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_ctx_destroy(imgcorr_ctx* c) {
    if (!c) return IMGCORR_OK;
    DeviceGuard g(c->device);
    cudaDeviceSynchronize();
    delete c;
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_set_output_scale(imgcorr_ctx* c, double offset, double gain) {
    if (!c) return fail(IMGCORR_ERR_INVALID, "null context");
    if (!std::isfinite(offset)) return fail(IMGCORR_ERR_INVALID, "output offset must be finite");
    if (!std::isfinite(gain) || !(gain > 0.0)) return fail(IMGCORR_ERR_INVALID, "output gain must be finite and > 0");
    c->out_scale = OutScale{offset, gain};
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_set_option(imgcorr_ctx* c, int key, int value) {
    if (!c) return fail(IMGCORR_ERR_INVALID, "null context");
    switch (key) {
        case IMGCORR_OPT_K1_VARIANT:
            if (value < 0 || value > 3) return fail(IMGCORR_ERR_INVALID, "k1 variant %d", value);
            c->k1_variant = value;
            return IMGCORR_OK;
        case IMGCORR_OPT_K2_VARIANT:
            if (value < 0 || value > 2) return fail(IMGCORR_ERR_INVALID, "k2 variant %d", value);
            c->k2_variant = value;
            return IMGCORR_OK;
        case IMGCORR_OPT_CHAIN_OVERLAP:
            c->chain_overlap = value ? 1 : 0;
            return IMGCORR_OK;
        case IMGCORR_OPT_K2_COORD_CACHE:
            c->k2_cache_on = value ? 1 : 0;
            if (!value && !c->k2_cache.empty()) {
                DeviceGuard g(c->device);
                cudaDeviceSynchronize();
                c->k2_cache.clear();
            }
            return IMGCORR_OK;
        case IMGCORR_OPT_K3_VARIANT:
            if (value < 0 || value > 2) return fail(IMGCORR_ERR_INVALID, "k3 variant %d", value);
            c->k3_variant = value;
            return IMGCORR_OK;
        case IMGCORR_OPT_PROFILE:
            if (value < 0) return fail(IMGCORR_ERR_INVALID, "profile stride %d", value);
            c->profile = value;
            return IMGCORR_OK;
        case IMGCORR_OPT_CHAIN_GROUP:
            if (value < 1 || value > 64) return fail(IMGCORR_ERR_INVALID, "chain group %d not in [1,64]", value);
            c->chain_group = value;
            return IMGCORR_OK;
        case IMGCORR_OPT_RAW_BIG_ENDIAN:
            c->raw_big_endian = value ? 1 : 0;
            return IMGCORR_OK;
        case IMGCORR_OPT_RAW_FRAME_GAP:
            if (value < 0) return fail(IMGCORR_ERR_INVALID, "frame gap %d", value);
            c->raw_gap = value;
            return IMGCORR_OK;
        case IMGCORR_OPT_K1_SEG_ROWS:
            if (value < 0) return fail(IMGCORR_ERR_INVALID, "seg rows %d", value);
            c->k1_seg_rows = value;
            return IMGCORR_OK;
        case IMGCORR_OPT_HOST_SLOTS:
            if (value < 2 || value > 64) return fail(IMGCORR_ERR_INVALID, "host slots %d not in [2,64]", value);
            if (value != c->host_slots) {
                DeviceGuard g(c->device);
                cudaDeviceSynchronize();
                c->slots.clear();
                c->host_slots = value;
            }
            return IMGCORR_OK;
    }
    return fail(IMGCORR_ERR_INVALID, "unknown option %d", key);
}

extern "C" IMGCORR_API long long imgcorr_launch_count(const imgcorr_ctx* c) { return c ? c->launches : 0; }

static void prof_mark(imgcorr_ctx* c, int which, cudaStream_t st) {
    Event e;
    if (new_event(e, cudaEventDefault) != cudaSuccess) return;
    cudaEventRecord(e.get(), st);
    c->prof_ev[which].push_back(std::move(e));
}

extern "C" IMGCORR_API int imgcorr_profile_read(imgcorr_ctx* c, double out[4]) {
    GUARD(c);
    if (!out) return fail(IMGCORR_ERR_INVALID, "out is null");
    for (int k = 0; k < 2; ++k) {
        double ms = 0.0;
        auto& v = c->prof_ev[k];
        const size_t pairs = v.size() / 2;
        for (size_t i = 0; i < pairs; ++i) {
            float t = 0.f;
            CK(cudaEventSynchronize(v[2 * i + 1].get()));
            CK(cudaEventElapsedTime(&t, v[2 * i].get(), v[2 * i + 1].get()));
            ms += t;
        }
        v.clear();
        out[2 * k] = ms;
        out[2 * k + 1] = c->prof_frames[k];
        c->prof_frames[k] = 0.0;
    }
    return IMGCORR_OK;
}

static bool all_finite(const float* p, size_t n) {
    // |x| <= FLT_MAX fails for NaN and inf; accumulate without branches
    bool ok = true;
    for (size_t i = 0; i < n; ++i) ok &= (fabsf(p[i]) <= 3.402823466e+38f);
    return ok;
}

static int upload_map(imgcorr_ctx* c, DevPtr<float>& slot, const float* src, int on_device, bool* finite,
                      std::vector<float>* host_copy = nullptr) {
    const size_t n = (size_t)c->H * c->W, bytes = n * sizeof(float);
    *finite = true;
    if (!src) {
        if (slot) { CK(cudaDeviceSynchronize()); slot.reset(); }
        return IMGCORR_OK;
    }
    if (!slot) CK(dev_alloc(slot, bytes));
    else CK(cudaDeviceSynchronize());      // launches on other (non-blocking) streams may still read the map being replaced
    CK(cudaMemcpy(slot.get(), src, bytes, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    std::vector<float> tmp;
    const float* h = src;
    if (on_device || host_copy) {
        std::vector<float>& dst = host_copy ? *host_copy : tmp;
        dst.resize(n);
        if (on_device) CK(cudaMemcpy(dst.data(), slot.get(), bytes, cudaMemcpyDeviceToHost));
        else memcpy(dst.data(), src, bytes);
        h = dst.data();
    }
    *finite = all_finite(h, n);
    return IMGCORR_OK;
}

// finiteness and the largest finite magnitude of a host map, read in place
static void scan_map(const float* h, size_t n, bool* finite, double* absmax) {
    bool ok = true;
    float mx = 0.0f;
    for (size_t i = 0; i < n; ++i) {
        const float av = fabsf(h[i]);
        ok &= av <= 3.402823466e+38f;
        if (av <= 3.402823466e+38f && av > mx) mx = av;
    }
    *finite = ok;
    *absmax = mx;
}

extern "C" IMGCORR_API int imgcorr_set_dark(imgcorr_ctx* c, const float* dark, const float* ascent, double exposure_time,
                                int depth_bits, int on_device) {
    GUARD(c);
    if (c->exposures) {                                // the times belong to the model being replaced; queued calls may read them
        CK(cudaDeviceSynchronize());
        c->exposures.reset();
        c->n_exposures = 0;
    }
    if (!dark && ascent) return fail(IMGCORR_ERR_INVALID, "ascent given without offset map");
    if (ascent && (depth_bits < 1 || depth_bits > 62)) return fail(IMGCORR_ERR_INVALID, "depth_bits %d", depth_bits);
    if (ascent && !(exposure_time == exposure_time)) return fail(IMGCORR_ERR_INVALID, "exposure_time is NaN");
    if (!ascent) {
        if (c->linear) {                               // the [2][H][W] block goes; upload_map allocates [H][W]
            CK(cudaDeviceSynchronize());
            c->dark.reset();
            c->linear = false;
        }
        std::vector<float> h;
        int r = upload_map(c, c->dark, dark, on_device, &c->dark_finite, &h);
        if (r) return r;
        c->dark_absmax = 0.0;
        for (float v : h) { const float av = fabsf(v); if (av <= 3.402823466e+38f && av > c->dark_absmax) c->dark_absmax = av; }
        c->exposure = exposure_time;
        c->maxval = 65535.0;
        return IMGCORR_OK;
    }
    // The line model keeps offset and ascent in one [2][H][W] block: the streaming kernel loads both boxes of a stage with
    // one 3-D copy.  A failed upload leaves no dark map.
    const size_t n = (size_t)c->H * c->W, bytes = n * sizeof(float);
    if (c->dark) CK(cudaDeviceSynchronize());          // launches on other streams may still read the map being replaced
    c->dark.reset();
    c->linear = false;
    DevPtr<float> blk;
    CK(dev_alloc(blk, 2 * bytes));
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    CK(cudaMemcpy(blk.get(), dark, bytes, kind));
    CK(cudaMemcpy(blk.get() + n, ascent, bytes, kind));
    if (on_device) {
        std::vector<float> h(2 * n);
        CK(cudaMemcpy(h.data(), blk.get(), 2 * bytes, cudaMemcpyDeviceToHost));
        scan_map(h.data(), n, &c->dark_finite, &c->dark_absmax);
        scan_map(h.data() + n, n, &c->ascent_finite, &c->ascent_absmax);
    } else {
        scan_map(dark, n, &c->dark_finite, &c->dark_absmax);
        scan_map(ascent, n, &c->ascent_finite, &c->ascent_absmax);
    }
    c->dark = std::move(blk);
    c->linear = true;
    c->exposure = exposure_time;
    c->maxval = ldexp(1.0, depth_bits) - 1.0;
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_set_dark_exposures(imgcorr_ctx* c, const double* t, int n) {
    GUARD(c);
    // launches on other (non-blocking) streams may still read the table being replaced or dropped; a failed call leaves
    // no table behind
    if (c->exposures) {
        CK(cudaDeviceSynchronize());
        c->exposures.reset();
        c->n_exposures = 0;
    }
    if (!t) return IMGCORR_OK;
    if (!c->linear) return fail(IMGCORR_ERR_STATE, "per-frame exposure times need the linear dark model (imgcorr_set_dark with ascent)");
    if (n <= 0) return fail(IMGCORR_ERR_INVALID, "n %d", n);
    double mx = 0.0;
    for (int i = 0; i < n; ++i) {
        if (!(t[i] == t[i])) return fail(IMGCORR_ERR_INVALID, "exposure time %d is NaN", i);
        if (fabs(t[i]) > mx) mx = fabs(t[i]);
    }
    DevPtr<double> d;
    CK(dev_alloc(d, (size_t)n * sizeof(double)));
    CK(cudaMemcpy(d.get(), t, (size_t)n * sizeof(double), cudaMemcpyHostToDevice));
    c->exposures = std::move(d);
    c->n_exposures = n;
    c->exposures_absmax = mx;
    return IMGCORR_OK;
}

// the refusal of a call that evaluates the line model over more frames than the per-frame exposure table holds, before
// anything is enqueued
static int check_exposures(const imgcorr_ctx* c, int flags, const void* bg, int n_frames) {
    if (!c->exposures || bg || !(flags & IMGCORR_DO_DARK) || n_frames <= c->n_exposures) return IMGCORR_OK;
    return fail(IMGCORR_ERR_INVALID, "%d frames but the exposure table holds %d times", n_frames, c->n_exposures);
}

extern "C" IMGCORR_API int imgcorr_set_flat(imgcorr_ctx* c, const float* flat, int on_device) {
    GUARD(c);
    std::vector<float> h;
    int r = upload_map(c, c->flat, flat, on_device, &c->flat_finite, &h);
    if (r) return r;
    if (!flat) {
        c->flat_nz.reset();                        // upload_map synchronised the device before it dropped the flat
        return IMGCORR_OK;
    }
    // zero-free copy for the streaming kernel + the smallest non-zero magnitude (overflow proof)
    double mn = 3.5e38;
    for (float& v : h) {
        if (v == 0.0f) v = 1.0f;
        const float av = fabsf(v);
        if (av <= 3.402823466e+38f && av < mn) mn = av;
    }
    c->flat_absmin = mn;
    if (!c->flat_nz) CK(dev_alloc(c->flat_nz, h.size() * sizeof(float)));
    else CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(c->flat_nz.get(), h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_set_lens_model(imgcorr_ctx* c, const double K[9], const double* dist, int n_dist, const double P[9]) {
    if (!c) return fail(IMGCORR_ERR_INVALID, "null context");
    if (!K) { c->has_lens = false; return IMGCORR_OK; }
    if (!dist || !P) return fail(IMGCORR_ERR_INVALID, "dist / P is null");
    if (n_dist != 4 && n_dist != 5 && n_dist != 8 && n_dist != 12 && n_dist != 14)
        return fail(IMGCORR_ERR_INVALID, "%d distortion coefficients (4, 5, 8, 12 or 14)", n_dist);
    // K, the coefficients zero-padded to 14, P and the count: two lenses that differ in any of them differ here
    double in[33] = {0};
    memcpy(in, K, 9 * sizeof(double)); memcpy(in + 9, dist, n_dist * sizeof(double)); memcpy(in + 23, P, 9 * sizeof(double));
    in[32] = n_dist;
    // the Python mirror sets the lens on every correct() call (the reference builds a new LensDistortion per call,
    // camera/CameraCalibration.py:565-568): the same lens again must not drop K2's geometry choice and coordinate cache
    if (c->has_lens && c->lens_dev && memcmp(in, c->lens_in, sizeof in) == 0) return IMGCORR_OK;
    LensConst L;
    if (!make_lens_const(K, dist, n_dist, P, L)) return fail(IMGCORR_ERR_INVALID, "new camera matrix P is singular");
    LensExt X;
    const bool ext = make_lens_ext(dist, n_dist, X);
    double pack[LP_EXT_COUNT] = {0};
    pack[LP_K1] = L.k1; pack[LP_K2] = L.k2; pack[LP_K3] = L.k3; pack[LP_P1] = L.p1; pack[LP_P2] = L.p2;
    pack[LP_P1X2] = L.p1x2; pack[LP_P2X2] = L.p2x2; pack[LP_FX] = L.fx; pack[LP_FY] = L.fy; pack[LP_CX] = L.cx;
    pack[LP_CY] = L.cy; pack[LP_IR0] = L.ir[0]; pack[LP_IR2] = L.ir[2]; pack[LP_IR4] = L.ir[4]; pack[LP_IR5] = L.ir[5];
    memcpy(pack + LP_COUNT, &X, sizeof X);
    {
        DeviceGuard g(c->device);
        if (!g.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
        if (!c->lens_dev) CK(dev_alloc(c->lens_dev, sizeof pack));
        CK(cudaMemcpy(c->lens_dev.get(), pack, sizeof pack, cudaMemcpyHostToDevice));
    }
    c->lens = L;
    c->lens_x = X;
    c->lens_ext = ext;
    c->has_lens = true;
    memcpy(c->lens_in, in, sizeof in);
    c->k2_geom.clear();
    if (!c->k2_cache.empty()) {
        DeviceGuard g(c->device);
        cudaDeviceSynchronize();                       // launches that still read the old lens' coordinates
        c->k2_cache.clear();
    }
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_set_lens(imgcorr_ctx* c, const double K[9], const double dist[5], const double P[9]) {
    return imgcorr_set_lens_model(c, K, dist, 5, P);
}

// bg: per-frame backgrounds [n][H][W] of bg_dtype in place of the dark map (checked by check_bg), or null.  first: the
// index of raw's first frame in the caller's call, which picks its per-frame exposure times (checked by check_exposures)
static int fill_k1(imgcorr_ctx* c, K1Args& a, const void* raw, int raw_dtype, void* out, uint8_t* mask, int n, double thr,
                   int ksize, int cond, int flags, const void* bg = nullptr, int bg_dtype = DT_F32, int first = 0) {
    if (!raw || !out) return fail(IMGCORR_ERR_INVALID, "null image pointer");
    if (n < 0) return fail(IMGCORR_ERR_INVALID, "n_frames %d", n);
    if (!(thr > 0.0)) ksize = 0;                      // also NaN
    if (ksize != 0 && ksize != 3 && ksize != 5) return fail(IMGCORR_ERR_INVALID, "ksize %d (0, 3 or 5)", ksize);
    if (cond != IMGCORR_COND_GT && cond != IMGCORR_COND_LT) return fail(IMGCORR_ERR_INVALID, "cond %d", cond);
    a = K1Args{};
    a.raw = raw; a.out = out; a.mask = ksize ? mask : nullptr;
    a.q = OutScale{0.0, 1.0};                         // saturate_cast; chain calls with integer output set the context's scale
    a.H = c->H; a.W = c->W; a.n_frames = n; a.ksize = ksize;
    a.raw_swap = (c->raw_big_endian && raw_dtype == DT_U16) ? 1 : 0;
    a.raw_gap = c->raw_gap;
    if (c->raw_big_endian && raw_dtype != DT_U16 && raw_dtype != DT_U8)
        return fail(IMGCORR_ERR_INVALID, "big-endian ingest is implemented for uint16 frames");
    if (c->raw_gap % (long long)dtype_size(raw_dtype)) return fail(IMGCORR_ERR_INVALID, "frame gap must be a multiple of the sample size");
    int f = 0;
    if (bg) {
        f |= FLAG_DARK; a.bg = bg; a.bg_dtype = bg_dtype;
    } else if ((flags & IMGCORR_DO_DARK) && c->dark) {
        f |= FLAG_DARK; a.dark = c->dark.get();
        if (c->linear) {
            f |= FLAG_DARK_LINEAR; a.ascent = c->dark.get() + (size_t)c->H * c->W;
            if (c->exposures) a.exposures = c->exposures.get() + first;
        }
    }
    if ((flags & IMGCORR_DO_FLAT) && c->flat) { f |= FLAG_FLAT; a.flat = c->flat.get(); }
    if (flags & IMGCORR_DO_NAN_TO_NUM) f |= FLAG_NAN_TO_NUM;
    a.pw.flags = f; a.pw.exposure_time = c->exposure; a.pw.max_value = c->maxval;
    a.maps_finite = ((!a.dark || c->dark_finite) && (!a.ascent || c->ascent_finite) && (!a.flat || c->flat_finite)) ? 1 : 0;
    a.flat_nz = a.flat ? c->flat_nz.get() : nullptr;
    if (!c->dump) CK(dev_alloc(c->dump, (size_t)4 << 20));
    a.dump = c->dump.get();
    // integer frames: |raw - dark| <= raw_max + max|dark|; divided by min|flat| it must stay below FLT_MAX.  Backgrounds of
    // the raw integer dtype: |raw - bg| <= raw_max.  Float32 backgrounds are not checked at upload: no proof
    // The line model: |bg| <= max|offset| + max|ascent| * max|t| over the scalar or the table in use, a finite bound or none.
    a.no_overflow = 0;
    double bg_max = a.dark ? c->dark_absmax : 0.0;
    if (a.ascent) {
        const double tmax = a.exposures ? c->exposures_absmax : fabs(c->exposure);
        bg_max = bg_max + c->ascent_absmax * tmax;
        // the streaming kernel's unchecked division needs |raw - bg| well inside float64's range: |bg| <= FLT_MAX.  A larger
        // bound (an infinite time, inf * 0) is no proof: the checked arithmetic
        if (!(bg_max <= 3.0e38)) a.maps_finite = 0;
    }
    if (a.maps_finite && (raw_dtype == DT_U8 || raw_dtype == DT_U16) && (!bg || bg_dtype == raw_dtype)) {
        const double num = (raw_dtype == DT_U8 ? 255.0 : 65535.0) + bg_max;
        const double den = a.flat ? c->flat_absmin : 1.0;
        a.no_overflow = (num / den < 3.0e38) ? 1 : 0;
    }
    a.pred = make_predicate(thr, cond == IMGCORR_COND_LT ? COND_LT : COND_GT);
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_pointwise_median(imgcorr_ctx* c, const void* raw_dev, int raw_dtype, void* out_dev, int out_dtype,
                                        uint8_t* mask_dev, int n_frames, double threshold, int ksize, int cond,
                                        int flags, void* stream) {
    GUARD(c);
    if ((out_dtype == DT_U8 || out_dtype == DT_U16) && out_dtype != raw_dtype)        // integer output keeps the input dtype here
        return fail(IMGCORR_ERR_INVALID, "unsupported dtype pair raw=%d out=%d", raw_dtype, out_dtype);
    K1Args a;
    if (int r = check_exposures(c, flags, nullptr, n_frames)) return r;
    int r = fill_k1(c, a, raw_dev, raw_dtype, out_dev, mask_dev, n_frames, threshold, ksize, cond, flags);
    if (r) return r;
    a.out_streaming = 1;
    int l = 0;
    cudaError_t e = launch_k1(a, raw_dtype, out_dtype, c->k1_variant, c->sm_count, c->k1_seg_rows, (cudaStream_t)stream, &l);
    return launched(c, l, e, "K1 launch", "requested K1 variant is not eligible for this shape / dtype / alignment",
                    "unsupported dtype pair raw=%d out=%d", raw_dtype, out_dtype);
}

static int run_k2(imgcorr_ctx* c, const void* src, int sdt, void* dst, int ddt, int n, const float* mapx,
                  const float* mapy, double border, int x0, int y0, int ow, int oh, OutScale q, cudaStream_t st) {
    if (!src || !dst) return fail(IMGCORR_ERR_INVALID, "null image pointer");
    if (n < 0) return fail(IMGCORR_ERR_INVALID, "n_frames %d", n);
    if (!mapx && !c->has_lens) return fail(IMGCORR_ERR_STATE, "no lens set");
    if (x0 < 0 || y0 < 0 || ow < 0 || oh < 0 || x0 + ow > c->W || y0 + oh > c->H)
        return fail(IMGCORR_ERR_INVALID, "output window (%d,%d,%d,%d) outside %dx%d frame", x0, y0, ow, oh, c->W, c->H);
    K2Args a{};
    a.src = src; a.dst = dst; a.mapx = mapx; a.mapy = mapy;
    a.H = c->H; a.W = c->W; a.n_frames = n;
    a.x0 = x0; a.y0 = y0; a.ow = ow; a.oh = oh;
    a.border = border_for_dtype(sdt == DT_U8, sdt == DT_U16, border);
    a.lens = c->lens;
    a.lens_dev = c->lens_dev.get();
    a.lens_ext = c->lens_ext ? 1 : 0;
    a.sm_count = c->sm_count;
    a.q = q;
    if (!c->k2_wtab) {
        std::vector<float4> t(32 * 32);
        for (int fy = 0; fy < 32; ++fy)
            for (int fx = 0; fx < 32; ++fx) {
                float4 w;
                bilinear_weights(fx, fy, w.x, w.y, w.z, w.w);
                t[fy * 32 + fx] = w;
            }
        DevPtr<float4> d;
        CK(dev_alloc(d, t.size() * sizeof(float4)));
        CK(cudaMemcpy(d.get(), t.data(), t.size() * sizeof(float4), cudaMemcpyHostToDevice));
        c->k2_wtab = std::move(d);
    }
    a.wtab = c->k2_wtab.get();
    a.geometry = 0;
    if (!mapx) {
        bool found = false;
        const int gesz = (int)dtype_size(sdt) > 4 ? 4 : (int)dtype_size(sdt);
        for (const auto& k : c->k2_geom)
            if (k.x0 == x0 && k.y0 == y0 && k.ow == ow && k.oh == oh && k.esz == gesz) { a.geometry = k.g; found = true; break; }
        if (!found) {
            a.geometry = k2_pick_geometry(c->lens, c->lens_ext ? &c->lens_x : nullptr, c->H, c->W, x0, y0, ow, oh, gesz);
            if (c->k2_geom.size() > 64) c->k2_geom.clear();
            c->k2_geom.push_back({x0, y0, ow, oh, gesz, a.geometry});
        }
    }
    // coordinate cache (tiled variant, analytic map): the first launch for this lens / window writes it, later ones read it
    imgcorr_ctx::K2Cache fresh{};                      // the entry this launch writes; it joins the cache once its event is recorded
    // Only launches of one or two frames use it: a batch amortises the analytic evaluation over its frames and the
    // per-tile kernel then streams faster (19 vs 33 us per 4096x3000 frame) than the cached one (49 vs 65 us for one frame).
    if (!mapx && c->k2_cache_on && n > 0 && n <= 2 && ow > 0 && oh > 0 && k2_will_tile(a, sdt, ddt, c->k2_variant)) {
        const int esz = (int)dtype_size(sdt);
        imgcorr_ctx::K2Cache* hit = nullptr;
        for (auto& k : c->k2_cache)
            if (k.x0 == x0 && k.y0 == y0 && k.ow == ow && k.oh == oh && k.g == a.geometry && k.esz == esz) { hit = &k; break; }
        if (hit) {
            if (hit->st != st) CK(cudaStreamWaitEvent(st, hit->ev.get(), 0));       // written on another stream
            hit->stamp = ++c->k2_stamp;
            a.cpack = hit->pack.get(); a.chdr = hit->hdr.get();
        } else {
            if (c->k2_cache.size() >= 2) {             // keep at most two windows (keep_size True / False): drop the older one
                size_t old = c->k2_cache[0].stamp < c->k2_cache[1].stamp ? 0 : 1;
                CK(cudaDeviceSynchronize());
                c->k2_cache.erase(c->k2_cache.begin() + old);
            }
            size_t words = 0, tiles = 0;
            k2_cache_size(a.geometry, ow, oh, &words, &tiles);
            imgcorr_ctx::K2Cache k{x0, y0, ow, oh, a.geometry, esz, {}, {}, {}, st, ++c->k2_stamp};
            if (dev_alloc(k.pack, words * sizeof(unsigned)) == cudaSuccess && dev_alloc(k.hdr, tiles * sizeof(int2)) == cudaSuccess &&
                new_event(k.ev) == cudaSuccess) {
                fresh = std::move(k);
                a.cpack_w = fresh.pack.get(); a.chdr_w = fresh.hdr.get();
            } else {                                   // no memory for the cache: compute every time
                cudaGetLastError();
            }
        }
    }
    int l = 0;
    cudaError_t e = launch_k2(a, sdt, ddt, c->k2_variant, st, &l);
    if (fresh.ev) {                                    // never leave a half-written cache behind
        if (e == cudaSuccess) e = cudaEventRecord(fresh.ev.get(), st);
        if (e == cudaSuccess) c->k2_cache.push_back(std::move(fresh));
        else cudaDeviceSynchronize();                  // a queued kernel may still write the buffers `fresh` frees on return
    }
    return launched(c, l, e, "K2 launch", "requested K2 variant is not eligible for this dtype / alignment",
                    "unsupported dtype pair src=%d dst=%d", sdt, ddt);
}

extern "C" IMGCORR_API int imgcorr_undistort(imgcorr_ctx* c, const void* src_dev, int src_dtype, void* dst_dev, int dst_dtype,
                                 int n_frames, double border_value, int x0, int y0, int ow, int oh, void* stream) {
    GUARD(c);
    if (src_dtype == DT_F32 && (dst_dtype == DT_U8 || dst_dtype == DT_U16))
        return fail(IMGCORR_ERR_INVALID, "unsupported dtype pair src=%d dst=%d", src_dtype, dst_dtype);
    return run_k2(c, src_dev, src_dtype, dst_dev, dst_dtype, n_frames, nullptr, nullptr, border_value, x0, y0, ow, oh,
                  OutScale{0.0, 1.0}, (cudaStream_t)stream);
}

extern "C" IMGCORR_API int imgcorr_remap(imgcorr_ctx* c, const void* src_dev, int src_dtype, void* dst_dev, int dst_dtype,
                             int n_frames, const float* mapx_dev, const float* mapy_dev, double border_value,
                             void* stream) {
    GUARD(c);
    if (!mapx_dev || !mapy_dev) return fail(IMGCORR_ERR_INVALID, "null map pointer");
    if (src_dtype == DT_F32 && (dst_dtype == DT_U8 || dst_dtype == DT_U16))
        return fail(IMGCORR_ERR_INVALID, "unsupported dtype pair src=%d dst=%d", src_dtype, dst_dtype);
    return run_k2(c, src_dev, src_dtype, dst_dev, dst_dtype, n_frames, mapx_dev, mapy_dev, border_value, 0, 0, c->W,
                  c->H, OutScale{0.0, 1.0}, (cudaStream_t)stream);
}

extern "C" IMGCORR_API int imgcorr_undistort_maps(imgcorr_ctx* c, float* mapx_dev, float* mapy_dev, void* stream) {
    GUARD(c);
    if (!c->has_lens) return fail(IMGCORR_ERR_STATE, "no lens set");
    if (!mapx_dev || !mapy_dev) return fail(IMGCORR_ERR_INVALID, "null map pointer");
    int l = 0;
    cudaError_t e = launch_write_maps(c->lens, c->lens_ext ? &c->lens_x : nullptr, mapx_dev, mapy_dev, c->H, c->W, (cudaStream_t)stream, &l);
    return launched(c, l, e, "map kernel launch");
}

// ---- K3 -------------------------------------------------------------------------------------
static int run_k3(imgcorr_ctx* c, const void* src_dev, int dtype, int src_h, int src_w, void* dst_dev, int dst_dtype, int dst_h,
                  int dst_w, int n_frames, const double M[9], const WarpConst* wcs, int interpolation, int inverse_map,
                  double border_value, OutScale q, cudaStream_t st);

extern "C" IMGCORR_API int imgcorr_warp_perspective(imgcorr_ctx* c, const void* src_dev, int dtype, int src_h, int src_w,
                                        void* dst_dev, int dst_h, int dst_w, int n_frames, const double M[9],
                                        int interpolation, int inverse_map, double border_value, void* stream) {
    GUARD(c);
    if (!src_dev || !dst_dev || !M) return fail(IMGCORR_ERR_INVALID, "null pointer");
    if (dtype < DT_U8 || dtype > DT_F64) return fail(IMGCORR_ERR_INVALID, "bad dtype %d", dtype);
    if (interpolation != IMGCORR_INTER_LANCZOS4 && interpolation != IMGCORR_INTER_CUBIC)
        return fail(IMGCORR_ERR_INVALID, "interpolation must be IMGCORR_INTER_LANCZOS4 or IMGCORR_INTER_CUBIC");
    if (src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0 || src_h > 32767 || src_w > 32767 || dst_h > 32767 || dst_w > 32767)
        return fail(IMGCORR_ERR_INVALID, "bad frame shape (%d x %d -> %d x %d)", src_h, src_w, dst_h, dst_w);
    if (n_frames < 0) return fail(IMGCORR_ERR_INVALID, "n_frames < 0");
    return run_k3(c, src_dev, dtype, src_h, src_w, dst_dev, dtype, dst_h, dst_w, n_frames, M, nullptr, interpolation, inverse_map,
                  border_value, OutScale{0.0, 1.0}, (cudaStream_t)stream);
}

// K3 on validated arguments; the coefficient tables are built on first use.  dst_dtype is dtype, or U16 / U8 for a float32
// source (the chain's integer output: float32 warp, then quantise with q).  wcs: a device table of n_frames inverted
// matrices (the chain's per-frame stage), used instead of M
static int run_k3(imgcorr_ctx* c, const void* src_dev, int dtype, int src_h, int src_w, void* dst_dev, int dst_dtype, int dst_h,
                  int dst_w, int n_frames, const double M[9], const WarpConst* wcs, int interpolation, int inverse_map,
                  double border_value, OutScale q, cudaStream_t st) {
    if (!c->warp_tab) {
        float h[32 * 8 + 32 * 4];
        warp_lanczos4_table(h);
        warp_cubic_table(h + 32 * 8);
        DevPtr<float> d;
        CK(dev_alloc(d, sizeof(h)));
        CK(cudaMemcpy(d.get(), h, sizeof(h), cudaMemcpyHostToDevice));
        c->warp_tab = std::move(d);
    }
    const int lz = interpolation == IMGCORR_INTER_LANCZOS4;
    if (dtype == DT_U8 && !c->warp_itab[lz]) {
        // OpenCV's fixed-point weight table for uint8 images, built on the host once per interpolation
        const int nn = lz ? 8 : 4;
        std::vector<float> t(32 * 8);
        if (lz) warp_lanczos4_table(t.data()); else warp_cubic_table(t.data());
        std::vector<int16_t> it((size_t)32 * 32 * nn * nn);
        warp_fixed_table(t.data(), nn, it.data());
        DevPtr<int16_t> d;
        CK(dev_alloc(d, it.size() * sizeof(int16_t)));
        CK(cudaMemcpy(d.get(), it.data(), it.size() * sizeof(int16_t), cudaMemcpyHostToDevice));
        c->warp_itab[lz] = std::move(d);
    }
    K3Args a;
    a.itab = dtype == DT_U8 ? c->warp_itab[lz].get() : nullptr;
    a.src = src_dev;
    a.dst = dst_dev;
    a.H = src_h;
    a.W = src_w;
    a.dh = dst_h;
    a.dw = dst_w;
    a.n_frames = n_frames;
    a.dst_dtype = dst_dtype;
    a.q = q;
    a.border = border_for_dtype(dtype == DT_U8, dtype == DT_U16, border_value);
    a.wc = wcs ? WarpConst{} : make_warp_const(M, inverse_map, dst_w, dst_h);
    a.wcs = wcs;
    a.tab = interpolation == IMGCORR_INTER_LANCZOS4 ? c->warp_tab.get() : c->warp_tab.get() + 32 * 8;
    int l = 0;
    cudaError_t e = launch_k3(a, dtype, interpolation, c->k3_variant, st, &l);
    return launched(c, l, e, "K3 launch", "the requested K3 variant is not eligible for this call");
}

extern "C" IMGCORR_API int imgcorr_divide_f64(imgcorr_ctx* c, const void* src_dev, int src_dtype, const double* divisor_dev,
                                  double* dst_dev, size_t pixels_per_frame, int n_frames, void* stream) {
    GUARD(c);
    if (!src_dev || !divisor_dev || !dst_dev) return fail(IMGCORR_ERR_INVALID, "null pointer");
    if (src_dtype < DT_U8 || src_dtype > DT_F64) return fail(IMGCORR_ERR_INVALID, "bad dtype %d", src_dtype);
    if (n_frames < 0) return fail(IMGCORR_ERR_INVALID, "n_frames < 0");
    int l = 0;
    cudaError_t e = launch_k3_divide(src_dev, src_dtype, divisor_dev, dst_dev, pixels_per_frame, n_frames, c->sm_count,
                                     (cudaStream_t)stream, &l);
    return launched(c, l, e, "divide kernel launch");
}

// ---- K4 -------------------------------------------------------------------------------------
static int ste_average_impl(imgcorr_ctx* c, const void* frames_dev, int dtype, int n_frames, double* avg_dev,
                            uint8_t* mask_dev, const double nlf[3], double n_std, const double* thr_dev, void* stream);

extern "C" IMGCORR_API int imgcorr_ste_average(imgcorr_ctx* c, const void* frames_dev, int dtype, int n_frames, double* avg_dev,
                                   uint8_t* mask_dev, const double nlf[3], double n_std, void* stream) {
    GUARD(c);
    if (!nlf) return fail(IMGCORR_ERR_INVALID, "null pointer");
    return ste_average_impl(c, frames_dev, dtype, n_frames, avg_dev, mask_dev, nlf, n_std, nullptr, stream);
}

extern "C" IMGCORR_API int imgcorr_ste_average_thr(imgcorr_ctx* c, const void* frames_dev, int dtype, int n_frames, double* avg_dev,
                                       uint8_t* mask_dev, const double* threshold_dev, void* stream) {
    GUARD(c);
    if (!threshold_dev) return fail(IMGCORR_ERR_INVALID, "null pointer");
    const double none[3] = {0.0, 0.0, 0.0};
    return ste_average_impl(c, frames_dev, dtype, n_frames, avg_dev, mask_dev, none, 1.0, threshold_dev, stream);
}

static int ste_average_impl(imgcorr_ctx* c, const void* frames_dev, int dtype, int n_frames, double* avg_dev,
                            uint8_t* mask_dev, const double nlf[3], double n_std, const double* thr_dev, void* stream) {
    if (!frames_dev || !avg_dev || !nlf) return fail(IMGCORR_ERR_INVALID, "null pointer");
    if (dtype < DT_U8 || dtype > DT_F64) return fail(IMGCORR_ERR_INVALID, "bad dtype %d", dtype);
    if (n_frames < 2) return fail(IMGCORR_ERR_INVALID, "single-time-effect removal needs at least 2 images (got %d)", n_frames);
    const size_t npx = (size_t)c->H * c->W, part = round256(npx * sizeof(double));
    cudaStream_t st = (cudaStream_t)stream;
    CK(c->ste_scratch.acquire(2 * part + npx * sizeof(int), st));    // [running average][thresholds][counts]
    SharedScratch::Guard release{c->ste_scratch, st};
    char* const s = c->ste_scratch.buf.get();
    // n_frames - 1 launches; ping-pong so that the last one writes avg_dev
    double* buf[2] = {avg_dev, (double*)s};
    int cur = (n_frames - 2) % 2;                  // buffer the FIRST launch writes
    K4Args a;
    a.H = c->H;
    a.W = c->W;
    a.thr = (double*)(s + part);
    a.thr_in = thr_dev;
    a.n = (int*)(s + 2 * part);
    a.mask = mask_dev;
    a.sc.minY = nlf[0];
    a.sc.ax = nlf[1];
    a.sc.ay = nlf[2];
    a.sc.nstd = n_std;
    const char* f = (const char*)frames_dev;
    const size_t fb = npx * dtype_size(dtype);
    int l = 0;
    cudaError_t e = cudaSuccess;
    for (int k = 1; k < n_frames && e == cudaSuccess; ++k) {
        a.img = k == 1 ? f : f + k * fb;
        a.img2 = k == 1 ? f + fb : nullptr;
        a.avg_in = buf[cur ^ 1];
        a.avg_out = buf[cur];
        e = launch_k4(a, dtype, st, &l);
        cur ^= 1;
    }
    return launched(c, l, e, "K4 launch");
}

// ---- the chain --------------------------------------------------------------------------------
extern "C" IMGCORR_API int imgcorr_set_perspective(imgcorr_ctx* c, const double M[9], int dst_h, int dst_w, double border_value,
                                       const double* tilt_factor, int tilt_h, int tilt_w, int on_device) {
    GUARD(c);
    imgcorr_ctx::Perspective& p = c->persp;
    // a failed call leaves no stage behind: a chain call with the bit then fails with IMGCORR_ERR_STATE instead of
    // writing frames of the previous destination shape into buffers sized for another
    p.on = false;
    if (M) {
        if (dst_h <= 0 || dst_w <= 0 || dst_h > 32767 || dst_w > 32767)
            return fail(IMGCORR_ERR_INVALID, "bad destination shape %d x %d", dst_h, dst_w);
        if (tilt_factor && (tilt_h <= 0 || tilt_w <= 0))
            return fail(IMGCORR_ERR_INVALID, "bad tilt factor shape %d x %d", tilt_h, tilt_w);
    }
    const size_t tilt_bytes = (M && tilt_factor) ? (size_t)tilt_h * tilt_w * sizeof(double) : 0;
    // launches on other (non-blocking) streams may still read the tilt factor or the per-frame table being replaced or dropped
    if (p.tilt || p.table) {
        CK(cudaDeviceSynchronize());
        if (tilt_bytes != (size_t)p.th * p.tw * sizeof(double)) { p.tilt.reset(); p.th = p.tw = 0; }
        p.table.reset();
        p.n_table = 0;
    }
    if (!M) return IMGCORR_OK;
    if (tilt_bytes) {
        if (!p.tilt) CK(dev_alloc(p.tilt, tilt_bytes));
        p.th = tilt_h;
        p.tw = tilt_w;
        CK(cudaMemcpy(p.tilt.get(), tilt_factor, tilt_bytes, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    } else {
        p.tilt.reset();
        p.th = p.tw = 0;
    }
    memcpy(p.M, M, sizeof p.M);
    p.dh = dst_h;
    p.dw = dst_w;
    p.border = border_value;
    p.on = true;
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_set_perspective_frames(imgcorr_ctx* c, const double* M, int n_matrices, int dst_h, int dst_w,
                                              double border_value) {
    GUARD(c);
    imgcorr_ctx::Perspective& p = c->persp;
    p.on = false;                                      // as imgcorr_set_perspective: a failed call leaves no stage behind
    if (M) {
        if (n_matrices <= 0) return fail(IMGCORR_ERR_INVALID, "n_matrices %d", n_matrices);
        if (dst_h <= 0 || dst_w <= 0 || dst_h > 32767 || dst_w > 32767)
            return fail(IMGCORR_ERR_INVALID, "bad destination shape %d x %d", dst_h, dst_w);
    }
    // launches on other (non-blocking) streams may still read the tilt factor or the table being replaced or dropped
    if (p.tilt || p.table) {
        CK(cudaDeviceSynchronize());
        p.tilt.reset();
        p.th = p.tw = 0;
        if (!M || p.n_table != n_matrices) { p.table.reset(); p.n_table = 0; }
    }
    if (!M) return IMGCORR_OK;
    std::vector<WarpConst> h((size_t)n_matrices);
    for (int i = 0; i < n_matrices; ++i) h[i] = make_warp_const(M + 9 * (size_t)i, 0, dst_w, dst_h);
    if (!p.table) {
        CK(dev_alloc(p.table, h.size() * sizeof(WarpConst)));
        p.n_table = n_matrices;
    }
    CK(cudaMemcpy(p.table.get(), h.data(), h.size() * sizeof(WarpConst), cudaMemcpyHostToDevice));
    p.dh = dst_h;
    p.dw = dst_w;
    p.border = border_value;
    p.on = true;
    return IMGCORR_OK;
}

// the refusals of a chain call with IMGCORR_DO_PERSPECTIVE whose chain frame is [oh][ow], before anything is enqueued
static int check_perspective(const imgcorr_ctx* c, int out_dtype, int ow, int oh, int n_frames) {
    const imgcorr_ctx::Perspective& p = c->persp;
    if (!p.on) return fail(IMGCORR_ERR_STATE, "perspective requested but no perspective set");
    if (ow > 32767 || oh > 32767) return fail(IMGCORR_ERR_INVALID, "perspective source %d x %d exceeds 32767 per side", oh, ow);
    if (p.table && n_frames > p.n_table)
        return fail(IMGCORR_ERR_INVALID, "%d frames but the perspective stage holds %d matrices", n_frames, p.n_table);
    if (!p.tilt) return IMGCORR_OK;
    if (out_dtype != DT_F64)
        return fail(IMGCORR_ERR_INVALID, "a tilt factor needs out_dtype F64: the division and the warp are computed in float64");
    if (p.th != oh || p.tw != ow)
        return fail(IMGCORR_ERR_INVALID, "tilt factor %d x %d does not match the chain frame %d x %d", p.th, p.tw, oh, ow);
    return IMGCORR_OK;
}

// one frame (or a group of frames) through K1 -> [K2] -> [tilt division] -> [K3] on `st`; `persp` was checked by
// check_perspective.  `first`: the index of raw's first frame in the caller's call (chunks of the host pipeline start
// later), which picks the matrices of a per-frame perspective table.
// Integer output (U16 / U8) is the float32 chain with the quantiser fused into the last kernel's store: K1 without a lens or
// perspective stage, K2 with a lens, K3 with the stage (which warps the float32 chain frame).
// `bg`: the call's per-frame backgrounds from raw's first frame on (dense, bg_dtype; checked by check_bg), or null.
// `first` also picks the frames' entries of a per-frame exposure table (checked by check_exposures).
static int chain_frames(imgcorr_ctx* c, const void* raw, int raw_dtype, void* out, int out_dtype, int n, double thr,
                        int ksize, int flags, bool lens, bool persp, double border, int x0, int y0, int ow, int oh,
                        cudaStream_t st, int first, const void* bg, int bg_dtype) {
    if (out_dtype < DT_U8 || out_dtype > DT_F64) return fail(IMGCORR_ERR_INVALID, "out_dtype must be U8, U16, F32 or F64");
    const bool quant = out_dtype == DT_U8 || out_dtype == DT_U16;
    const int frame_dtype = quant ? DT_F32 : out_dtype;    // the chain frame: what K2 (or K1) returns before the stage
    if (raw_dtype == DT_F64) return fail(IMGCORR_ERR_INVALID, "float64 frames: convert to float32 first (the chain computes in float32)");
    const size_t npx = (size_t)c->H * c->W;
    const size_t raw_stride = npx * dtype_size(raw_dtype) + (size_t)c->raw_gap;
    if (!lens && (x0 != 0 || y0 != 0 || ow != c->W || oh != c->H))
        return fail(IMGCORR_ERR_INVALID, "output window without a lens");
    if (!lens && !persp) {                             // K1 alone: one launch for the whole batch, no scratch
        K1Args a;
        int r = fill_k1(c, a, raw, raw_dtype, out, nullptr, n, thr, ksize, IMGCORR_COND_GT, flags, bg, bg_dtype, first);
        if (r) return r;
        if (quant) a.q = c->out_scale;
        int l = 0;
        cudaError_t e = launch_k1(a, raw_dtype, out_dtype, c->k1_variant, c->sm_count, c->k1_seg_rows, st, &l);
        return launched(c, l, e, "K1 launch");
    }
    // K1 -> [K2] -> [tilt division] -> [K3] in groups of `chain_group` frames.  With a lens, the K1 output of a group stays
    // in two alternating halves of the chain scratch (L2-resident for small groups) and K2 evaluates each pixel's map once
    // per group.  With the perspective stage, the frames the call returns without it (K2's window, or K1's output) go to a
    // third part, the warp source, and K3 writes `out`.
    const int grp = c->chain_group < n ? c->chain_group : (n > 0 ? n : 1);
    const size_t half = lens ? round256(npx * sizeof(float) * grp) : 0;
    const size_t src_px = (size_t)ow * oh;              // pixels of a chain frame, the warp source
    const size_t src_bytes = persp ? src_px * dtype_size(frame_dtype) * grp : 0;
    // the wait for another stream's last use precedes ev_entry, so the overlap stream inherits it
    CK(c->chain_scratch.acquire(2 * half + src_bytes, st));
    SharedScratch::Guard release{c->chain_scratch, st};    // every launch of this call is ordered before the end of `st`
    char* const scratch = c->chain_scratch.buf.get();
    float* const mids[2] = {(float*)scratch, (float*)(scratch + half)};
    void* const wsrc = scratch + 2 * half;
    const imgcorr_ctx::Perspective& p = c->persp;
    const size_t out_stride = (persp ? (size_t)p.dw * p.dh : src_px) * dtype_size(out_dtype);
    // Overlap mode (with a lens): K1 of group g+1 runs on an internal high-priority stream while K2 of group g runs on the
    // caller's stream, so that K2's blocks fill the SM slots K1's last, partially filled wave leaves idle (and vice versa).
    // The two halves of the scratch are handed back and forth with events; every K2, division and K3 stays on the caller's
    // stream, so the call is stream-ordered as before.  A profiled group (IMGCORR_OPT_PROFILE) runs unoverlapped so that
    // its brackets time the kernel alone.
    const bool overlap = lens && c->chain_overlap && n > grp;
    imgcorr_ctx::ChainOverlap& ov = c->ov;
    cudaStream_t s1 = st;
    if (overlap) {
        if (!ov.st) {
            int lo = 0, hi = 0;
            CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            imgcorr_ctx::ChainOverlap o;
            CK(new_stream(o.st, hi));
            for (int i = 0; i < 2; ++i) {
                CK(new_event(o.k1[i]));
                CK(new_event(o.k2[i]));
            }
            CK(new_event(o.entry));
            ov = std::move(o);
        }
        s1 = ov.st.get();
        CK(cudaEventRecord(ov.entry.get(), st));      // K1 must not start before the caller's earlier work on `st`
        CK(cudaStreamWaitEvent(s1, ov.entry.get(), 0));
    }
    int gi = 0;
    bool exclusive_next = false;
    for (int f = 0; f < n; f += grp, ++gi) {
        const int nf = n - f < grp ? n - f : grp;
        float* mid = mids[gi & 1];
        void* const frames = persp ? wsrc : (char*)out + f * out_stride;     // what the call returns without the stage
        const bool prof = lens && c->profile > 0 && (c->chain_groups_seen++ % c->profile) == 0;
        if (prof) { c->prof_frames[0] += nf; c->prof_frames[1] += nf; }
        if (overlap) {
            // this half was last read by K2 of group gi-2; a profiled group (or the one after it) also waits for gi-1
            if (gi >= 2) CK(cudaStreamWaitEvent(s1, ov.k2[gi & 1].get(), 0));
            if ((prof || exclusive_next) && gi >= 1) CK(cudaStreamWaitEvent(s1, ov.k2[(gi - 1) & 1].get(), 0));
            exclusive_next = prof;
        }
        K1Args a;
        int r = fill_k1(c, a, (const char*)raw + f * raw_stride, raw_dtype, lens ? (void*)mid : frames, nullptr, nf, thr, ksize,
                        IMGCORR_COND_GT, flags, bg ? (const char*)bg + f * npx * dtype_size(bg_dtype) : nullptr, bg_dtype, first + f);
        if (r) return r;
        int l = 0;
        if (prof) prof_mark(c, 0, s1);
        cudaError_t e = launch_k1(a, raw_dtype, lens ? DT_F32 : frame_dtype, c->k1_variant, c->sm_count, c->k1_seg_rows, s1, &l);
        if (prof) prof_mark(c, 0, s1);
        if ((r = launched(c, l, e, "K1 launch"))) return r;
        if (lens) {
            if (overlap) {
                CK(cudaEventRecord(ov.k1[gi & 1].get(), s1));
                CK(cudaStreamWaitEvent(st, ov.k1[gi & 1].get(), 0));
            }
            if (prof) prof_mark(c, 1, st);
            r = run_k2(c, mid, DT_F32, frames, persp ? frame_dtype : out_dtype, nf, nullptr, nullptr, border, x0, y0, ow, oh,
                       c->out_scale, st);
            if (prof) prof_mark(c, 1, st);
            if (r) return r;
            if (overlap) CK(cudaEventRecord(ov.k2[gi & 1].get(), st));
        }
        if (!persp) continue;
        if (p.tilt) {                                  // float64, in place (launch_k3_divide's in-place kernel)
            l = 0;
            e = launch_k3_divide(frames, DT_F64, p.tilt.get(), (double*)frames, src_px, nf, c->sm_count, st, &l);
            if ((r = launched(c, l, e, "divide kernel launch"))) return r;
        }
        r = run_k3(c, frames, frame_dtype, oh, ow, (char*)out + f * out_stride, out_dtype, p.dh, p.dw, nf, p.M,
                   p.table ? p.table.get() + first + f : nullptr, IMGCORR_INTER_LANCZOS4, 0, p.border, c->out_scale, st);
        if (r) return r;
    }
    return IMGCORR_OK;
}

// the refusals of a chain call with per-frame backgrounds, before anything is enqueued
static int check_bg(int raw_dtype, const void* bg, int bg_dtype, int flags) {
    if (!bg) return IMGCORR_OK;
    if (!(flags & IMGCORR_DO_DARK)) return fail(IMGCORR_ERR_INVALID, "per-frame backgrounds need IMGCORR_DO_DARK");
    if (raw_dtype < DT_U8 || raw_dtype > DT_F32) return fail(IMGCORR_ERR_INVALID, "raw_dtype %d (U8, U16 or F32)", raw_dtype);
    if (bg_dtype != raw_dtype && bg_dtype != DT_F32)
        return fail(IMGCORR_ERR_INVALID, "bg_dtype %d: the raw dtype (%d) or F32", bg_dtype, raw_dtype);
    return IMGCORR_OK;
}

static int correct_batch(imgcorr_ctx* c, const void* raw_dev, int raw_dtype, const void* bg_dev, int bg_dtype, void* out_dev,
                         int out_dtype, int n_frames, double threshold, int ksize, int flags, int use_lens,
                         double border_value, int x0, int y0, int ow, int oh, void* stream) {
    if (!raw_dev || !out_dev) return fail(IMGCORR_ERR_INVALID, "null image pointer");
    if (int r = check_bg(raw_dtype, bg_dev, bg_dtype, flags)) return r;
    if (int r = check_exposures(c, flags, bg_dev, n_frames)) return r;
    const bool lens = use_lens && c->has_lens;
    if (!lens) { x0 = 0; y0 = 0; ow = c->W; oh = c->H; }
    const bool persp = flags & IMGCORR_DO_PERSPECTIVE;
    if (persp) { int r = check_perspective(c, out_dtype, ow, oh, n_frames); if (r) return r; }
    return chain_frames(c, raw_dev, raw_dtype, out_dev, out_dtype, n_frames, threshold, ksize, flags, lens, persp,
                        border_value, x0, y0, ow, oh, (cudaStream_t)stream, 0, bg_dev, bg_dtype);
}

extern "C" IMGCORR_API int imgcorr_correct_batch(imgcorr_ctx* c, const void* raw_dev, int raw_dtype, void* out_dev, int out_dtype,
                                     int n_frames, double threshold, int ksize, int flags, int use_lens,
                                     double border_value, int x0, int y0, int ow, int oh, void* stream) {
    GUARD(c);
    return correct_batch(c, raw_dev, raw_dtype, nullptr, DT_F32, out_dev, out_dtype, n_frames, threshold, ksize, flags, use_lens,
                         border_value, x0, y0, ow, oh, stream);
}

extern "C" IMGCORR_API int imgcorr_correct_batch_bg(imgcorr_ctx* c, const void* raw_dev, int raw_dtype, const void* bg_dev, int bg_dtype,
                                        void* out_dev, int out_dtype, int n_frames, double threshold, int ksize, int flags,
                                        int use_lens, double border_value, int x0, int y0, int ow, int oh, void* stream) {
    GUARD(c);
    return correct_batch(c, raw_dev, raw_dtype, bg_dev, bg_dtype, out_dev, out_dtype, n_frames, threshold, ksize, flags, use_lens,
                         border_value, x0, y0, ow, oh, stream);
}

// ---- host-buffer pipeline ---------------------------------------------------------------------
static bool is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

// bg_bytes: the per-slot background buffer of a call with backgrounds (0: none needed, none allocated)
static int ensure_pipeline(imgcorr_ctx* c, size_t raw_bytes, size_t out_bytes, size_t bg_bytes) {
    if (!c->s_in) {
        Stream in, k, out;
        CK(new_stream(in));
        CK(new_stream(k));
        CK(new_stream(out));
        c->s_in = std::move(in);
        c->s_k = std::move(k);
        c->s_out = std::move(out);
    }
    if ((int)c->slots.size() == c->host_slots && c->slot_raw_bytes >= raw_bytes && c->slot_out_bytes >= out_bytes) {
        if (c->slot_bg_bytes >= bg_bytes) return IMGCORR_OK;
        // the ring stays; its slots get (larger) background buffers.  Every earlier host call has drained the ring.
        for (auto& s : c->slots) {
            s.d_bg.reset();
            s.h_bg.reset();
        }
        c->slot_bg_bytes = 0;
        for (auto& s : c->slots) CK(dev_alloc(s.d_bg, bg_bytes));
        c->slot_bg_bytes = bg_bytes;
        return IMGCORR_OK;
    }
    CK(cudaDeviceSynchronize());
    c->slots.clear();                                  // the old ring goes first, so peak memory stays one ring
    std::vector<HostSlot> ring(c->host_slots);
    for (auto& s : ring) {
        CK(dev_alloc(s.d_raw, raw_bytes));
        CK(dev_alloc(s.d_out, out_bytes));
        if (bg_bytes) CK(dev_alloc(s.d_bg, bg_bytes));
        CK(new_event(s.ev_in));
        CK(new_event(s.ev_k));
        CK(new_event(s.ev_out));
    }
    c->slots = std::move(ring);
    c->slot_raw_bytes = raw_bytes;
    c->slot_out_bytes = out_bytes;
    c->slot_bg_bytes = bg_bytes;
    return IMGCORR_OK;
}

static int correct_host(imgcorr_ctx* c, const void* raw_host, int raw_dtype, const void* bg_host, int bg_dtype, void* out_host,
                        int out_dtype, int n_frames, double threshold, int ksize, int flags, int use_lens,
                        double border_value, int x0, int y0, int ow, int oh) {
    if (!raw_host || !out_host) return fail(IMGCORR_ERR_INVALID, "null image pointer");
    if (int r = check_bg(raw_dtype, bg_host, bg_dtype, flags)) return r;
    if (n_frames < 0) return fail(IMGCORR_ERR_INVALID, "n_frames %d", n_frames);
    if (int r = check_exposures(c, flags, bg_host, n_frames)) return r;
    if (raw_dtype < DT_U8 || raw_dtype > DT_F32) return fail(IMGCORR_ERR_INVALID, "raw_dtype %d (U8, U16 or F32)", raw_dtype);
    if (c->raw_gap) return fail(IMGCORR_ERR_INVALID, "IMGCORR_OPT_RAW_FRAME_GAP is not available for host frames (pass the pixel blocks)");
    if (out_dtype < DT_U8 || out_dtype > DT_F64) return fail(IMGCORR_ERR_INVALID, "out_dtype must be U8, U16, F32 or F64");
    const bool lens = use_lens && c->has_lens;
    if (!lens) { x0 = 0; y0 = 0; ow = c->W; oh = c->H; }
    const bool persp = flags & IMGCORR_DO_PERSPECTIVE;
    if (persp) { int r = check_perspective(c, out_dtype, ow, oh, n_frames); if (r) return r; }
    const size_t frame_raw = (size_t)c->H * c->W * dtype_size(raw_dtype);
    const size_t frame_bg = bg_host ? (size_t)c->H * c->W * dtype_size(bg_dtype) : 0;
    const size_t frame_out = (persp ? (size_t)c->persp.dw * c->persp.dh : (size_t)ow * oh) * dtype_size(out_dtype);
    // small frames travel in chunks of G frames per ring slot (up to 32 MB of raw data and backgrounds, at most 16 frames):
    // one copy each way and one K1 / K2 launch per chunk instead of per frame; frames above 16 MB (the 4096x3000 workload)
    // keep one frame per slot
    const size_t frame_in = frame_raw + frame_bg;
    int G = 1;
    if (frame_in <= ((size_t)16 << 20)) G = (int)std::min<size_t>(16, ((size_t)32 << 20) / frame_in);
    if (G > n_frames) G = n_frames > 0 ? n_frames : 1;
    const size_t raw_bytes = frame_raw * G, out_bytes = frame_out * G, bg_bytes = frame_bg * G;
    int r = ensure_pipeline(c, raw_bytes, out_bytes, bg_bytes);
    if (r) return r;
    const bool in_pinned = is_pinned(raw_host), out_pinned = is_pinned(out_host);
    const bool bg_pinned = bg_host && is_pinned(bg_host);
    for (auto& s : c->slots) {
        if (!in_pinned && !s.h_raw) CK(host_alloc(s.h_raw, c->slot_raw_bytes));
        if (!out_pinned && !s.h_out) CK(host_alloc(s.h_out, c->slot_out_bytes));
        if (bg_host && !bg_pinned && !s.h_bg) CK(host_alloc(s.h_bg, c->slot_bg_bytes));
    }
    const int ns = (int)c->slots.size();
    const int chunks = (n_frames + G - 1) / G;
    cudaStream_t const s_in = c->s_in.get(), s_k = c->s_k.get(), s_out = c->s_out.get();
    // whatever happens below, no copy from / into the caller's buffers may still be in flight when this call returns
    struct Drain {
        cudaStream_t s_in, s_k, s_out; bool armed = true;
        ~Drain() { if (armed) { cudaStreamSynchronize(s_in); cudaStreamSynchronize(s_k); cudaStreamSynchronize(s_out); } }
    } drain{s_in, s_k, s_out};
    auto frames_of = [&](int k) { return n_frames - k * G < G ? n_frames - k * G : G; };
    auto retire = [&](int k) -> int {          // chunk k's D2H has been enqueued on s_out in slot k % ns
        HostSlot& s = c->slots[k % ns];
        CK(cudaEventSynchronize(s.ev_out.get()));
        if (!out_pinned) memcpy((char*)out_host + (size_t)k * out_bytes, s.h_out.get(), frame_out * frames_of(k));
        return IMGCORR_OK;
    };
    for (int k = 0; k < chunks; ++k) {
        HostSlot& s = c->slots[k % ns];
        if (k >= ns) { r = retire(k - ns); if (r) return r; }
        const int nf = frames_of(k);
        const char* src = (const char*)raw_host + (size_t)k * raw_bytes;
        if (!in_pinned) { memcpy(s.h_raw.get(), src, frame_raw * nf); src = (const char*)s.h_raw.get(); }
        CK(cudaMemcpyAsync(s.d_raw.get(), src, frame_raw * nf, cudaMemcpyHostToDevice, s_in));
        if (bg_host) {
            const char* bsrc = (const char*)bg_host + (size_t)k * bg_bytes;
            if (!bg_pinned) { memcpy(s.h_bg.get(), bsrc, frame_bg * nf); bsrc = (const char*)s.h_bg.get(); }
            CK(cudaMemcpyAsync(s.d_bg.get(), bsrc, frame_bg * nf, cudaMemcpyHostToDevice, s_in));
        }
        CK(cudaEventRecord(s.ev_in.get(), s_in));
        CK(cudaStreamWaitEvent(s_k, s.ev_in.get(), 0));
        r = chain_frames(c, s.d_raw.get(), raw_dtype, s.d_out.get(), out_dtype, nf, threshold, ksize, flags, lens, persp,
                         border_value, x0, y0, ow, oh, s_k, k * G, bg_host ? s.d_bg.get() : nullptr, bg_dtype);
        if (r) return r;
        CK(cudaEventRecord(s.ev_k.get(), s_k));
        CK(cudaStreamWaitEvent(s_out, s.ev_k.get(), 0));
        void* dst = out_pinned ? (void*)((char*)out_host + (size_t)k * out_bytes) : s.h_out.get();
        CK(cudaMemcpyAsync(dst, s.d_out.get(), frame_out * nf, cudaMemcpyDeviceToHost, s_out));
        CK(cudaEventRecord(s.ev_out.get(), s_out));
    }
    for (int k = (chunks > ns ? chunks - ns : 0); k < chunks; ++k) { r = retire(k); if (r) return r; }
    drain.armed = false;                               // every chunk was retired: nothing is in flight
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_correct_host(imgcorr_ctx* c, const void* raw_host, int raw_dtype, void* out_host, int out_dtype,
                                    int n_frames, double threshold, int ksize, int flags, int use_lens,
                                    double border_value, int x0, int y0, int ow, int oh) {
    GUARD(c);
    return correct_host(c, raw_host, raw_dtype, nullptr, DT_F32, out_host, out_dtype, n_frames, threshold, ksize, flags, use_lens,
                        border_value, x0, y0, ow, oh);
}

extern "C" IMGCORR_API int imgcorr_correct_host_bg(imgcorr_ctx* c, const void* raw_host, int raw_dtype, const void* bg_host, int bg_dtype,
                                       void* out_host, int out_dtype, int n_frames, double threshold, int ksize, int flags,
                                       int use_lens, double border_value, int x0, int y0, int ow, int oh) {
    GUARD(c);
    return correct_host(c, raw_host, raw_dtype, bg_host, bg_dtype, out_host, out_dtype, n_frames, threshold, ksize, flags, use_lens,
                        border_value, x0, y0, ow, oh);
}

extern "C" IMGCORR_API int imgcorr_selftest_division(imgcorr_ctx* c, int numerators_per_divisor, unsigned long long seed, double out[2]) {
    GUARD(c);
    if (!out || numerators_per_divisor < 1) return fail(IMGCORR_ERR_INVALID, "bad self-test arguments");
    DevPtr<unsigned long long> d;
    unsigned long long h[2] = {0, 0};
    CK(dev_alloc(d, sizeof h));
    cudaError_t e = cudaMemset(d.get(), 0, sizeof h);
    if (e == cudaSuccess) e = launch_selftest_division(numerators_per_divisor, seed, d.get(), nullptr);
    if (e == cudaSuccess) e = cudaMemcpy(h, d.get(), sizeof h, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return cuda_fail(e, "division self-test");
    c->launches += 1;
    out[0] = (double)h[0];
    double worst;
    memcpy(&worst, &h[1], sizeof worst);
    out[1] = worst;
    return IMGCORR_OK;
}

// ---- K5 -------------------------------------------------------------------------------------
extern "C" IMGCORR_API int imgcorr_stack_mean(imgcorr_ctx* c, const void* frames_dev, int dtype, int n_frames, size_t elems,
                                  const double* minus_dev, double minus_scalar, int use_scalar, int gray3, double* out_dev, void* stream) {
    GUARD(c);
    if (!frames_dev || !out_dev) return fail(IMGCORR_ERR_INVALID, "null pointer");
    if (dtype < DT_U8 || dtype > DT_F64) return fail(IMGCORR_ERR_INVALID, "bad dtype %d", dtype);
    if (n_frames < 1) return fail(IMGCORR_ERR_INVALID, "n_frames %d", n_frames);
    if (gray3 && elems % 3) return fail(IMGCORR_ERR_INVALID, "gray conversion needs 3 interleaved channels");
    int l = 0;
    cudaError_t e = launch_k5_stack_mean(frames_dev, dtype, n_frames, elems, minus_dev, minus_scalar, use_scalar, gray3, out_dev, c->sm_count,
                                         (cudaStream_t)stream, &l);
    return launched(c, l, e, "stack mean launch");
}

extern "C" IMGCORR_API int imgcorr_scale_f64(imgcorr_ctx* c, double* data_dev, size_t elems, double divisor, void* stream) {
    GUARD(c);
    if (!data_dev) return fail(IMGCORR_ERR_INVALID, "null pointer");
    int l = 0;
    cudaError_t e = launch_k5_scale(data_dev, elems, divisor, c->sm_count, (cudaStream_t)stream, &l);
    return launched(c, l, e, "scale launch");
}

extern "C" IMGCORR_API int imgcorr_subsample_f64(imgcorr_ctx* c, const double* src_dev, int height, int width, int step_y, int step_x,
                                     double* dst_dev, void* stream) {
    GUARD(c);
    if (!src_dev || !dst_dev) return fail(IMGCORR_ERR_INVALID, "null pointer");
    if (height <= 0 || width <= 0 || step_y <= 0 || step_x <= 0) return fail(IMGCORR_ERR_INVALID, "bad shape / step");
    int l = 0;
    cudaError_t e = launch_k5_subsample(src_dev, height, width, step_y, step_x, dst_dev, (cudaStream_t)stream, &l);
    return launched(c, l, e, "subsample launch");
}

extern "C" IMGCORR_API int imgcorr_linear_fit(imgcorr_ctx* c, const void* frames_dev, int dtype, int n_frames, size_t pixels, const double* x_host,
                                  double max_intensity, double min_ascent, double* offset_dev, double* ascent_dev, double* rmse_dev,
                                  void* stream) {
    GUARD(c);
    if (!frames_dev || !x_host || !offset_dev || !ascent_dev) return fail(IMGCORR_ERR_INVALID, "null pointer");
    if (dtype < DT_U8 || dtype > DT_F64) return fail(IMGCORR_ERR_INVALID, "bad dtype %d", dtype);
    if (n_frames < 2) return fail(IMGCORR_ERR_INVALID, "a line needs at least 2 exposure times (got %d)", n_frames);
    double mn = x_host[0], mx = x_host[0];
    for (int k = 1; k < n_frames; ++k) { mn = x_host[k] < mn ? x_host[k] : mn; mx = x_host[k] > mx ? x_host[k] : mx; }
    DevPtr<double> xs;
    CK(dev_alloc(xs, n_frames * sizeof(double)));
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyAsync(xs.get(), x_host, n_frames * sizeof(double), cudaMemcpyHostToDevice, st);
    int l = 0;
    if (e == cudaSuccess)
        e = launch_k5_linear_fit(frames_dev, dtype, n_frames, pixels, xs.get(), max_intensity, min_ascent, 0.5 * (mn + mx), offset_dev,
                                 ascent_dev, rmse_dev, c->sm_count, st, &l);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);       // x_host / xs may go away when this returns
    return launched(c, l, e, "linear fit");
}

// ---- host-side fingerprint of a calibration array ---------------------------------------------------------
static unsigned long long fp_chunk(const unsigned char* p, size_t n) {
    // four independent multiply-xor lanes over 8-byte words (the loop is load bound), tail bytes folded in at the end
    const unsigned long long K = 0x9E3779B97F4A7C15ull;
    unsigned long long a0 = 1, a1 = 2, a2 = 3, a3 = 4;
    size_t i = 0;
    for (; i + 32 <= n; i += 32) {
        unsigned long long w[4];
        memcpy(w, p + i, 32);
        a0 = (a0 ^ w[0]) * K; a1 = (a1 ^ w[1]) * K; a2 = (a2 ^ w[2]) * K; a3 = (a3 ^ w[3]) * K;
    }
    unsigned long long t = 0;
    for (int s = 0; i < n; ++i, s += 8) t ^= (unsigned long long)p[i] << (s & 63);
    unsigned long long h = (a0 ^ (a1 >> 17) ^ (a1 << 47)) * K;
    h = (h ^ a2 ^ (a3 >> 29) ^ (a3 << 35)) * K;
    h = (h ^ t ^ (unsigned long long)n) * K;
    return h ^ (h >> 32);
}

extern "C" IMGCORR_API int imgcorr_host_fingerprint(const void* host_ptr, size_t bytes, unsigned long long* out) {
    if (!out || (!host_ptr && bytes)) return fail(IMGCORR_ERR_INVALID, "null pointer");
    const unsigned char* p = (const unsigned char*)host_ptr;
    unsigned nt = std::thread::hardware_concurrency();
    if (nt > 16) nt = 16;
    if (nt < 1 || bytes < ((size_t)4 << 20)) nt = 1;
    std::vector<unsigned long long> part(nt, 0);
    const size_t chunk = ((bytes / nt) + 31) & ~(size_t)31;
    auto work = [&](unsigned t) {
        const size_t lo = (size_t)t * chunk < bytes ? (size_t)t * chunk : bytes;
        const size_t hi = lo + chunk < bytes && t + 1 < nt ? lo + chunk : bytes;
        part[t] = fp_chunk(p + lo, hi - lo);
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
    unsigned long long h = 0x243F6A8885A308D3ull;
    for (unsigned t = 0; t < nt; ++t) h = (h ^ part[t]) * 0x9E3779B97F4A7C15ull + t;
    *out = h;
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_host_alloc(size_t bytes, void** out_ptr) {
    if (!out_ptr) return fail(IMGCORR_ERR_INVALID, "out_ptr is null");
    *out_ptr = nullptr;
    CK(cudaHostAlloc(out_ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return IMGCORR_OK;
}

extern "C" IMGCORR_API int imgcorr_host_free(void* ptr) {
    if (!ptr) return IMGCORR_OK;
    CK(cudaFreeHost(ptr));
    return IMGCORR_OK;
}
