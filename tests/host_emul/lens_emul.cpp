// Host emulation of K2's map with OpenCV's full distortion model (rational, thin-prism and tilted-sensor terms):
// compiles imgprocessor_b200/csrc/imgcorr_core.cuh, the functions the CUDA kernels call per pixel, with g++ and runs
// them over a whole map.  TEST-ONLY (built into tests/_build/libimgcorr_lens_emul.so by tests/lens_ref.py).
#include "../../imgprocessor_b200/csrc/imgcorr_core.cuh"

using namespace imgcorr;

// n_dist coefficients in OpenCV's order.  The 5-term functions run when every extra term is zero, as in the library.
// Returns -1 for a singular P, else 1 if the extended model ran, 0 if the 5-term one did.
extern "C" __attribute__((visibility("default")))
int emul_maps_ext(const double* K, const double* dist, int n_dist, const double* P, int H, int W, float* mapx, float* mapy,
                  int force_ext) {
    LensConst L;
    LensExt E;
    if (!make_lens_const(K, dist, n_dist, P, L)) return -1;
    const bool ext = make_lens_ext(dist, n_dist, E) || force_ext;
    for (int v = 0; v < H; ++v)
        for (int u = 0; u < W; ++u) {
            const size_t i = (size_t)v * W + u;
            if (ext) undistort_map_ext(L, E, u, v, mapx[i], mapy[i]);
            else undistort_map(L, u, v, mapx[i], mapy[i]);
        }
    return ext ? 1 : 0;
}

extern "C" __attribute__((visibility("default")))
void emul_tilt(double tau_x, double tau_y, double* t) {
    const double d[14] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, tau_x, tau_y};
    LensExt E;
    make_lens_ext(d, 14, E);
    for (int i = 0; i < 9; ++i) t[i] = E.t[i];
}
