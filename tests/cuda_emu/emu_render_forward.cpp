// Host harness: the fp32 tile-per-CTA forward (seganygaussians_b200/csrc/render_forward_kernels.cuh) under the execution shim.
// TEST INFRASTRUCTURE ONLY.
#define SAGARS_CUDA_EMU 1
#include <cuda_runtime.h>            // the shim (this directory comes first on the include path)
#include "render_forward_kernels.cuh"
#include "math.cuh"

using namespace sagars;

// the 32-byte records the preprocess kernel writes: {x, y, conic.x, conic.y, conic.z, opacity, accept_threshold, 0}
extern "C" void emu_make_geo(int P, const float* means2D, const float* conic_opacity, float* geo)
{
    for (int i = 0; i < P; i++) {
        float* g = geo + 8 * (size_t)i;
        g[0] = means2D[2 * i]; g[1] = means2D[2 * i + 1];
        g[2] = conic_opacity[4 * i]; g[3] = conic_opacity[4 * i + 1]; g[4] = conic_opacity[4 * i + 2]; g[5] = conic_opacity[4 * i + 3];
        g[6] = accept_threshold(g[5]); g[7] = 0.f;
    }
}

extern "C" int emu_render_forward(int md, int W, int H, int K, const uint2* ranges, const uint32_t* point_list,
                                  const float* geo, const float* features, const float* mask, const float* depths, const float* bg,
                                  float* final_T, uint32_t* n_contrib, float* out_color, float* out_mask, float* out_depth)
{
    cuda_emu::thread_exit_hook = emu_async::flush_thread;
    const unsigned tx = (W + TILE_X - 1) / TILE_X, ty = (H + TILE_Y - 1) / TILE_Y;
    const bool vec = (K % 4) == 0;
    const int nq = (K + 3) / 4;
#define GO(NQ_, VEC_, MD_) cuda_emu::launch2d(tx, ty, TILE_PIX, sizeof(FwdSmem<NQ_>), render_forward_kernel<NQ_, VEC_, MD_, true>, ranges, point_list, \
                                              W, H, K, geo, features, mask, depths, bg, final_T, n_contrib, out_color, out_mask, out_depth)
    if (md) { if (nq == 1 && !vec) { GO(1, false, true); return 0; } return -1; }
    if (nq == 1 && !vec) { GO(1, false, false); return 0; }
    if (nq == 2 && vec) { GO(2, true, false); return 0; }
    if (nq == 2 && !vec) { GO(2, false, false); return 0; }
    if (nq <= 8 && vec) { GO(8, true, false); return 0; }
#undef GO
    return -1;
}
