// render_forward.cu -- per-tile front-to-back alpha compositing of C feature channels
// (+ optional mask / depth channels).
//
// Semantics: CF cuda_rasterizer/forward.cu:264-385 (DEPTH forward.cu:262-387 adds the mask/depth
// accumulators), SURVEY.md Appendix A.10-A.12.  One CTA per 16x16 tile, one thread per pixel.
// What is this library's own:
//   * the per-instance records ({xy, conic, opacity, depth} = 32 B) and the C-float feature rows of
//     a batch of instances are staged in shared memory by asynchronous 16-byte copies
//     (cp.async / LDGSTS), double buffered so the copies of batch b+1 overlap the blending of batch
//     b; the reference re-reads every feature from global memory per pixel per channel;
//   * a warp covers an 8x4 pixel block (the reference: 16x2), which cuts the number of
//     (warp, Gaussian) pairs that have any pixel to blend;
//   * a warp stops as soon as its 32 pixels are saturated (the reference only stops per CTA, per
//     256-instance batch);
//   * a (warp, splat) pair in which no pixel can pass the reference's tests (power <= 0 and a conservative
//     per-splat lower bound on power that implies alpha >= 1/255) is rejected with one warp vote, before expf;
//   * C is a run-time value (<= 64), dispatched onto float4-group templates.
// The per-pixel arithmetic (power, alpha, the 1/255 and 1e-4 tests, the order of accumulation)
// is kept operation for operation so that n_contrib / final_T / colours match the reference.
#include "common.cuh"
#include <cstdlib>
#include "cp_async.cuh"
#include "render_forward_kernels.cuh"

namespace sagars {

template <int NQ, bool VEC, bool MD, bool COLOR>
static int launch_fwd_t(const sagars_forward_args& a, const Dims& d, GeomView g, ImageView im,
                        const uint32_t* point_list, const float* features, cudaStream_t s, bool debug)
{
    auto kern = render_forward_kernel<NQ, VEC, MD, COLOR>;
    const size_t smem = sizeof(FwdSmem<NQ>);
    {   // opt in to the dynamic shared-memory size once per device (not on every launch: the call takes the context lock)
        static DeviceOnce once;
        int dev = 0;
        SAGARS_CUDA(cudaGetDevice(&dev));
        if (once.need(dev)) {
            SAGARS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            once.done(dev);
        }
    }
    dim3 grid(d.tiles_x, d.tiles_y);
    kern<<<grid, TILE_PIX, smem, s>>>(im.ranges, point_list, d.W, d.H, d.C, g.geo, features, a.mask, g.depths, a.background,
                                      im.final_T, im.n_contrib, a.out_color, a.out_mask, a.out_depth);
    SAGARS_LAUNCH_CHECK(s, debug);
    return SAGARS_OK;
}

int launch_render_forward(const sagars_forward_args& a, const Dims& d, GeomView g, ImageView im,
                          const uint32_t* point_list, cudaStream_t s, bool debug)
{
    const bool md = (a.flags & SAGARS_FLAG_MASK_DEPTH) != 0;
    const bool mask_only = (a.flags & SAGARS_FLAG_MASK_ONLY) != 0;
    const float* features = a.colors_precomp != nullptr ? a.colors_precomp : g.rgb;
    const int K = d.C;
    if (mask_only) return launch_fwd_t<1, false, true, false>(a, d, g, im, point_list, features, s, debug);
    // colour-only rendering with the channel contraction on the tensor cores.  K = 32 (SAGA's feature rendering): the
    // warp-per-block mma.sync kernel (render_forward_warp.cu), or with SAGARS_FLAG_FWD_TILE the tile-per-CTA tcgen05 / TMEM
    // kernel (render_forward_tc.cu); SAGARS_FLAG_FWD_WARP_ANY extends the warp kernel to every channel count.  Everything
    // else (DEPTH, other channel counts, SAGARS_FLAG_NO_TENSOR_CORES) is the fp32 SIMT kernel below, whose colours are
    // bit-identical to the reference's.
    if (!md && !(a.flags & SAGARS_FLAG_NO_TENSOR_CORES)) {
        if (K == 32 && a.colors_precomp != nullptr) {
            if (a.flags & SAGARS_FLAG_FWD_TILE) return launch_render_forward_tc(a, d, g, im, point_list, s, debug);
            return launch_render_forward_warp(a, d, g, im, point_list, s, debug);
        }
        if (a.flags & SAGARS_FLAG_FWD_WARP_ANY) return launch_render_forward_warp(a, d, g, im, point_list, s, debug);
    }
    const bool vec = (K % 4) == 0;
    const int nq = (K + 3) / 4;
#define SAGARS_FWD_CASE(NQ_)                                                                               \
    if (nq <= NQ_) {                                                                                       \
        if (md) return vec ? launch_fwd_t<NQ_, true, true, true>(a, d, g, im, point_list, features, s, debug) \
                           : launch_fwd_t<NQ_, false, true, true>(a, d, g, im, point_list, features, s, debug); \
        return vec ? launch_fwd_t<NQ_, true, false, true>(a, d, g, im, point_list, features, s, debug)       \
                   : launch_fwd_t<NQ_, false, false, true>(a, d, g, im, point_list, features, s, debug);     \
    }
    SAGARS_FWD_CASE(1)
    SAGARS_FWD_CASE(2)
    SAGARS_FWD_CASE(4)
    SAGARS_FWD_CASE(8)
    SAGARS_FWD_CASE(16)
#undef SAGARS_FWD_CASE
    set_error("unsupported channel count %d (max %d)", K, SAGARS_MAX_CHANNELS);
    return SAGARS_EINVAL;
}

}  // namespace sagars
