/*
 * sagars.h -- C ABI of the B200-native (sm_100a) differentiable Gaussian feature rasterizer.
 *
 * This is the drop-in boundary for ONE hot path of Jumpat/SegAnyGAussians: the tile-based
 * differentiable Gaussian rasterizer behind `GaussianRasterizer` / `gaussian_renderer.render*`.
 * Plain C: raw device pointers, sizes, scalars; no torch / C++ types.  Every entry point names the
 * reference interface it replaces (paths relative to the reference repository root; CF = the
 * contrastive-feature variant `submodules/diff-gaussian-rasterization_contrastive_f`, DEPTH =
 * `submodules/diff-gaussian-rasterization-depth`, BASE = `submodules/diff-gaussian-rasterization`).
 *
 * Conventions
 *  - all pointers are DEVICE pointers on device `device` unless a field says "host";
 *  - tensors are contiguous fp32 (int32 for radii), exactly as the reference glue requires
 *    (CF rasterize_points.cu:94-111 calls .contiguous() on everything);
 *  - optional inputs are NULL when absent (the reference maps 0-element tensors to nullptr,
 *    CF diff_gaussian_rasterization_contrastive_f/__init__.py:196-206);
 *  - matrices are the reference's transposed (row-vector) 4x4s read column-major
 *    (CF cuda_rasterizer/auxiliary.h:58-77);
 *  - every function returns 0 on success or a SAGARS_E* code; `sagars_last_error()` returns the
 *    thread-local message (the Python shim raises RuntimeError with it, mirroring the C++
 *    exceptions of CF rasterize_points.cu:57-59 and rasterizer_impl.cu:242-245);
 *  - the library never allocates or frees device memory: scratch comes from the three allocator
 *    callbacks, which mirror the reference's `std::function<char*(size_t)>` resize lambdas
 *    (CF rasterize_points.cu:27-33, rasterizer_impl.cu:226,239,284).  The caller keeps the three
 *    buffers alive and unmodified until the matching backward call (the reference does this via
 *    ctx.save_for_backward, CF __init__.py:96);
 *  - all work is enqueued on the caller's `stream` (the reference used the legacy default stream).
 *    Forward performs ONE stream synchronisation (it must read `num_rendered` on the host to size
 *    the binning buffer, like CF rasterizer_impl.cu:280-281); backward performs none.
 */
#ifndef SAGARS_H_INCLUDED
#define SAGARS_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAGARS_ABI_VERSION 4

#if defined(__GNUC__)
#define SAGARS_API __attribute__((visibility("default")))
#else
#define SAGARS_API
#endif

/* tile geometry is part of the contract: tile ids must be bit-exact (CF config_contrastive_f.h:16-17) */
#define SAGARS_TILE_X 16
#define SAGARS_TILE_Y 16
#define SAGARS_MAX_CHANNELS 64

enum {
    SAGARS_OK = 0,
    SAGARS_EINVAL = 1,      /* bad argument (shape / NULL / unsupported channel count)              */
    SAGARS_ECUDA = 2,       /* a CUDA runtime call or kernel failed                                  */
    SAGARS_ENOCOLOR = 3,    /* "For non-RGB, provide precomputed Gaussian colors!"                   */
    SAGARS_EALLOC = 4,      /* an allocator callback returned NULL                                   */
    SAGARS_EPREFILTER = 5   /* a point was culled although `prefiltered` was set (reference traps)   */
};

/* flags */
#define SAGARS_FLAG_PREFILTERED 1u   /* CF auxiliary.h:156-160                                        */
#define SAGARS_FLAG_DEBUG 2u         /* sync + check after every stage (CF auxiliary.h:166-173)       */
#define SAGARS_FLAG_MASK_DEPTH 4u    /* DEPTH variant: extra per-Gaussian mask + view-depth channels  */
#define SAGARS_FLAG_MASK_ONLY 8u     /* DEPTH mask-only path (forward_mask / mask_forward)            */
#define SAGARS_FLAG_CUB_SORT 16u     /* use cub::DeviceRadixSort instead of the library's own sort    */
#define SAGARS_FLAG_NO_TENSOR_CORES 32u /* force the fp32 SIMT blend kernels (bit-exact colours) instead of the tensor-core ones */
#define SAGARS_FLAG_FWD_TILE 64u     /* forward at C = 32: tile-per-CTA tcgen05 / TMEM kernel (render_forward_tc.cu) instead of
                                        the default warp-per-block mma.sync kernel (render_forward_warp.cu)              */
#define SAGARS_FLAG_BWD_TILE 128u    /* backward: one CTA per 16x16 tile (render_backward_mma.cu) instead of the default
                                        one warp per 8x4 pixel block (render_backward_warp.cu)                          */
#define SAGARS_FLAG_FWD_WARP_ANY 256u /* forward: the warp-per-block tensor-core kernel for every colour-only channel count
                                        (default: only C = 32; other counts use the fp32 SIMT kernel, bit-exact colours)  */

/* 512u: unassigned and ignored.  Callers built against earlier v4 headers may still set it, so it is not reused */

#define SAGARS_FLAG_TILE_SORT 1024u  /* binning without a global sort: per-tile instance counts -> scan -> scatter -> one CTA per tile
                                        sorts its own segment (tile_sort.cu) instead of duplicate + 6 radix passes + range
                                        detection.  Bit-identical point_list / keys / ranges; opt-in until measured            */

#define SAGARS_FLAG_DEPTH_FIRST 4096u /* binning: sort the P Gaussians by depth (4 passes over P), emit their instances in that order, then ONE
                                        stable sort of the instances on the tile bits (2 passes for <= 65,536 tiles) instead of 6 passes
                                        over the R duplicated (tile | depth) keys.  Bit-identical point_list / keys / ranges          */
#define SAGARS_FLAG_BWD_TC 2048u     /* backward at C = 32 precomputed colours: tcgen05 / TMEM kernel, one CTA per 16x8 pixel group
                                        (render_backward_tc.cu) instead of the mma.sync warp-per-block kernel                  */

/* Allocator callback: return a device pointer to at least `bytes` bytes (256-B aligned), or NULL.
 * Replaces: std::function<char*(size_t)> geometryBuffer / binningBuffer / imageBuffer
 *           (CF cuda_rasterizer/rasterizer.h:33-35). */
typedef void* (*sagars_alloc_fn)(void* user, size_t bytes);

/* Arguments of the forward pass.
 * Replaces: CudaRasterizer::Rasterizer::forward (CF cuda_rasterizer/rasterizer.h:32-56,
 *           rasterizer_impl.cu:198-336; DEPTH rasterizer_impl.cu:198-345 adds mask/out_mask/out_depth)
 *           as called from RasterizeGaussiansCUDA (CF rasterize_points.cu:35-115). */
typedef struct sagars_forward_args {
    int32_t device;             /* CUDA device ordinal                                               */
    uint32_t flags;             /* SAGARS_FLAG_*                                                     */
    int32_t P;                  /* number of Gaussians                                               */
    int32_t D;                  /* active SH degree                                                  */
    int32_t M;                  /* SH coefficients per Gaussian (0 if shs == NULL)                   */
    int32_t num_channels;       /* C: 3 (BASE/DEPTH) or 32 (CF); runtime here, NUM_CHANNELS there    */
    int32_t width, height;
    float tan_fovx, tan_fovy;
    float scale_modifier;
    const float* background;    /* >= C floats; only the first C are read (CF forward.cu:383)        */
    const float* means3D;       /* [P,3]                                                             */
    const float* shs;           /* [P,M,3] or NULL                                                   */
    const float* colors_precomp;/* [P,C] or NULL                                                     */
    const float* opacities;     /* [P] (or [P,1])                                                    */
    const float* mask;          /* [P] DEPTH only, else NULL                                         */
    const float* scales;        /* [P,3] or NULL                                                     */
    const float* rotations;     /* [P,4] or NULL                                                     */
    const float* cov3D_precomp; /* [P,6] or NULL                                                     */
    const float* viewmatrix;    /* [16]                                                              */
    const float* projmatrix;    /* [16]                                                              */
    const float* cam_pos;       /* [3]                                                               */
    float* out_color;           /* [C,H,W]; written in full (NULL allowed for MASK_ONLY)             */
    float* out_mask;            /* [1,H,W] DEPTH only                                                */
    float* out_depth;           /* [1,H,W] DEPTH only                                                */
    int32_t* radii;             /* [P]; written in full                                              */
    /* Speculative binning (0 = off: size the binning buffer from the exact instance count after the
     * host read-back, exactly like the reference, CF rasterizer_impl.cu:280-285).  When > 0 the binning
     * buffer is requested for `binning_capacity_hint` instances BEFORE the read-back and sort / ranges /
     * blend are queued behind it reading the count from device memory, so the GPU keeps working while
     * the host waits for the count.  If the count turns out larger than the hint, the queued kernels
     * skip their work, the allocator is called again with the exact size and the stages are re-issued:
     * results are identical either way; only the size of the binning buffer differs. */
    int32_t binning_capacity_hint;
    int32_t* binning_capacity_out; /* host, optional: capacity the binning buffer was finally laid out for */
    /* Optional cudaEvent_t (NULL = none).  The per-tile blend -- the FIRST stage that reads colors_precomp / shs -- is made to
     * wait for this event on `stream`; preprocess, key emission, sort and tile ranges (which read geometry only) are not.  A
     * data-parallel trainer records the event after the all-reduce (and optimiser step) of the feature tensor on a side
     * stream: that exchange then overlaps the geometry stages of the next forward instead of serialising with it
     * (seganygaussians_b200/data_parallel.py).  The reference has nothing comparable (single stream, single GPU). */
    void* blend_wait_event;
} sagars_forward_args;

/* Forward: preprocess -> scan -> duplicate keys -> radix sort -> tile ranges -> per-tile blend.
 * On success *num_rendered receives the number of (Gaussian, tile) instances (the reference's
 * return value, CF rasterizer_impl.cu:335). */
SAGARS_API int sagars_forward(const sagars_forward_args* args,
                   sagars_alloc_fn geom_alloc, void* geom_user,
                   sagars_alloc_fn binning_alloc, void* binning_user,
                   sagars_alloc_fn image_alloc, void* image_user,
                   int32_t* num_rendered /* host */,
                   void* stream /* cudaStream_t */);

/* Arguments of the backward pass.
 * Replaces: CudaRasterizer::Rasterizer::backward (CF cuda_rasterizer/rasterizer.h:58-85,
 *           rasterizer_impl.cu:340-434; DEPTH adds dL_dout_mask / dL_dmask) as called from
 *           RasterizeGaussiansBackwardCUDA (CF rasterize_points.cu:117-196).
 * Output gradient tensors are written IN FULL by the library (no pre-zeroing needed), except
 * `dL_dcolors`, which the library zero-fills itself before accumulating into it.
 * `dL_dconic` of the reference ([P,2,2], internal) is replaced by library scratch `grad_scratch`. */
typedef struct sagars_backward_args {
    int32_t device;
    uint32_t flags;
    int32_t P, D, M, R;         /* R = num_rendered returned by the matching forward                 */
    int32_t num_channels;
    int32_t width, height;
    float tan_fovx, tan_fovy;
    float scale_modifier;
    const float* background;
    const float* means3D;
    const float* shs;
    const float* colors_precomp;
    const float* mask;          /* DEPTH only (not read by the gradient; kept for symmetry)          */
    const float* scales;
    const float* rotations;
    const float* cov3D_precomp;
    const float* viewmatrix;
    const float* projmatrix;
    const float* cam_pos;
    const int32_t* radii;       /* [P] as written by forward                                         */
    const void* geom_buffer;    /* the three scratch buffers of the matching forward                 */
    const void* binning_buffer;
    const void* image_buffer;
    const float* dL_dout_color; /* [C,H,W]                                                           */
    const float* dL_dout_mask;  /* [1,H,W] DEPTH only                                                */
    void* grad_scratch;         /* sagars_grad_scratch_bytes(P) bytes of device scratch              */
    float* dL_dmeans2D;         /* [P,3] (z = 0)                                                     */
    float* dL_dopacity;         /* [P,1]                                                             */
    float* dL_dcolors;          /* [P,C]                                                             */
    float* dL_dmask;            /* [P,1] DEPTH only                                                  */
    float* dL_dmeans3D;         /* [P,3]                                                             */
    float* dL_dcov3D;           /* [P,6]                                                             */
    float* dL_dsh;              /* [P,M,3] (may be NULL when M == 0)                                 */
    float* dL_dscales;          /* [P,3]                                                             */
    float* dL_drotations;       /* [P,4]                                                             */
} sagars_backward_args;

SAGARS_API int sagars_backward(const sagars_backward_args* args, void* stream);

/* Frustum test: present[i] = (view-space z of means3D[i] > 0.2).
 * Replaces: CudaRasterizer::Rasterizer::markVisible (CF rasterizer.h:24-30, rasterizer_impl.cu:141-153)
 *           as called from markVisible (CF rasterize_points.cu:198-217). */
SAGARS_API int sagars_mark_visible(int32_t device, int32_t P, const float* means3D, const float* viewmatrix,
                        const float* projmatrix, uint8_t* present /* bool[P] */, void* stream);

/* Scratch sizes. Replace: required<GeometryState/ImageState/BinningState> (CF rasterizer_impl.h:67-73). */
SAGARS_API size_t sagars_geom_bytes(int32_t P);
SAGARS_API size_t sagars_image_bytes(int32_t width, int32_t height);
SAGARS_API size_t sagars_binning_bytes(int32_t num_rendered);
SAGARS_API size_t sagars_grad_scratch_bytes(int32_t P);

/* Layout of the scratch buffers (byte offsets from the buffer start), for parity tests that must
 * compare the integer state bit-exactly with the reference's GeometryState / ImageState /
 * BinningState (CF rasterizer_impl.cu:155-194).  The layout is otherwise private. */
typedef struct sagars_geom_layout {
    size_t depths;          /* f32[P]   view-space z                                                 */
    size_t geo;             /* f32[P,8] {x, y, conic.x, conic.y, conic.z, opacity, accept_threshold, 0}         */
    size_t cov3D;           /* f32[P,6]                                                              */
    size_t rgb;             /* f32[P,3] SH->RGB result (only when shs given)                         */
    size_t clamped;         /* u8[P,3]                                                               */
    size_t tiles_touched;   /* u32[P]                                                                */
    size_t point_offsets;   /* u32[P]   inclusive prefix sum of tiles_touched                        */
    size_t status;          /* u32[8]   device status words                                          */
    size_t total;
} sagars_geom_layout;

typedef struct sagars_image_layout {
    size_t final_T;         /* f32[H*W]                                                              */
    size_t n_contrib;       /* u32[H*W]                                                              */
    size_t ranges;          /* uint2[tiles]                                                          */
    size_t total;
} sagars_image_layout;

typedef struct sagars_binning_layout {
    size_t point_list;      /* u32[R] Gaussian index per sorted instance                             */
    size_t point_list_keys; /* u64[R] sorted keys (tile << 32 | depth bits)                          */
    size_t total;
} sagars_binning_layout;

SAGARS_API int sagars_get_geom_layout(int32_t P, sagars_geom_layout* out);
SAGARS_API int sagars_get_image_layout(int32_t width, int32_t height, sagars_image_layout* out);
SAGARS_API int sagars_get_binning_layout(int32_t num_rendered, sagars_binning_layout* out);

/* Stand-alone stable LSD radix sort of (u64 key, u32 value) pairs on key bits [0, end_bit), the
 * library's replacement for cub::DeviceRadixSort::SortPairs at CF rasterizer_impl.cu:303-308.
 * `temp` must hold sagars_sort_temp_bytes(n) bytes.  Exposed so tests can pin it against CUB / the
 * CPU oracle on adversarial inputs. */
SAGARS_API size_t sagars_sort_temp_bytes(int32_t n);
SAGARS_API int sagars_sort_pairs(int32_t device, int32_t n, int32_t end_bit,
                      const uint64_t* keys_in, const uint32_t* vals_in,
                      uint64_t* keys_out, uint32_t* vals_out,
                      void* temp, int32_t use_cub, void* stream);

/* Exact K nearest neighbours (squared Euclidean distance, ascending) of every query in a reference cloud, on a uniform
 * grid; runs on `stream` without host synchronisation.  `queries == NULL` (or == points): the cloud against itself.
 * `exclude_self` (cloud against itself only): point i is never its own neighbour.  Outputs are optional:
 * idx_out [Q,K] (-1 where the cloud has fewer than K eligible points), dist2_out [Q,K], mean_dist2_out [Q] = mean of the
 * K distances.  1 <= K <= 32.  `temp`: sagars_knn_temp_bytes(num_points) bytes of device scratch.
 * Replaces (SURVEY.md section 8(f) rank 1, imports the reference's scripts need to start):
 *   simple_knn._C.distCUDA2  -- submodules/simple-knn/simple_knn.cu:146-219 (K = 3, exclude_self, mean_dist2_out;
 *                               same distance expression and summation order, results equal to fp32 rounding);
 *   pytorch3d.ops.knn_points -- call sites scene/gaussian_model_ff.py:326-331, 345-350 (K = 16, self included). */
SAGARS_API size_t sagars_knn_temp_bytes(int32_t num_points);
SAGARS_API int sagars_knn(int32_t device, int32_t num_points, const float* points /* [N,3] */,
                          int32_t num_queries, const float* queries /* [Q,3] or NULL */, int32_t K, int32_t exclude_self,
                          int64_t* idx_out, float* dist2_out, float* mean_dist2_out, void* temp, void* stream);

/* Loss-side consumer of the K-feature render (SURVEY.md section 8(f) rank 3), fused.
 * Replaces the tensor expression of train_contrastive_feature.py:232-254:
 *     norm = render.norm(dim=0, p=2).mean();  up = F.interpolate(render[None], (out_h, out_w), mode='bilinear')[0];
 *     samples = up.reshape(C, -1)[:, ray_index]
 * forward : samples[C, num_rays] and norm_sum[0] = sum over the pixels of ||render[:, p]||_2 (the caller divides by H*W);
 * backward: dL_dimage[C, H, W] = dL_dnorm_mean / (H W) * render / ||render[:, p]|| + the four bilinear taps of every ray
 *           (written in full).  ray_index: flat indices into the RESIZED image (row-major), int64. */
SAGARS_API int sagars_sample_rays_forward(int32_t device, int32_t C, int32_t H, int32_t W, int32_t out_h, int32_t out_w,
                                          const float* image, const int64_t* ray_index, int32_t num_rays, float* samples,
                                          float* norm_sum, void* stream);
SAGARS_API int sagars_sample_rays_backward(int32_t device, int32_t C, int32_t H, int32_t W, int32_t out_h, int32_t out_w,
                                           const float* image, const int64_t* ray_index, int32_t num_rays, const float* dL_dsamples,
                                           const float* dL_dnorm_mean, float* dL_dimage, void* stream);

/* Fused feature smoothing in front of the rasterizer (SURVEY.md section 8(f) rank 2):
 *     out_i = mean_k( F[idx[i,k]] / max(||F[idx[i,k]]||, 1e-12) ),   optionally  out_i /= (||out_i|| + 1e-9)
 * Replaces the tensor expression of scene/gaussian_model_ff.py:338-364 (`F.normalize(...)[select_idx, :].mean(dim=1)`)
 * and gaussian_renderer/__init__.py:362-363 (`colors_precomp / (colors_precomp.norm(dim=1, keepdim=True) + 1e-9)`)
 * and their autograd backward (a [P,Ks,C] scatter-add).  features [P,C] fp32, nbr_idx [P,Ks] int64 (entries in [0,P)),
 * out [P,C]; (when normalize_out) mean_norm [P] is an output of the forward that the backward needs.
 * The backward accumulates through dL_dn_scratch [P,C] (zeroed by the library) and writes dL_dfeatures [P,C] in full. */
SAGARS_API int sagars_smooth_forward(int32_t device, int32_t P, int32_t C, int32_t Ks, const float* features,
                                     const int64_t* nbr_idx, int32_t normalize_out, float* out,
                                     float* mean_norm, void* stream);
SAGARS_API int sagars_smooth_backward(int32_t device, int32_t P, int32_t C, int32_t Ks, const float* features,
                                      const int64_t* nbr_idx, int32_t normalize_out,
                                      const float* mean_norm, const float* out, const float* dL_dout,
                                      float* dL_dn_scratch, float* dL_dfeatures, void* stream);

/* The library's own all-reduce (sum, fp32, in place) over an NVSwitch multicast mapping (opt-in alternative to the NCCL call of
 * seganygaussians_b200/data_parallel.py; SURVEY.md section 8(e)).  `multicast_ptr` is the multicast address of a buffer of
 * `numel` floats (numel % 4 == 0) that belongs to a symmetric allocation spanning all `world` GPUs of the process group; the
 * caller orders it against producers and consumers of the buffer with device-side barriers of that allocation (before and
 * after).  Rank r reduces and re-broadcasts the r-th 1/world slice with multimem.ld_reduce / multimem.st. */
SAGARS_API int sagars_multimem_allreduce_f32(int32_t device, void* multicast_ptr, int64_t numel, int32_t rank, int32_t world,
                                             void* stream);

/* number of kernels launched by this library (process-wide) since the last reset
 * (bench.py reports it as `gpu_launches`). */
SAGARS_API int64_t sagars_launch_count(void);
SAGARS_API void sagars_reset_launch_count(void);

/* Optional per-stage device timing: when enabled, every stage of forward / backward is bracketed by CUDA
 * events recorded on the caller's stream.  sagars_profile_read() waits for the recorded events and
 * returns accumulated milliseconds / launch counts per stage (bench.py derives the roofline of the
 * dominant kernel from these). */
SAGARS_API void sagars_profile_enable(int on);
SAGARS_API int sagars_profile_num_stages(void);
SAGARS_API const char* sagars_profile_stage_name(int stage);
SAGARS_API int sagars_profile_read(double* ms_out, int64_t* count_out, int reset);

/* sizeof(sagars_forward_args) / sizeof(sagars_backward_args) as this library was compiled: a binding in another language checks
 * its own struct layout against these before the first call. */
SAGARS_API size_t sagars_sizeof_forward_args(void);
SAGARS_API size_t sagars_sizeof_backward_args(void);

SAGARS_API const char* sagars_last_error(void);
SAGARS_API int sagars_abi_version(void);
/* "sm_100a" -- the only architecture this library carries code for. */
SAGARS_API const char* sagars_arch(void);

#ifdef __cplusplus
}
#endif
#endif /* SAGARS_H_INCLUDED */
