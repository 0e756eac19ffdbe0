// render_forward_kernels.cuh -- the device code of render_forward.cu (see there).  Free of host-side runtime calls so that
// tests/test_render_forward_emulated.py can compile the kernel for the CPU against tests/cuda_emu/ and run it against the oracle.
#pragma once
#include "common.cuh"
#include "cp_async.cuh"

#ifndef SAGARS_DYNAMIC_SMEM
#define SAGARS_DYNAMIC_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#endif

namespace sagars {


constexpr int FWD_BATCH = 64;   // instances staged per pipeline stage

template <int NQ>
struct FwdSmem {
    float4 geo[2][FWD_BATCH][2];        // x, y, cx, cy | cz, opacity, accept_threshold, -
    float4 feat[2][FWD_BATCH][NQ];      // feature rows, zero padded to 4*NQ channels
    uint32_t ids[2][FWD_BATCH];
    float maskv[2][FWD_BATCH];          // DEPTH variant: per-instance mask value
    float depthv[2][FWD_BATCH];         // DEPTH variant: per-instance view depth
};

// issue the asynchronous copies of one batch (ids already in smem)
template <int NQ, bool VEC, bool MD, bool COLOR>
__device__ __forceinline__ void fwd_issue_batch(FwdSmem<NQ>& sm, int stage, int idbuf, int cnt, int K,
                                                const float* __restrict__ geo, const float* __restrict__ features,
                                                const float* __restrict__ mask, const float* __restrict__ depths)
{
    const int tid = threadIdx.x;
    // geometry records: 2 x 16 B per instance
    for (int c = tid; c < cnt * 2; c += TILE_PIX) {
        const int j = c >> 1, h = c & 1;
        const uint32_t id = sm.ids[idbuf][j];
        cp_async16(&sm.geo[stage][j][h], geo + 8 * (size_t)id + 4 * h);
    }
    if (MD) {
        if (tid < cnt) {
            const uint32_t id = sm.ids[idbuf][tid];
            sm.maskv[stage][tid] = mask[id];
            sm.depthv[stage][tid] = depths[id];
        }
    }
    if (!COLOR) return;
    if (VEC) {
        const int nq = K >> 2;   // == NQ or fewer (remaining quads stay zero)
        for (int c = tid; c < cnt * nq; c += TILE_PIX) {
            const int j = c / nq, q = c - j * nq;
            const uint32_t id = sm.ids[idbuf][j];
            cp_async16(&sm.feat[stage][j][q], features + (size_t)id * K + 4 * q);
        }
    } else {
        float* f = reinterpret_cast<float*>(&sm.feat[stage][0][0]);
        for (int c = tid; c < cnt * K; c += TILE_PIX) {
            const int j = c / K, k = c - j * K;
            const uint32_t id = sm.ids[idbuf][j];
            f[j * (4 * NQ) + k] = features[(size_t)id * K + k];
        }
    }
}

// records past the end of the tile's list (up to the next multiple of 4): never accepted (threshold = +inf)
template <int NQ>
__device__ __forceinline__ void fwd_pad_batch(FwdSmem<NQ>& sm, int stage, int cnt)
{
    const int tid = threadIdx.x;
    if (tid >= cnt && tid < FWD_BATCH) {
        sm.geo[stage][tid][0] = make_float4(0.f, 0.f, 0.f, 0.f);
        sm.geo[stage][tid][1] = make_float4(0.f, 0.f, __int_as_float(0x7f800000), 0.f);
    }
}

template <int NQ, bool VEC, bool MD, bool COLOR>
__global__ void __launch_bounds__(TILE_PIX)
render_forward_kernel(const uint2* __restrict__ ranges, const uint32_t* __restrict__ point_list,
                      int W, int H, int K,
                      const float* __restrict__ geo, const float* __restrict__ features,
                      const float* __restrict__ mask, const float* __restrict__ depths, const float* __restrict__ bg,
                      float* __restrict__ final_T, uint32_t* __restrict__ n_contrib,
                      float* __restrict__ out_color, float* __restrict__ out_mask, float* __restrict__ out_depth)
{
    SAGARS_DYNAMIC_SMEM(smem_raw);
    FwdSmem<NQ>& sm = *reinterpret_cast<FwdSmem<NQ>*>(smem_raw);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tiles_x = gridDim.x;
    const uint32_t px = blockIdx.x * TILE_X + (warp & 1) * 8 + (lane & 7);
    const uint32_t py = blockIdx.y * TILE_Y + (warp >> 1) * 4 + (lane >> 3);
    const bool inside = px < (uint32_t)W && py < (uint32_t)H;
    const uint32_t pix_id = (uint32_t)W * py + px;
    float pixx = (float)px, pixy = (float)py;
    // opaque to the optimiser: otherwise nvcc rematerialises both from %ctaid / %tid inside the hot loop
    SAGARS_PIN_F2(pixx, pixy);
    const uint2 range = ranges[blockIdx.y * tiles_x + blockIdx.x];
    const int total = (int)(range.y - range.x);
    const int nbatch = (total + FWD_BATCH - 1) / FWD_BATCH;

    // zero the padded feature channels once (cp.async only ever writes the first K of each row)
    if (!VEC || (K >> 2) < NQ) {
        float* f = reinterpret_cast<float*>(&sm.feat[0][0][0]);
        for (int c = tid; c < 2 * FWD_BATCH * 4 * NQ; c += TILE_PIX) f[c] = 0.f;
    }

    float T = 1.0f;
    uint32_t last_contributor = 0;
    float C[4 * NQ];
#pragma unroll
    for (int k = 0; k < 4 * NQ; k++) C[k] = 0.f;
    float Macc = 0.f, Dacc = 0.f;
    bool done = !inside;

    // prologue: ids(0) -> smem, copies of batch 0, ids(1) -> smem
    if (nbatch > 0) {
        if (tid < min(FWD_BATCH, total)) sm.ids[0][tid] = point_list[range.x + tid];
        __syncthreads();
        fwd_issue_batch<NQ, VEC, MD, COLOR>(sm, 0, 0, min(FWD_BATCH, total), K, geo, features, mask, depths);
        cp_async_commit();
        if (nbatch > 1 && tid < min(FWD_BATCH, total - FWD_BATCH)) sm.ids[1][tid] = point_list[range.x + FWD_BATCH + tid];
        cp_async_wait_all();
        fwd_pad_batch<NQ>(sm, 0, min(FWD_BATCH, total));
        __syncthreads();
    }

    for (int b = 0; b < nbatch; b++) {
        const int stage = b & 1;
        const int cnt = min(FWD_BATCH, total - b * FWD_BATCH);
        // all pixels of the tile saturated -> nothing left to do (block-uniform)
        if (__syncthreads_and(done)) break;

        // (A) start the copies of batch b+1 (its ids were stored one iteration ago)
        if (b + 1 < nbatch) {
            fwd_issue_batch<NQ, VEC, MD, COLOR>(sm, stage ^ 1, (b + 1) & 1, min(FWD_BATCH, total - (b + 1) * FWD_BATCH),
                                         K, geo, features, mask, depths);
            cp_async_commit();
        }
        // (B) ids of batch b+2 into a register
        uint32_t next_id = 0;
        const int rem2 = total - (b + 2) * FWD_BATCH;
        const bool have_next_id = (b + 2 < nbatch) && tid < min(FWD_BATCH, rem2);
        if (have_next_id) next_id = point_list[range.x + (b + 2) * FWD_BATCH + tid];

        // (C) blend batch b
        if (!__all_sync(0xffffffffu, done)) {
            // four splats at a time: independent `power` tests (ILP, one vote per four), accepted ones taken in order.
            // Records beyond the tile's list are sentinels (accept_threshold = +inf): no bounds checks needed.
            const float4* gp = &sm.geo[stage][0][0];
            for (int j0 = 0; j0 < cnt; j0 += 4, gp += 8) {
                float pw[4], op[4];
                bool cd[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const float4 g0 = gp[2 * i];
                    const float4 g1 = gp[2 * i + 1];
                    const float dx = g0.x - pixx, dy = g0.y - pixy;
                    pw[i] = -0.5f * (g0.z * dx * dx + g1.x * dy * dy) - g0.w * dx * dy;
                    cd[i] = !(pw[i] > 0.0f) && (pw[i] >= g1.z);
                    op[i] = g1.y;
                }
                const bool anyc = (cd[0] || cd[1] || cd[2] || cd[3]) && !done;
                if (!__any_sync(0xffffffffu, anyc)) continue;
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    if (cd[i] && !done) {
                        const int j = j0 + i;
                        const float alpha = fminf(0.99f, op[i] * expf(pw[i]));
                        if (!(alpha < 1.0f / 255.0f)) {
                            const float test_T = T * (1 - alpha);
                            if (test_T < 0.0001f) {
                                done = true;
                            } else {
                                if (COLOR) {
#pragma unroll
                                    for (int q = 0; q < NQ; q++) {
                                        const float4 f = sm.feat[stage][j][q];
                                        C[4 * q + 0] += f.x * alpha * T;
                                        C[4 * q + 1] += f.y * alpha * T;
                                        C[4 * q + 2] += f.z * alpha * T;
                                        C[4 * q + 3] += f.w * alpha * T;
                                    }
                                }
                                if (MD) {
                                    Macc += sm.maskv[stage][j] * alpha * T;
                                    Dacc += sm.depthv[stage][j] * alpha * T;
                                }
                                T = test_T;
                                last_contributor = (uint32_t)(b * FWD_BATCH + j + 1);
                            }
                        }
                    }
                }
                if (__all_sync(0xffffffffu, done)) break;   // only reached when some pixel was a candidate
            }
        }

        // (D) publish ids(b+2); wait for batch b+1
        if (have_next_id) sm.ids[b & 1][tid] = next_id;
        cp_async_wait_all();
        if (b + 1 < nbatch) fwd_pad_batch<NQ>(sm, stage ^ 1, min(FWD_BATCH, total - (b + 1) * FWD_BATCH));
        __syncthreads();
    }

    if (inside) {
        final_T[pix_id] = T;
        n_contrib[pix_id] = last_contributor;
        const size_t plane = (size_t)H * W;
        if (COLOR) {
#pragma unroll
            for (int k = 0; k < 4 * NQ; k++)
                if (k < K) out_color[(size_t)k * plane + pix_id] = C[k] + T * bg[k];
        }
        if (MD) {
            out_mask[pix_id] = Macc;
            if (out_depth != nullptr) out_depth[pix_id] = Dacc;
        }
    }
}

}  // namespace sagars
