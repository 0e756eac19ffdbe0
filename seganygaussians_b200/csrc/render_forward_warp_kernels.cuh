// render_forward_warp_kernels.cuh -- the device code of render_forward_warp.cu (see there).  Free of host-side runtime calls
// so that tests/test_warp_kernels_emulated.py can compile it for the CPU against tests/cuda_emu/.
#pragma once
#include "common.cuh"
#include "candidate.cuh"
#include "cp_async.cuh"
#include "mma.cuh"

#ifndef SAGARS_DYNAMIC_SMEM
#define SAGARS_DYNAMIC_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#endif

namespace sagars {


constexpr int FW_WS = 40;    // row stride (words) of the W tile
constexpr int FW_N = 8;      // candidates per group = k extent of one mma step
constexpr int FW_TAB = 40;   // candidate table: up to 7 carried over + 32 new

template <int NQ>
struct FwCfg {
    static constexpr int NQE = NQ < 2 ? 2 : NQ;                 // quads per feature row (power of two)
    static constexpr int ROW = 4 * NQE;                         // padded channel count
    static constexpr int NT = ROW / 8;                          // 8-channel n-tiles
    // row stride of the feature tile (floats): 8 (mod 32) for ROW >= 16, so that the B-fragment reads (lane = (channel fg,
    // candidate ft), address = ft * RS + fg + immediate) hit 32 different banks without any per-row rotation
    static constexpr int RS = (ROW >= 16) ? ROW + 8 : ROW;
};

template <int NQ>
struct FwSmem {
    float rowW[FW_N][FW_WS];              // weight of candidate r for pixel p at r * FW_WS + p (stride 40 = 8 mod 32: the scalar pass
                                          // and the A-fragment reads are both conflict-free with base + immediate addresses)
    float F[FW_N][FwCfg<NQ>::RS];         // gathered feature rows
    float4 ctab[FW_TAB][2];               // candidate records (x, y, cx, cy | cz, opacity, accept_threshold, -), list order
    uint32_t cid[FW_TAB];                 // their Gaussian ids
    float4 stage[2][32][2];               // the next chunk's records, one 32-byte slot per lane (cp.async, double buffered)
};

// NQ : float4 groups covering the K colour channels;  VEC: K % 4 == 0 -> feature rows are read as float4
template <int NQ, bool VEC>
__global__ void __launch_bounds__(32, (NQ <= 8) ? 28 : 12)
render_forward_warp_kernel(const uint2* __restrict__ ranges, const uint32_t* __restrict__ point_list, int W, int H, int K,
                           const float* __restrict__ geo, const float* __restrict__ features, const float* __restrict__ bg,
                           float* __restrict__ final_T, uint32_t* __restrict__ n_contrib, float* __restrict__ out_color)
{
    using Cfg = FwCfg<NQ>;
    constexpr int NQE = Cfg::NQE, ROW = Cfg::ROW, NT = Cfg::NT, RS = Cfg::RS;
    SAGARS_DYNAMIC_SMEM(smem_raw);
    FwSmem<NQ>& sm = *reinterpret_cast<FwSmem<NQ>*>(smem_raw);

    const int lane = threadIdx.x;
    const int tiles_x = (int)(gridDim.x >> 1);
    const uint32_t blk_x0 = blockIdx.x * 8, blk_y0 = blockIdx.y * 4;
    const uint32_t px = blk_x0 + (lane & 7), py = blk_y0 + (lane >> 3);
    const bool inside = px < (uint32_t)W && py < (uint32_t)H;
    const uint32_t pix_id = (uint32_t)W * py + px;
    float pixx = (float)px, pixy = (float)py;
    SAGARS_PIN_F2(pixx, pixy);   // keep nvcc from rematerialising them in the hot loop

    const uint2 range = ranges[(blockIdx.y >> 2) * tiles_x + (blockIdx.x >> 1)];
    const int total = (int)(range.y - range.x);
    const int nchunk = (total + 31) >> 5;

    float T = 1.0f;
    float Tc = inside ? 1.0f : 0.0f;   // 0: this pixel takes no more splats
    uint32_t last_contributor = 0;

    float acc[2][NT][4];
#pragma unroll
    for (int mt = 0; mt < 2; mt++)
#pragma unroll
        for (int nt = 0; nt < NT; nt++) acc[mt][nt][0] = acc[mt][nt][1] = acc[mt][nt][2] = acc[mt][nt][3] = 0.f;

    const int fg = lane >> 2, ft = lane & 3;
    const float bx0 = (float)blk_x0, bx1 = bx0 + 7.f, by0 = (float)blk_y0, by1 = by0 + 3.f;   // block of pixel centres
    const uint32_t lt = (1u << lane) - 1u;
    float* const rowW = &sm.rowW[0][0];
    float* const Ft = &sm.F[0][0];

    // one group: candidates in table slots [gs, gs + m), m <= 8
    auto process_group = [&](int gs, int m) {
        // ---- feature rows of the group: issued now, needed after the scalar loop.  Full float4 rows (K == ROW) are copied
        //      straight into the F tile with cp.async (no registers held across the loop); other K go through registers ----
        constexpr int QR = ROW / 4;
        constexpr int NLD = (FW_N * QR + 31) / 32;
        const bool direct = VEC && K == ROW;      // warp-uniform
        float4 fv[NLD];
#pragma unroll
        for (int l = 0; l < NLD; l++) {
            const int idx = lane + 32 * l;
            fv[l] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (idx < FW_N * QR) {
                const int r = idx / QR, qd = idx - r * QR;
                const uint32_t id = sm.cid[gs + min(r, m - 1)];
                const int c0 = 4 * qd;
                if (direct) {
                    cp_async16(Ft + r * RS + 4 * qd, features + (size_t)id * K + c0);
                } else if (VEC) {
                    if (c0 < K) fv[l] = __ldg(reinterpret_cast<const float4*>(features + (size_t)id * K + c0));
                } else {
                    const float* f = features + (size_t)id * K;
                    if (c0 + 0 < K) fv[l].x = __ldg(f + c0 + 0);
                    if (c0 + 1 < K) fv[l].y = __ldg(f + c0 + 1);
                    if (c0 + 2 < K) fv[l].z = __ldg(f + c0 + 2);
                    if (c0 + 3 < K) fv[l].w = __ldg(f + c0 + 3);
                }
            }
        }
        if (direct) cp_async_commit();
        // The reference's chain as selects (no divergent branch, so the chains of neighbouring candidates interleave).  Tc is the
        // transmittance the chain tests with: it drops to 0 when the pixel saturates (or lies outside the image), after which
        // every test_T is 0 < 1e-4 and nothing is accepted -- no separate `done` flag; T keeps the value the reference reports.
        // A rejected pair computes on garbage (expf of a large or NaN power) and selects nothing.  Full groups (the common
        // case) run fully unrolled: table and W-tile addresses become immediates.
        auto one = [&](int i) {
            const float4 g0 = sm.ctab[gs + i][0];
            const float4 g1 = sm.ctab[gs + i][1];
            const float dx = g0.x - pixx, dy = g0.y - pixy;
            const float pw = -0.5f * (g0.z * dx * dx + g1.x * dy * dy) - g0.w * dx * dy;
            const bool ok = !(pw > 0.0f) && (pw >= g1.z);
            const float alpha = fminf(0.99f, g1.y * expf(pw));
            const bool ok2 = ok && !(alpha < 1.0f / 255.0f);
            const float test_T = Tc * (1 - alpha);
            const bool low = test_T < 0.0001f;
            const bool go = ok2 && !low;
            const float w = go ? alpha * Tc : 0.f;
            T = go ? test_T : T;
            Tc = go ? test_T : ((ok2 && low) ? 0.f : Tc);
            last_contributor = go ? (uint32_t)(__float_as_int(g1.w) + 1) : last_contributor;
            rowW[i * FW_WS + lane] = w;
        };
        if (m == FW_N) {
#pragma unroll
            for (int i = 0; i < FW_N; i++) one(i);
        } else {
#pragma unroll 1
            for (int i = 0; i < FW_N; i++) {
                if (i < m) one(i);
                else rowW[i * FW_WS + lane] = 0.f;
            }
        }
        if (direct) {
            cp_async_wait_all();
        } else {
#pragma unroll
            for (int l = 0; l < NLD; l++) {
                const int idx = lane + 32 * l;
                if (idx < FW_N * QR) {
                    const int r = idx / QR, qd = idx - r * QR;
                    *reinterpret_cast<float4*>(Ft + r * RS + 4 * qd) = fv[l];
                }
            }
        }
        __syncwarp();
        // ---- C (32 pixels x C) += W^T (32 x 8) F (8 x C), 3xTF32 ----
        uint32_t ah[2][4], al[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
            // a0 = (pixel 16 mt + fg, candidate ft), a1 = (pixel + 8, ft), a2 = (pixel, ft + 4), a3 = (pixel + 8, ft + 4)
            const int pa = 16 * mt + fg, pb = pa + 8;
            split_tf32(rowW[ft * FW_WS + pa], ah[mt][0], al[mt][0]);
            split_tf32(rowW[ft * FW_WS + pb], ah[mt][1], al[mt][1]);
            split_tf32(rowW[(ft + 4) * FW_WS + pa], ah[mt][2], al[mt][2]);
            split_tf32(rowW[(ft + 4) * FW_WS + pb], ah[mt][3], al[mt][3]);
        }
#pragma unroll
        for (int nt = 0; nt < NT; nt++) {
            // b0 = (candidate ft, channel 8 nt + fg), b1 = (candidate ft + 4, same channel)
            const int ch = 8 * nt + fg;
            uint32_t bh0, bl0, bh1, bl1;
            split_tf32(Ft[ft * RS + ch], bh0, bl0);
            split_tf32(Ft[(ft + 4) * RS + ch], bh1, bl1);
#pragma unroll
            for (int mt = 0; mt < 2; mt++) {
                mma_16n8k8(acc[mt][nt], al[mt][0], al[mt][1], al[mt][2], al[mt][3], bh0, bh1);
                mma_16n8k8(acc[mt][nt], ah[mt][0], ah[mt][1], ah[mt][2], ah[mt][3], bl0, bl1);
                mma_16n8k8(acc[mt][nt], ah[mt][0], ah[mt][1], ah[mt][2], ah[mt][3], bh0, bh1);
            }
        }
        __syncwarp();   // the tiles and the table slots may be overwritten
    };

    if (nchunk > 0) {
        // list ids run two chunks ahead in registers, records one chunk ahead through a per-lane staging slot (cp.async): nothing
        // of the next chunk occupies registers while the groups of this one are worked on
        int pos_cur = lane;
        uint32_t id_cur = pos_cur < total ? point_list[range.x + pos_cur] : 0u;
        cp_async16(&sm.stage[0][lane][0], geo + 8 * (size_t)id_cur);
        cp_async16(&sm.stage[0][lane][1], geo + 8 * (size_t)id_cur + 4);
        cp_async_commit();
        uint32_t id_nxt = (32 + lane) < total ? point_list[range.x + 32 + lane] : 0u;
        int ntab = 0;   // candidates waiting in table slots [0, ntab)
        for (int c = 0; c < nchunk; c++) {
            if (__all_sync(0xffffffffu, Tc == 0.0f)) { ntab = 0; break; }   // the block is saturated: nothing later can contribute
            cp_async_wait_all();                                          // this lane's own slot: no warp barrier needed
            const float4 r0_cur = sm.stage[c & 1][lane][0];
            const float4 r1_cur = sm.stage[c & 1][lane][1];
            const int pos_nxt = 32 * (c + 1) + lane;
            if (c + 1 < nchunk) {                                         // warp-uniform; lanes past the end copy record 0 (ignored)
                cp_async16(&sm.stage[(c + 1) & 1][lane][0], geo + 8 * (size_t)id_nxt);
                cp_async16(&sm.stage[(c + 1) & 1][lane][1], geo + 8 * (size_t)id_nxt + 4);
                cp_async_commit();
            }
            const int pos_nn = 32 * (c + 2) + lane;
            const uint32_t id_nn = pos_nn < total ? point_list[range.x + pos_nn] : 0u;

            // block-level candidate test (candidate.cuh), lane = splat; survivors join the table in list order
            const bool keep = pos_cur < total && !block_rejects(r0_cur, r1_cur, bx0, bx1, by0, by1);
            const uint32_t km = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int slot = ntab + __popc(km & lt);
                sm.ctab[slot][0] = r0_cur;
                float4 r1p = r1_cur;
                r1p.w = __int_as_float(pos_cur);
                sm.ctab[slot][1] = r1p;
                sm.cid[slot] = id_cur;
            }
            ntab += __popc(km);
            __syncwarp();

            // full groups now, the rest is carried over (the last chunk flushes everything)
            int gs = 0;
            const bool last = (c + 1 == nchunk);
            while (ntab - gs >= FW_N || (last && ntab - gs > 0)) {
                process_group(gs, min(FW_N, ntab - gs));
                gs += FW_N;
            }
            if (gs > 0 && gs < ntab) {   // carry the leftovers (< 8) to the front: sources are slots >= 8, destinations < 7
                const int left = ntab - gs;
                float4 a0, a1;
                uint32_t ci = 0;
                if (lane < left) { a0 = sm.ctab[gs + lane][0]; a1 = sm.ctab[gs + lane][1]; ci = sm.cid[gs + lane]; }
                __syncwarp();
                if (lane < left) { sm.ctab[lane][0] = a0; sm.ctab[lane][1] = a1; sm.cid[lane] = ci; }
                __syncwarp();
            }
            ntab = (gs >= ntab) ? 0 : ntab - gs;

            pos_cur = pos_nxt;
            id_cur = id_nxt;
            id_nxt = id_nn;
        }
        // an early exit can leave carried candidates behind: the saturated block ignores them (they come later in the list)
        (void)ntab;
    }

    // ---- epilogue: accumulator fragments -> planar image ----
    if (inside) {
        final_T[pix_id] = T;
        n_contrib[pix_id] = last_contributor;
    }
    const size_t plane = (size_t)H * W;
#pragma unroll
    for (int mt = 0; mt < 2; mt++) {
        // fragment rows: block pixels 16 mt + fg (image row 2 mt, x = fg) and + 8 (image row 2 mt + 1)
        const float Ta = __shfl_sync(0xffffffffu, T, 16 * mt + fg);
        const float Tb = __shfl_sync(0xffffffffu, T, 16 * mt + fg + 8);
        const uint32_t xa = blk_x0 + fg, ya = blk_y0 + 2 * mt, yb = ya + 1;
        const bool ina = xa < (uint32_t)W && ya < (uint32_t)H, inb = xa < (uint32_t)W && yb < (uint32_t)H;
        const size_t pa = (size_t)W * ya + xa, pb = (size_t)W * yb + xa;
#pragma unroll
        for (int nt = 0; nt < NT; nt++) {
            const int ch = 8 * nt + 2 * ft;
            if (ch < K) {
                const float b = bg[ch];
                if (ina) out_color[(size_t)ch * plane + pa] = acc[mt][nt][0] + Ta * b;
                if (inb) out_color[(size_t)ch * plane + pb] = acc[mt][nt][2] + Tb * b;
            }
            if (ch + 1 < K) {
                const float b = bg[ch + 1];
                if (ina) out_color[(size_t)(ch + 1) * plane + pa] = acc[mt][nt][1] + Ta * b;
                if (inb) out_color[(size_t)(ch + 1) * plane + pb] = acc[mt][nt][3] + Tb * b;
            }
        }
    }
}

}  // namespace sagars
