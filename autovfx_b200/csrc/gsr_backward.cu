// gsr_b200 backward pass.
//
// Replaces CudaRasterizer::Rasterizer::backward (DGR/cuda_rasterizer/rasterizer_impl.cu:343-446):
//   k_blend_backward     <- BACKWARD::render        (backward.cu:415-599)
//   k_gaussian_backward  <- computeCov2DCUDA + BACKWARD::preprocessCUDA (backward.cu:144-274, :346-412,
//                           with the SH backward :20-139 and the scale/rotation backward :278-341)
//
// The per-pixel recursion of the blend backward is the reference's (it must replay the forward's decisions); the per-Gaussian
// chain rule is derived here in matrix form (see sh_grad, geometry_grad, cov3d_grad).  Differences in mechanism:
//   * the reference issues 10 global atomicAdds per contributing (pixel, Gaussian) pair; here each warp
//     (an 8x4 pixel footprint) sums the gradients of a splat over its pixels as moments (see the kernel's
//     comment) and issues one global reduction per (warp, Gaussian, component);
//   * a warp only visits the splats whose footprint-ballot bit is set (the forward's survivor lists);
//   * the two per-Gaussian backward kernels are fused; SH rows are staged through shared memory with
//     coalesced accesses in both directions, and the kernel writes every output row itself (zeros for
//     culled Gaussians) so only the 48 B/Gaussian of atomically accumulated gradients need a memset
//     (the reference zero-fills all 304 B/Gaussian, rasterize_points.cu:158-168).
// Gradient sums are accumulated in a different order than the reference's atomics (which are themselves
// unordered), so parity is to a tolerance, not bitwise.
#include <cstdlib>
#include <type_traits>
#include "gsr_common.cuh"
#include "gsr_packed.cuh"

namespace gsr {

__device__ __forceinline__ float4 lds128b(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts128b(uint32_t a, const float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// -----------------------------------------------------------------------------------------------------------------------
// Blend backward over the footprint lists.
//
// Like the forward blend (gsr_blend.cu) one WARP owns an 8x4-pixel footprint and walks that footprint's own survivors — the
// entries of the tile's sorted list whose ballot bit says the splat can reach alpha >= 1/255 inside the footprint — this time
// from the back (position n_contrib of the furthest pixel) to the front.  No block-level staging, no barrier, no cull.
//
// Per batch of 16 survivors the work is split into two phases with different lane roles:
//   phase 1, lane = pixel: the per-pixel recursion (it has to replay the forward's decisions, forward.cu:330-366, so `power`
//            is evaluated with the forward's instruction sequence and alpha with the same expf).  The reference carries one
//            running "colour behind" per channel (backward.cu:533-562); everything downstream only needs its inner product
//            with the pixel's loss gradient, so the five channel recursions collapse into ONE scalar recursion
//                D_k = dL/dC . c_k + dL/dDepth * depth_k + dL/dAlpha,      R <- alpha_last * D_last + (1 - alpha_last) * R,
//                dL/dalpha_k = (D_k - R) * T_k - T_final / (1 - alpha_k) * (bg . dL/dC).
//            The phase leaves two numbers per (survivor, pixel) in shared memory: w = alpha_k T_k and s = G_k dL/dalpha_k.
//   phase 2, lane = survivor (x half of the pixels): every gradient of the splat is a moment of w or s over the footprint,
//                dL/dcolour = sum w dL/dC,   dL/ddepth = sum w dL/dDepth,   dL/dopacity = sum s,
//                dL/dmean2D = -o (W/2, H/2) * (a Sx + b Sy, b Sx + c Sy),   dL/dconic = -o/2 (Sxx, Sxy, Syy),
//            with S* = sum s {dx, dy, dx^2, dx dy, dy^2}.  The lane accumulates them over 16 pixels with plain FMAs — no
//            shuffle reduction per (splat, component) — the two halves meet in one exchange, and ten lanes-wide reductions
//            (RED.ADD.F32) per 16 splats go to global memory.
//
// EXTRA: the backward of gsr_forward_multi, whose second colour set e_k is blended with the same weights over the same
// background.  That second image is one more linear term of the loss, so the recursion stays scalar:
//     D_k += dL/dE . e_k,   tfbg -= T_final (bg . dL/dE),   dL/dextra = sum w dL/dE  (three more moments in phase 2),
// and every geometric gradient comes out as the sum of the two single-image backward passes (up to summation order).
// -----------------------------------------------------------------------------------------------------------------------
struct BwdArgs {
    const uint2* ranges; const uint32_t* point_list; const float4* records; const uint32_t* bal;
    int W, H, gx;
    const float *bg, *accum_alphas; const uint32_t* n_contrib;
    const float *dL_dpixels, *dL_dpixel_depths, *dL_dpixel_alphas;
    float *dL_dmean2D /*[P,3]*/, *dL_dconic /*[P,4]*/, *dL_dopacity, *dL_dcolors /*[P,3]*/, *dL_ddepths;
    // EXTRA only (appended, so that the offsets of the fields above stay what the single-image kernel reads)
    const float* extra /*[P,3]*/; const float* dL_dpixel_extras /*[3,H,W]*/; float* dL_dextra /*[P,3]*/;
};

constexpr int BWL_WARPS = 4;
constexpr float BWL_LOG2E = 1.4426950408889634f;
struct BwlCfg {
    // one gather of 32 survivors, two per 112-byte pair so that phase 1 runs both on the halves of packed fp32 registers:
    // {x0,x1,y0,y1 | a0,a1,-b0,-b1 | c0,c1,o0,o1 | r0,r1,g0,g1 | b0,b1,depth0,depth1 | pos0,pos1,-,- | pad}, then the 32 ids
    static constexpr int PAIRB = 112;
    static constexpr int REC = 16 * PAIRB + 32 * 4;
    static constexpr int WROW = 66;            // words per (w, s) row: 32 pixels x 2, + 2 so that rows start 2 banks apart
    static constexpr int WS = 16 * WROW * 4;   // one 16-survivor batch
    static constexpr int DLP = 32 * 16;        // the footprint's loss gradients {dL/dC.rgb, dL/dDepth} per pixel
    static constexpr int RING = 128;           // expanded survivor positions (u32)
    static constexpr int WB = REC + WS + DLP + 4 * RING;
};
// EXTRA: the pair record keeps its size — its last 24 bytes hold the two splats' extra colours
// {.. | pos0,pos1,e0_0,e0_1 | e1_0,e1_1,e2_0,e2_1} — and a pixel's loss-gradient row grows to 32 bytes
// {dL/dC.rgb, dL/dDepth | dL/dE.rgb, 0}.
struct BwlCfgExtra : BwlCfg {
    static constexpr int DLP = 32 * 32;
    static constexpr int WB = REC + WS + DLP + 4 * RING;
};

__device__ __forceinline__ void sts64b(uint32_t a, float x, float y) {
    asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(a), "f"(x), "f"(y) : "memory");
}
__device__ __forceinline__ float lds32b(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float2 lds64b(uint32_t a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
    return v;
}

template <int OCC, bool EXTRA = false>
__global__ void __launch_bounds__(BWL_WARPS * 32, OCC) k_blend_backward(const BwdArgs a) {
    typedef typename std::conditional<EXTRA, BwlCfgExtra, BwlCfg>::type Cfg;
    constexpr uint32_t DLROW = Cfg::DLP / 32;  // bytes of one pixel's loss-gradient row
    constexpr int PARTS = GSR_FOOTS / BWL_WARPS;
    constexpr int RING = Cfg::RING;
    __shared__ __align__(16) unsigned char sm[BWL_WARPS * Cfg::WB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tx = blockIdx.x / PARTS, part = blockIdx.x - tx * PARTS;
    const int f = part * BWL_WARPS + warp;
    const int tile = blockIdx.y * a.gx + tx;
    const int X0 = tx * GSR_TILE + (f & 1) * 8, Y0 = blockIdx.y * GSR_TILE + (f >> 1) * 4;
    const int pxi = X0 + (lane & 7), pyi = Y0 + (lane >> 3);
    const bool inside = pxi < a.W && pyi < a.H;
    const float pixx = (float)pxi, pixy = (float)pyi;
    const uint32_t rec_base = (uint32_t)__cvta_generic_to_shared(sm) + (uint32_t)warp * Cfg::WB;
    const uint32_t id_base = rec_base + 16 * Cfg::PAIRB, ws_base = rec_base + Cfg::REC, dlp_base = ws_base + Cfg::WS;
    uint32_t* ring = reinterpret_cast<uint32_t*>(sm + (size_t)warp * Cfg::WB + Cfg::REC + Cfg::WS + Cfg::DLP);

    const uint2 rg = a.ranges[tile];
    if (rg.y == rg.x) return;
    const size_t pid = (size_t)a.W * pyi + pxi, HW = (size_t)a.H * a.W;
    const uint32_t last_contributor = inside ? a.n_contrib[pid] : 0u;  // 1-based position of the pixel's last contributor
    uint32_t warp_last = last_contributor;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) warp_last = max(warp_last, __shfl_xor_sync(GSR_FULL, warp_last, o));
    if (warp_last == 0u) return;  // nothing contributed anywhere in this footprint

    // ---- pixel state (phase 1) ----
    float dLp0 = 0, dLp1 = 0, dLp2 = 0, dLd = 0, dLa = 0, T_final = 0;
    float dLe0 = 0, dLe1 = 0, dLe2 = 0;  // dL/dE (EXTRA)
    if (inside) {
        T_final = 1.0f - a.accum_alphas[pid];
        dLp0 = a.dL_dpixels[pid]; dLp1 = a.dL_dpixels[HW + pid]; dLp2 = a.dL_dpixels[2 * HW + pid];
        dLd = a.dL_dpixel_depths[pid];
        dLa = a.dL_dpixel_alphas[pid];
        if constexpr (EXTRA) { dLe0 = a.dL_dpixel_extras[pid]; dLe1 = a.dL_dpixel_extras[HW + pid]; dLe2 = a.dL_dpixel_extras[2 * HW + pid]; }
    }
    sts128b(dlp_base + (uint32_t)lane * DLROW, make_float4(dLp0, dLp1, dLp2, dLd));
    if constexpr (EXTRA) sts128b(dlp_base + (uint32_t)lane * DLROW + 16, make_float4(dLe0, dLe1, dLe2, 0.0f));
    float T = T_final;
    // -T_final (bg . dL/dC), backward.cu:566-572; EXTRA: the second image is blended over the same background
    const float tfbg = EXTRA ? -T_final * (a.bg[0] * dLp0 + a.bg[1] * dLp1 + a.bg[2] * dLp2 + (a.bg[0] * dLe0 + a.bg[1] * dLe1 + a.bg[2] * dLe2))
                             : -T_final * (a.bg[0] * dLp0 + a.bg[1] * dLp1 + a.bg[2] * dLp2);
    float Rn = 0.f;  // the "behind" term of the recursion for the next splat that hits
    const f32x2 npx2 = pk2(-pixx, -pixx), npy2 = pk2(-pixy, -pixy);

    const uint32_t* __restrict__ balcol = a.bal + bal_row_base(rg.x, tile) * GSR_FOOTS + f;
    const uint32_t* __restrict__ plist = a.point_list + rg.x;

    // ---- survivor stream, back to front: stream index 0 is the set bit with the highest list position <= warp_last - 1 ----
    const uint32_t pmax = warp_last - 1u, row_top = pmax >> 5;
    const uint32_t nblocks = (row_top + 32u) >> 5;  // 32-row blocks, block b holds rows row_top - 32 b - lane
    uint32_t rbits = 0, roff = 0, rrow = 0, sbase = 0, nblk = 0, filled = 0, consumed = 0;
    bool block_open = false;
    auto col_word = [&](uint32_t blk) -> uint32_t {
        const uint32_t back = blk * 32u + (uint32_t)lane;
        if (back > row_top) return 0u;
        uint32_t w = balcol[(size_t)(row_top - back) * GSR_FOOTS];
        if (back == 0u) w &= (2u << (pmax & 31u)) - 1u;  // entries behind the last contributor of every pixel
        return w;
    };
    uint32_t wnext = col_word(0);
    auto refill = [&]() {
        const uint32_t limit = consumed + RING;
        while (true) {
            if (!block_open) {
                if (nblk == nblocks) break;
                rbits = wnext;
                rrow = (row_top - min(row_top, nblk * 32u + (uint32_t)lane)) * 32u;
                nblk++;
                wnext = nblk < nblocks ? col_word(nblk) : 0u;
                const uint32_t c = (uint32_t)__popc(rbits);
                uint32_t incl = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t v = __shfl_up_sync(GSR_FULL, incl, o);
                    if (lane >= o) incl += v;
                }
                roff = sbase + incl - c;
                sbase += __shfl_sync(GSR_FULL, incl, 31);
                block_open = true;
            }
            while (rbits && roff < limit) {
                const uint32_t bit = 31u - (uint32_t)__clz(rbits);
                rbits ^= 1u << bit;
                ring[roff & (RING - 1)] = rrow + bit;
                roff++;
            }
            if (__any_sync(GSR_FULL, rbits != 0u)) { filled = limit; return; }
            block_open = false;
            filled = sbase;
            if (filled >= limit) return;
        }
        filled = sbase;
    };

    float4 ra = make_float4(0, 0, 0, 0), rb = ra, rc = ra;
    float re0 = 0, re1 = 0, re2 = 0;  // the survivor's extra colour (EXTRA)
    uint32_t pos_c = 0, id_c = 0, pos1 = 0, id1 = 0;
    refill();
    __syncwarp();
    if (consumed + lane < filled) {
        pos_c = ring[(consumed + lane) & (RING - 1)];
        id_c = plist[pos_c];
        const float4* r = a.records + 3 * (size_t)id_c;
        ra = r[0]; rb = r[1]; rc = r[2];
        if constexpr (EXTRA) { const float* e = a.extra + 3 * (size_t)id_c; re0 = e[0]; re1 = e[1]; re2 = e[2]; }
    }
    if (consumed + 32 + lane < filled) { pos1 = ring[(consumed + 32 + lane) & (RING - 1)]; id1 = plist[pos1]; }

    const float half_w = 0.5f * a.W, half_h = 0.5f * a.H;  // d(pixel)/d(ndc), backward.cu:488-489
    const int j = lane & 15, h = lane >> 4;
    while (consumed < filled) {
        const int cnt = (int)min(32u, filled - consumed);
        {
            const uint32_t qa = rec_base + (uint32_t)(lane >> 1) * Cfg::PAIRB + (uint32_t)(lane & 1) * 4;
            if (lane < cnt) {
                sts32(qa, ra.x); sts32(qa + 8, ra.y); sts32(qa + 16, ra.z); sts32(qa + 24, -ra.w);
                sts32(qa + 32, rb.x); sts32(qa + 40, rb.y);
                sts32(qa + 48, rc.x); sts32(qa + 56, rc.y); sts32(qa + 64, rc.z); sts32(qa + 72, rb.z);
                sts32(qa + 80, __uint_as_float(pos_c + 1u));  // 1-based position in the tile's list, compared with n_contrib
                if constexpr (EXTRA) { sts32(qa + 88, re0); sts32(qa + 96, re1); sts32(qa + 104, re2); }
                sts32(id_base + (uint32_t)lane * 4, __uint_as_float(id_c));
            } else if (lane == cnt && (cnt & 1)) {  // completes the last pair of an odd batch: a splat behind every pixel's last contributor
                sts32(qa, 0.f); sts32(qa + 8, 0.f); sts32(qa + 16, 0.f); sts32(qa + 24, 0.f); sts32(qa + 32, 0.f); sts32(qa + 40, 0.f);
                sts32(qa + 48, 0.f); sts32(qa + 56, 0.f); sts32(qa + 64, 0.f); sts32(qa + 72, 0.f);
                sts32(qa + 80, __uint_as_float(0xffffffffu));
                if constexpr (EXTRA) { sts32(qa + 88, 0.f); sts32(qa + 96, 0.f); sts32(qa + 104, 0.f); }
            }
        }
        consumed += (uint32_t)cnt;
        if (filled - consumed < 64u && (block_open || nblk < nblocks)) refill();
        __syncwarp();
        pos_c = pos1; id_c = id1;
        if (consumed + lane < filled) {
            const float4* r = a.records + 3 * (size_t)id_c;
            ra = r[0]; rb = r[1]; rc = r[2];
            if constexpr (EXTRA) { const float* e = a.extra + 3 * (size_t)id_c; re0 = e[0]; re1 = e[1]; re2 = e[2]; }
        }
        if (consumed + 32 + lane < filled) { pos1 = ring[(consumed + 32 + lane) & (RING - 1)]; id1 = plist[pos1]; }

        for (int sub = 0; sub < cnt; sub += 16) {
            const int c16 = min(16, cnt - sub);
            // ---- phase 1: lane = pixel ----
            // Straight-line code (a splat that does not contribute runs the recursion with alpha = 0, which leaves the state
            // unchanged) so that the independent front parts of consecutive splats overlap the serial T / R chain.
            // G = exp(power) comes from one MUFU (relative error < 1.2e-6 against expf).  The only place that needs more is the
            // forward's skip decision alpha < 1/255: if any evaluation of the batch lands inside the error band, the warp restores
            // its state and repeats the batch with the forward's own expf (a fraction of a percent of the batches).
            bool anyc = false;
            auto phase1 = [&](auto exact_tag) -> bool {
                constexpr bool EXACT = decltype(exact_tag)::value;
                bool near = false;
                uint32_t qa = rec_base + (uint32_t)(sub >> 1) * Cfg::PAIRB, wa = ws_base + (uint32_t)lane * 8;
                // the recursion: T, Rn and the (w, s) pair of this (splat, pixel)
                auto step = [&](float G, float alpha, bool hit, float D, float& w, float& sv) {
                    const float a_eff = hit ? alpha : 0.0f;
                    const float om = 1.0f - a_eff;  // in [0.01, 1]: the approximate reciprocal (1 ulp, exact for 1) needs no special cases
                    float rcp;
                    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rcp) : "f"(om));
                    T *= rcp;                       // transmittance in front of this splat
                    w = a_eff * T;
                    const float dL_dalpha = fmaf(tfbg, rcp, (D - Rn) * T);
                    sv = hit ? G * dL_dalpha : 0.0f;
                    Rn = hit ? fmaf(alpha, D, om * Rn) : Rn;
                    anyc |= hit;
                };
                const f32x2 mhalf2 = pk2(-0.5f, -0.5f), l2e2 = pk2(BWL_LOG2E, BWL_LOG2E);
                const f32x2 g0 = pk2(dLp0, dLp0), g1 = pk2(dLp1, dLp1), g2 = pk2(dLp2, dLp2), gd2 = pk2(dLd, dLd), ga2 = pk2(dLa, dLa);
                for (int k = 0; k < c16; k += 2, qa += Cfg::PAIRB, wa += 2 * Cfg::WROW * 4) {  // two splats per iteration (an odd batch ends on a dummy)
                    const float4 L0 = lds128b(qa), L1 = lds128b(qa + 16), L2 = lds128b(qa + 32), L3 = lds128b(qa + 48), L4 = lds128b(qa + 64);
                    float2 P5;
                    f32x2 Dbase = ga2;  // the part of D that is not dL/dC . c + dL/dDepth depth
                    if constexpr (EXTRA) {
                        const float4 L5 = lds128b(qa + 80), L6 = lds128b(qa + 96);
                        P5 = make_float2(L5.x, L5.y);
                        Dbase = fma2(pk2(L5.z, L5.w), pk2(dLe0, dLe0), fma2(pk2(L6.x, L6.y), pk2(dLe1, dLe1), fma2(pk2(L6.z, L6.w), pk2(dLe2, dLe2), ga2)));
                    } else {
                        P5 = lds64b(qa + 80);
                    }
                    // everything that does not depend on the pixel's running state, both splats in the halves of packed registers.
                    // `power` with the forward's rounding sequence (gsr_blend.cu): the decisions below replay the forward's
                    const f32x2 dx = add2(pk2(L0.x, L0.y), npx2), dy = add2(pk2(L0.z, L0.w), npy2);
                    const f32x2 t1 = mul2(pk2(L2.x, L2.y), dy), t3 = mul2(pk2(L1.x, L1.y), dx), t2 = mul2(pk2(L1.z, L1.w), dx);
                    const f32x2 t4 = mul2(dy, t1), t5 = mul2(dy, t2), t6 = fma2(dx, t3, t4);
                    const f32x2 pw = fma2(t6, mhalf2, t5);
                    float p0, p1, G0, G1;
                    upk2(pw, p0, p1);
                    if (EXACT) { G0 = exp(p0); G1 = exp(p1); }
                    else {
                        float e0, e1;
                        upk2(mul2(pw, l2e2), e0, e1);
                        G0 = ex2_approx(e0); G1 = ex2_approx(e1);
                    }
                    float oG0, oG1;
                    upk2(mul2(pk2(L2.z, L2.w), pk2(G0, G1)), oG0, oG1);
                    if (!EXACT) near |= fabsf(fmaf(oG0, 255.0f, -1.0f)) < 8.0e-6f || fabsf(fmaf(oG1, 255.0f, -1.0f)) < 8.0e-6f;
                    const float al0 = min(0.99f, oG0), al1 = min(0.99f, oG1);
                    const bool h0 = __float_as_uint(P5.x) <= last_contributor && !(p0 > 0.0f) && !(al0 < 1.0f / 255.0f);
                    const bool h1 = __float_as_uint(P5.y) <= last_contributor && !(p1 > 0.0f) && !(al1 < 1.0f / 255.0f);
                    float D0, D1;
                    upk2(fma2(pk2(L3.x, L3.y), g0, fma2(pk2(L3.z, L3.w), g1, fma2(pk2(L4.x, L4.y), g2, fma2(pk2(L4.z, L4.w), gd2, Dbase)))), D0, D1);
                    float w0, w1, s0, s1;
                    step(G0, al0, h0, D0, w0, s0);
                    step(G1, al1, h1, D1, w1, s1);
                    sts64b(wa, w0, s0);
                    sts64b(wa + Cfg::WROW * 4, w1, s1);
                }
                return near;
            };
            {
                const float T0 = T, R0 = Rn;
                if (__any_sync(GSR_FULL, phase1(std::false_type()))) {
                    T = T0; Rn = R0;
                    anyc = false;
                    phase1(std::true_type());
                }
            }
            const bool anyw = __any_sync(GSR_FULL, anyc);
            __syncwarp();
            // ---- phase 2: lane = (survivor j, pixel half h) ----
            if (anyw) {
                // packed fp32: (colour r, g), (colour b, depth), (Sx, Sy) and (Sxx, Syy) live in register pairs
                f32x2 G01 = pk2(0.f, 0.f), G2D = G01, SXY = G01, SQ = G01;
                f32x2 E01 = G01;  // EXTRA: sum w dL/dE (r, g); E2 holds b
                float S0 = 0, Sxy = 0, E2 = 0;
                float ca = 0, cb = 0, cc = 0, op = 0;
                uint32_t gid = 0;
                const bool mine = j < c16;
                if (mine) {
                    const uint32_t sa = rec_base + (uint32_t)((sub + j) >> 1) * Cfg::PAIRB + (uint32_t)((sub + j) & 1) * 4;
                    gid = __float_as_uint(lds32b(id_base + (uint32_t)(sub + j) * 4));
                    ca = lds32b(sa + 16); cb = -lds32b(sa + 24); cc = lds32b(sa + 32); op = lds32b(sa + 40);
                    const float dx0 = lds32b(sa) - (float)X0, dy0 = lds32b(sa + 8) - (float)(Y0 + 2 * h);
                    const uint32_t wr = ws_base + (uint32_t)(j * Cfg::WROW + 32 * h) * 4, dr = dlp_base + (uint32_t)h * (16 * DLROW);
#pragma unroll 1
                    for (int q = 0; q < 4; q++) {  // four pixels at a time: row q >> 1 of the half, columns 4 (q & 1) ..
                        const f32x2 dq = pk2(dx0 - (float)(4 * (q & 1)), dy0 - (float)(q >> 1));
#pragma unroll
                        for (int c = 0; c < 4; c++) {
                            const float2 ws2 = lds64b(wr + (uint32_t)(q * 4 + c) * 8);
                            const float4 dl = lds128b(dr + (uint32_t)(q * 4 + c) * DLROW);
                            const f32x2 dxy = c ? add2(dq, pk2(-(float)c, 0.0f)) : dq;
                            const f32x2 ww = pk2(ws2.x, ws2.x), ss = pk2(ws2.y, ws2.y);
                            G01 = fma2(ww, pk2(dl.x, dl.y), G01);
                            G2D = fma2(ww, pk2(dl.z, dl.w), G2D);
                            if constexpr (EXTRA) {
                                const float4 de = lds128b(dr + (uint32_t)(q * 4 + c) * DLROW + 16);
                                E01 = fma2(ww, pk2(de.x, de.y), E01);
                                E2 = fmaf(ws2.x, de.z, E2);
                            }
                            const f32x2 sxy = mul2(ss, dxy);  // s (dx, dy)
                            SXY = add2(SXY, sxy);
                            SQ = fma2(sxy, dxy, SQ);          // s (dx^2, dy^2)
                            float sx, sy_, dx_, dy;
                            upk2(sxy, sx, sy_);
                            upk2(dxy, dx_, dy);
                            Sxy = fmaf(sx, dy, Sxy);
                            S0 += ws2.y;
                        }
                    }
                }
                float gc0, gc1, gc2, gd, Sx, Sy, Sxx, Syy;
                upk2(G01, gc0, gc1); upk2(G2D, gc2, gd); upk2(SXY, Sx, Sy); upk2(SQ, Sxx, Syy);
                // the two halves of the footprint meet
                gc0 += __shfl_xor_sync(GSR_FULL, gc0, 16); gc1 += __shfl_xor_sync(GSR_FULL, gc1, 16);
                gc2 += __shfl_xor_sync(GSR_FULL, gc2, 16); gd += __shfl_xor_sync(GSR_FULL, gd, 16);
                S0 += __shfl_xor_sync(GSR_FULL, S0, 16); Sx += __shfl_xor_sync(GSR_FULL, Sx, 16); Sy += __shfl_xor_sync(GSR_FULL, Sy, 16);
                Sxx += __shfl_xor_sync(GSR_FULL, Sxx, 16); Sxy += __shfl_xor_sync(GSR_FULL, Sxy, 16); Syy += __shfl_xor_sync(GSR_FULL, Syy, 16);
                float ge0 = 0, ge1 = 0;
                if constexpr (EXTRA) {
                    upk2(E01, ge0, ge1);
                    ge0 += __shfl_xor_sync(GSR_FULL, ge0, 16); ge1 += __shfl_xor_sync(GSR_FULL, ge1, 16); E2 += __shfl_xor_sync(GSR_FULL, E2, 16);
                }
                if (mine) {
                    // half 0 sends colour, depth, mean2D.x; half 1 mean2D.y, conic (xx, xy, yy), opacity
                    const float nop = -op;
                    const float v0 = h ? nop * half_h * fmaf(cb, Sx, cc * Sy) : gc0;
                    const float v1 = h ? 0.5f * nop * Sxx : gc1;
                    const float v2 = h ? 0.5f * nop * Sxy : gc2;
                    const float v3 = h ? 0.5f * nop * Syy : gd;
                    const float v4 = h ? S0 : nop * half_w * fmaf(ca, Sx, cb * Sy);
                    float* const p0 = h ? a.dL_dmean2D + 3 * (size_t)gid + 1 : a.dL_dcolors + 3 * (size_t)gid;
                    float* const p1 = h ? a.dL_dconic + 4 * (size_t)gid : a.dL_dcolors + 3 * (size_t)gid + 1;
                    float* const p2 = h ? a.dL_dconic + 4 * (size_t)gid + 1 : a.dL_dcolors + 3 * (size_t)gid + 2;
                    float* const p3 = h ? a.dL_dconic + 4 * (size_t)gid + 3 : a.dL_ddepths + gid;
                    float* const p4 = h ? a.dL_dopacity + gid : a.dL_dmean2D + 3 * (size_t)gid;
                    if (v0 != 0.0f) atomicAdd(p0, v0);
                    if (v1 != 0.0f) atomicAdd(p1, v1);
                    if (v2 != 0.0f) atomicAdd(p2, v2);
                    if (v3 != 0.0f) atomicAdd(p3, v3);
                    if (v4 != 0.0f) atomicAdd(p4, v4);
                    if constexpr (EXTRA) {  // half 0 sends extra r, g; half 1 extra b
                        float* const pe = a.dL_dextra + 3 * (size_t)gid + (h ? 2 : 0);
                        const float e0 = h ? E2 : ge0;
                        if (e0 != 0.0f) atomicAdd(pe, e0);
                        if (!h && ge1 != 0.0f) atomicAdd(pe + 1, ge1);
                    }
                }
            }
            __syncwarp();  // the (w, s) rows and, after the second batch, the staged records are free again
        }
    }
}

// =====================================================================================================
// per-Gaussian backward (fused computeCov2DCUDA + preprocessCUDA backward)
// =====================================================================================================
struct GBParams {
    int P, D, M, W, H;
    float scale_modifier, tanfovx, tanfovy, h_x, h_y;
    const float *means3D, *shs, *scales, *rotations, *cov3Ds, *view, *proj, *campos;
    const int* radii;
    const uint8_t* clamped;
    const float *dL_dmean2D, *dL_dconic, *dL_dcolor, *dL_ddepth;
    float *dL_dmeans3D, *dL_dcov3D, *dL_dsh, *dL_dscale, *dL_drot;
};

constexpr int GB_THREADS = 128;
constexpr int GB_STRIDE = 49;  // 48 SH floats per row, odd stride -> conflict-free

// ---- SH colour backward ------------------------------------------------------------------------------------------
// rgb_c = 0.5 + sum_k Y_k(d) sh[k][c] with d = (pos - campos) / |pos - campos| (forward.cu:20-71).  Two results:
//   * dL/dsh[k][c] = Y_k(d) g_c, written over the staged row (coefficients beyond the active degree get 0);
//   * dL/dpos: the three channels are contracted FIRST, u_k = sum_c g_c sh[k][c] (one scalar per basis function), so the
//     gradient of the basis is evaluated once instead of once per channel: dL/dd = sum_k u_k grad Y_k(d), and the
//     normalisation contributes the projector (I - d d^T) / |pos - campos|.
// g_c is the colour gradient with the channels the forward clamped at 0 masked out (clamp_bits, forward.cu:63-70).
__device__ float3 sh_grad(int deg, float* sh, float3 pos, const float* campos, unsigned clamp_bits, float3 dL_dcolor) {
    const float vx = pos.x - campos[0], vy = pos.y - campos[1], vz = pos.z - campos[2];
    const float inv_len = 1.0f / sqrtf(vx * vx + vy * vy + vz * vz);
    const float x = vx * inv_len, y = vy * inv_len, z = vz * inv_len;
    const float g[3] = {(clamp_bits & 1u) ? 0.f : dL_dcolor.x, (clamp_bits & 2u) ? 0.f : dL_dcolor.y, (clamp_bits & 4u) ? 0.f : dL_dcolor.z};
    const int ncoef = (deg + 1) * (deg + 1);
    const float xx = x * x, yy = y * y, zz = z * z;
    // basis values Y_k(d) (real SH up to degree 3, the constants of auxiliary.h:22-39)
    float Y[16];
    Y[0] = SH_C0;
    Y[1] = -SH_C1 * y; Y[2] = SH_C1 * z; Y[3] = -SH_C1 * x;
    const float q = 2.f * zz - xx - yy, r4 = 4.f * zz - xx - yy, dxy = xx - yy;
    Y[4] = SH_C2_0 * x * y; Y[5] = SH_C2_1 * y * z; Y[6] = SH_C2_2 * q; Y[7] = SH_C2_3 * x * z; Y[8] = SH_C2_4 * dxy;
    Y[9] = SH_C3_0 * y * (3.f * xx - yy); Y[10] = SH_C3_1 * x * y * z; Y[11] = SH_C3_2 * y * r4;
    Y[12] = SH_C3_3 * z * (q - 2.f * (xx + yy)); Y[13] = SH_C3_4 * x * r4; Y[14] = SH_C3_5 * z * dxy; Y[15] = SH_C3_6 * x * (xx - 3.f * yy);
    // channel contraction u_k, then the row is overwritten with dL/dsh
    float u[16];
#pragma unroll
    for (int k = 0; k < 16; k++) {
        float* row = sh + 3 * k;
        u[k] = k < ncoef ? g[0] * row[0] + g[1] * row[1] + g[2] * row[2] : 0.f;
        const float yk = k < ncoef ? Y[k] : 0.f;
        row[0] = yk * g[0]; row[1] = yk * g[1]; row[2] = yk * g[2];
    }
    // dL/dd = sum_k u_k grad Y_k  (u_k = 0 beyond the active degree, so no branches are needed)
    float gx = -SH_C1 * u[3], gy = -SH_C1 * u[1], gz = SH_C1 * u[2];
    gx += SH_C2_0 * y * u[4] - 2.f * SH_C2_2 * x * u[6] + SH_C2_3 * z * u[7] + 2.f * SH_C2_4 * x * u[8];
    gy += SH_C2_0 * x * u[4] + SH_C2_1 * z * u[5] - 2.f * SH_C2_2 * y * u[6] - 2.f * SH_C2_4 * y * u[8];
    gz += SH_C2_1 * y * u[5] + 4.f * SH_C2_2 * z * u[6] + SH_C2_3 * x * u[7];
    const float xy = x * y, yz = y * z, xz = x * z;
    gx += 6.f * SH_C3_0 * xy * u[9] + SH_C3_1 * yz * u[10] - 2.f * SH_C3_2 * xy * u[11] - 6.f * SH_C3_3 * xz * u[12] +
          SH_C3_4 * (r4 - 2.f * xx) * u[13] + 2.f * SH_C3_5 * xz * u[14] + 3.f * SH_C3_6 * dxy * u[15];
    gy += 3.f * SH_C3_0 * dxy * u[9] + SH_C3_1 * xz * u[10] + SH_C3_2 * (r4 - 2.f * yy) * u[11] - 6.f * SH_C3_3 * yz * u[12] -
          2.f * SH_C3_4 * xy * u[13] - 2.f * SH_C3_5 * yz * u[14] - 6.f * SH_C3_6 * xy * u[15];
    gz += SH_C3_1 * xy * u[10] + 8.f * SH_C3_2 * yz * u[11] + 3.f * SH_C3_3 * q * u[12] + 8.f * SH_C3_4 * xz * u[13] + SH_C3_5 * dxy * u[14];
    // through d = v / |v|:  (I - d d^T) grad / |v|
    const float along = x * gx + y * gy + z * gz;
    return make_float3((gx - x * along) * inv_len, (gy - y * along) * inv_len, (gz - z * along) * inv_len);
}

// ---- geometry backward -------------------------------------------------------------------------------------------
// Forward chain (forward.cu:74-152, 196-237):  t = W m + w0 (view space, W[k][j] = view[4 j + k]);  (u, v) = t.xy clamped to
// +-1.3 tan(fov) t.z;  A = J W with J = [[fx/tz, 0, -fx u/tz^2], [0, fy/tz, -fy v/tz^2]] (2x3);  S = A Sigma A^T + 0.3 I (2x2);
// conic K = adj(S) / det S.   Given the symmetric gradient G of K (dL_dconic holds G00, G01, -, G11 with G01 the gradient of
// ONE off-diagonal entry):
//     dL/dS     = -q adj(S) G adj(S),  q = 1 / (det^2 + 1e-7)   (the reference regularises 1/det^2 this way, backward.cu:203)
//     dL/dSigma = A^T H A                (H = dL/dS; the six outputs double the off-diagonal entries, each stands for two)
//     dL/dA     = 2 H A Sigma
//     dL/dJ     = (dL/dA) W^T, only J00, J02, J11, J12 are functions of t
// and from the screen position (ndc = P^T m / w) and the view-space depth the remaining two terms of dL/dm.
struct GeoGrad {
    float3 dmean;
    float dcov[6];
};
__device__ __forceinline__ GeoGrad geometry_grad(const float3 m, const float* c3, const float* view, const float* proj, float fx, float fy,
                                                 float limx, float limy, float G00, float G01, float G11, float d2x, float d2y, float ddepth) {
    GeoGrad o;
    // view-space position and the clamped image-plane coordinates
    const float tx = view[0] * m.x + view[4] * m.y + view[8] * m.z + view[12];
    const float ty = view[1] * m.x + view[5] * m.y + view[9] * m.z + view[13];
    const float tz = view[2] * m.x + view[6] * m.y + view[10] * m.z + view[14];
    const float itz = 1.f / tz;
    const float rx = tx * itz, ry = ty * itz;
    const bool in_x = !(rx < -limx || rx > limx), in_y = !(ry < -limy || ry > limy);
    const float u = fminf(limx, fmaxf(-limx, rx)) * tz, v = fminf(limy, fmaxf(-limy, ry)) * tz;
    const float j00 = fx * itz, j11 = fy * itz, j02 = -fx * u * itz * itz, j12 = -fy * v * itz * itz;
    // A = J W: row 0 = j00 W[0][:] + j02 W[2][:], row 1 = j11 W[1][:] + j12 W[2][:]   (W[k][j] = view[4 j + k])
    float A0[3], A1[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        A0[j] = j00 * view[4 * j] + j02 * view[4 * j + 2];
        A1[j] = j11 * view[4 * j + 1] + j12 * view[4 * j + 2];
    }
    // B = A Sigma (2x3), S = B A^T + 0.3 I
    const float Sg[3][3] = {{c3[0], c3[1], c3[2]}, {c3[1], c3[3], c3[4]}, {c3[2], c3[4], c3[5]}};
    float B0[3], B1[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        B0[j] = A0[0] * Sg[0][j] + A0[1] * Sg[1][j] + A0[2] * Sg[2][j];
        B1[j] = A1[0] * Sg[0][j] + A1[1] * Sg[1][j] + A1[2] * Sg[2][j];
    }
    const float a = B0[0] * A0[0] + B0[1] * A0[1] + B0[2] * A0[2] + 0.3f;
    const float b = B0[0] * A1[0] + B0[1] * A1[1] + B0[2] * A1[2];
    const float c = B1[0] * A1[0] + B1[1] * A1[1] + B1[2] * A1[2] + 0.3f;
    const float det = a * c - b * b;
    const float q = 1.0f / (det * det + 0.0000001f);
    // H = -q adj(S) G adj(S), adj(S) = [[c, -b], [-b, a]]
    const float e0 = c * G00 - b * G01, e1 = c * G01 - b * G11;    // (adj G) row 0
    const float f0 = a * G01 - b * G00, f1 = a * G11 - b * G01;    // (adj G) row 1
    const float H00 = -q * (e0 * c - e1 * b), H01 = -q * (e1 * a - e0 * b), H11 = -q * (f1 * a - f0 * b);
    // P = H A (2x3);  dL/dSigma = A^T P
    float P0[3], P1[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        P0[j] = H00 * A0[j] + H01 * A1[j];
        P1[j] = H01 * A0[j] + H11 * A1[j];
    }
    o.dcov[0] = A0[0] * P0[0] + A1[0] * P1[0];
    o.dcov[3] = A0[1] * P0[1] + A1[1] * P1[1];
    o.dcov[5] = A0[2] * P0[2] + A1[2] * P1[2];
    o.dcov[1] = 2.f * (A0[0] * P0[1] + A1[0] * P1[1]);
    o.dcov[2] = 2.f * (A0[0] * P0[2] + A1[0] * P1[2]);
    o.dcov[4] = 2.f * (A0[1] * P0[2] + A1[1] * P1[2]);
    // dL/dA = 2 H B;  dL/dJ entries = rows of dL/dA against rows of W
    float dA0[3], dA1[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        dA0[j] = 2.f * (H00 * B0[j] + H01 * B1[j]);
        dA1[j] = 2.f * (H01 * B0[j] + H11 * B1[j]);
    }
    const float dJ00 = dA0[0] * view[0] + dA0[1] * view[4] + dA0[2] * view[8];
    const float dJ02 = dA0[0] * view[2] + dA0[1] * view[6] + dA0[2] * view[10];
    const float dJ11 = dA1[0] * view[1] + dA1[1] * view[5] + dA1[2] * view[9];
    const float dJ12 = dA1[0] * view[2] + dA1[1] * view[6] + dA1[2] * view[10];
    // J(t): J00 = fx/tz, J11 = fy/tz, J02 = -fx u/tz^2, J12 = -fy v/tz^2; the clamp removes the u / v dependence on t.xy
    const float itz2 = itz * itz;
    const float du = in_x ? -fx * itz2 * dJ02 : 0.f, dv = in_y ? -fy * itz2 * dJ12 : 0.f;
    const float dtz = -itz2 * (fx * dJ00 + fy * dJ11) + 2.f * itz2 * itz * (fx * u * dJ02 + fy * v * dJ12);
    // back to world space: W^T (du, dv, dtz)
    float3 dm;
    dm.x = view[0] * du + view[1] * dv + view[2] * dtz;
    dm.y = view[4] * du + view[5] * dv + view[6] * dtz;
    dm.z = view[8] * du + view[9] * dv + view[10] * dtz;
    // screen position: ndc = (h.x, h.y) / (h.w + 1e-7), h = P^T m; d2x, d2y are gradients in ndc units (backward.cu:376-391)
    const float hx = proj[0] * m.x + proj[4] * m.y + proj[8] * m.z + proj[12];
    const float hy = proj[1] * m.x + proj[5] * m.y + proj[9] * m.z + proj[13];
    const float hw = proj[3] * m.x + proj[7] * m.y + proj[11] * m.z + proj[15];
    const float iw = 1.0f / (hw + 0.0000001f);
    const float dhx = d2x * iw, dhy = d2y * iw, dhw = -(d2x * hx + d2y * hy) * iw * iw;
    dm.x += proj[0] * dhx + proj[1] * dhy + proj[3] * dhw;
    dm.y += proj[4] * dhx + proj[5] * dhy + proj[7] * dhw;
    dm.z += proj[8] * dhx + proj[9] * dhy + proj[11] * dhw;
    // depth image: the reference differentiates z / w of the view transform at w = 1 (backward.cu:393-398)
    dm.x += (view[2] - view[3] * tz) * ddepth;
    dm.y += (view[6] - view[7] * tz) * ddepth;
    dm.z += (view[10] - view[11] * tz) * ddepth;
    o.dmean = dm;
    return o;
}

// Sigma = L L^T with L = R(q) diag(s), s = scale_modifier * scale (forward.cu:118-152).  D = dL/dSigma as a symmetric matrix
// (off-diagonals = half of the stored doubled entries):  dL/dL = 2 D L;  dL/ds_j = sum_i (dL/dL)_ij R_ij;  dL/dR_ij = (dL/dL)_ij s_j,
// and the quaternion gradient from the antisymmetric / symmetric parts of dL/dR.  The reference returns dL/ds for the EFFECTIVE
// scale (it omits the factor scale_modifier, backward.cu:318-321) and does not normalise q; both are kept.
__device__ __forceinline__ void cov3d_grad(const float* dcov, float3 scale, float mod, float4 qt, float3& dscale, float4& drot) {
    const float r = qt.x, x = qt.y, y = qt.z, z = qt.w;
    const float R[3][3] = {{1.f - 2.f * (y * y + z * z), 2.f * (x * y - r * z), 2.f * (x * z + r * y)},
                           {2.f * (x * y + r * z), 1.f - 2.f * (x * x + z * z), 2.f * (y * z - r * x)},
                           {2.f * (x * z - r * y), 2.f * (y * z + r * x), 1.f - 2.f * (x * x + y * y)}};
    const float s[3] = {mod * scale.x, mod * scale.y, mod * scale.z};
    const float D[3][3] = {{dcov[0], 0.5f * dcov[1], 0.5f * dcov[2]}, {0.5f * dcov[1], dcov[3], 0.5f * dcov[4]}, {0.5f * dcov[2], 0.5f * dcov[4], dcov[5]}};
    // E = D R (3x3); dL/dL_ij = 2 E_ij s_j
    float E[3][3];
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) E[i][j] = D[i][0] * R[0][j] + D[i][1] * R[1][j] + D[i][2] * R[2][j];
    float ds[3];
#pragma unroll
    for (int j = 0; j < 3; j++) ds[j] = 2.f * s[j] * (E[0][j] * R[0][j] + E[1][j] * R[1][j] + E[2][j] * R[2][j]);
    dscale = make_float3(ds[0], ds[1], ds[2]);
    // G = dL/dR, G_ij = 2 E_ij s_j^2
    float Gm[3][3];
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) Gm[i][j] = 2.f * E[i][j] * s[j] * s[j];
    const float ax = Gm[2][1] - Gm[1][2], ay = Gm[0][2] - Gm[2][0], az = Gm[1][0] - Gm[0][1];
    const float sxy = Gm[0][1] + Gm[1][0], sxz = Gm[0][2] + Gm[2][0], syz = Gm[1][2] + Gm[2][1];
    drot.x = 2.f * (x * ax + y * ay + z * az);
    drot.y = 2.f * (r * ax + y * sxy + z * sxz) - 4.f * x * (Gm[1][1] + Gm[2][2]);
    drot.z = 2.f * (r * ay + x * sxy + z * syz) - 4.f * y * (Gm[0][0] + Gm[2][2]);
    drot.w = 2.f * (r * az + x * sxz + y * syz) - 4.f * z * (Gm[0][0] + Gm[1][1]);
}

// M16: shs has exactly 16 coefficients (48 floats, 16-byte aligned rows): rows move as float4 with compile-time indexing
template <bool M16>
__global__ void __launch_bounds__(GB_THREADS) k_gaussian_backward(const GBParams p) {
    __shared__ CamConsts cam;
    __shared__ float stage[GB_THREADS * GB_STRIDE];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 16) cam.view[tid] = p.view[tid];
    else if (tid < 32) cam.proj[tid - 16] = p.proj[tid - 16];
    else if (tid < 35) cam.campos[tid - 32] = p.campos[tid - 32];
    __syncthreads();
    const int idx = blockIdx.x * GB_THREADS + tid;
    const bool valid = idx < p.P;
    const bool vis = valid && p.radii[idx] > 0;
    const float* view = cam.view;
    const float* proj = cam.proj;

    // ---- stage the SH rows of visible Gaussians (first 16 coefficients) ----
    float* wstage = stage + warp * 32 * GB_STRIDE;
    const size_t gbase = (size_t)(blockIdx.x * GB_THREADS + warp * 32);
    const size_t row_floats = (size_t)p.M * 3;
    const int nf = p.shs ? min(48, (int)row_floats) : 0;
    const unsigned vismask = __ballot_sync(GSR_FULL, vis);
    if (p.shs) {
        if (M16) {  // 12 float4 per row, consecutive lanes fetch consecutive 16-byte parts
#pragma unroll
            for (int it = 0; it < 12; it++) {
                const int item = it * 32 + lane;
                const int gl = item / 12, part = item - gl * 12;
                if ((vismask >> gl) & 1u) {
                    const float4 v = reinterpret_cast<const float4*>(p.shs + (gbase + gl) * 48)[part];
                    float* d = wstage + gl * GB_STRIDE + part * 4;
                    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
                }
            }
        } else {
            for (int it = 0; it < nf; it++) {
                const int item = it * 32 + lane;
                const int gl = item / nf, part = item - gl * nf;
                if ((vismask >> gl) & 1u) wstage[gl * GB_STRIDE + part] = p.shs[(gbase + gl) * row_floats + part];
            }
        }
        __syncwarp();
    }

    float3 dmean = {0, 0, 0};
    float dcov[6] = {0, 0, 0, 0, 0, 0};
    float3 dscale = {0, 0, 0};
    float4 drot = {0, 0, 0, 0};
    if (vis) {
        const float3 mean = {p.means3D[3 * (size_t)idx], p.means3D[3 * (size_t)idx + 1], p.means3D[3 * (size_t)idx + 2]};
        float c3[6];
#pragma unroll
        for (int k = 0; k < 6; k++) c3[k] = p.cov3Ds[6 * (size_t)idx + k];
        const float4 gK = (((uintptr_t)p.dL_dconic & 15) == 0) ? reinterpret_cast<const float4*>(p.dL_dconic)[idx]  // (G00, G01, -, G11)
                                                                : make_float4(p.dL_dconic[4 * (size_t)idx], p.dL_dconic[4 * (size_t)idx + 1], 0.f,
                                                                              p.dL_dconic[4 * (size_t)idx + 3]);
        const GeoGrad gg = geometry_grad(mean, c3, view, proj, p.h_x, p.h_y, 1.3f * p.tanfovx, 1.3f * p.tanfovy, gK.x, gK.y, gK.w,
                                         p.dL_dmean2D[3 * (size_t)idx], p.dL_dmean2D[3 * (size_t)idx + 1], p.dL_ddepth[idx]);
        dmean = gg.dmean;
#pragma unroll
        for (int k = 0; k < 6; k++) dcov[k] = gg.dcov[k];
        if (p.shs) {
            const float3 dcol = {p.dL_dcolor[3 * (size_t)idx], p.dL_dcolor[3 * (size_t)idx + 1], p.dL_dcolor[3 * (size_t)idx + 2]};
            const float3 dm = sh_grad(p.D, wstage + lane * GB_STRIDE, mean, cam.campos, p.clamped[idx], dcol);
            dmean.x += dm.x; dmean.y += dm.y; dmean.z += dm.z;
        }
        if (p.scales) {
            const float3 sc = {p.scales[3 * (size_t)idx], p.scales[3 * (size_t)idx + 1], p.scales[3 * (size_t)idx + 2]};
            const float4 qt = (((uintptr_t)p.rotations & 15) == 0) ? reinterpret_cast<const float4*>(p.rotations)[idx]
                                                                  : make_float4(p.rotations[4 * (size_t)idx], p.rotations[4 * (size_t)idx + 1],
                                                                                p.rotations[4 * (size_t)idx + 2], p.rotations[4 * (size_t)idx + 3]);
            cov3d_grad(dcov, sc, p.scale_modifier, qt, dscale, drot);
        }
    }
    if (valid) {
        p.dL_dmeans3D[3 * (size_t)idx] = dmean.x; p.dL_dmeans3D[3 * (size_t)idx + 1] = dmean.y; p.dL_dmeans3D[3 * (size_t)idx + 2] = dmean.z;
#pragma unroll
        for (int k = 0; k < 6; k++) p.dL_dcov3D[6 * (size_t)idx + k] = dcov[k];
        if (p.dL_dscale) { p.dL_dscale[3 * (size_t)idx] = dscale.x; p.dL_dscale[3 * (size_t)idx + 1] = dscale.y; p.dL_dscale[3 * (size_t)idx + 2] = dscale.z; }
        if (p.dL_drot) { p.dL_drot[4 * (size_t)idx] = drot.x; p.dL_drot[4 * (size_t)idx + 1] = drot.y; p.dL_drot[4 * (size_t)idx + 2] = drot.z; p.dL_drot[4 * (size_t)idx + 3] = drot.w; }
    }
    // ---- write dL/dsh rows: coalesced, zeros for culled Gaussians and for coefficients beyond 16 ----
    if (p.shs && p.dL_dsh) {
        __syncwarp();
        const int valid_rows = min(32, p.P - (int)gbase);
        if (M16) {
#pragma unroll
            for (int it = 0; it < 12; it++) {
                const int item = it * 32 + lane;
                const int gl = item / 12, part = item - gl * 12;
                if (gl < valid_rows) {
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if ((vismask >> gl) & 1u) {
                        const float* s = wstage + gl * GB_STRIDE + part * 4;
                        v = make_float4(s[0], s[1], s[2], s[3]);
                    }
                    reinterpret_cast<float4*>(p.dL_dsh + (gbase + gl) * 48)[part] = v;
                }
            }
        } else {
            const int rf = (int)row_floats;
            for (int item = lane; item < valid_rows * rf; item += 32) {
                const int gl = item / rf, part = item - gl * rf;
                float v = 0.f;
                if (((vismask >> gl) & 1u) && part < nf) v = wstage[gl * GB_STRIDE + part];
                p.dL_dsh[gbase * row_floats + item] = v;
            }
        }
    }
}

int backward_impl(const gsr_frame* f, const gsr_workspace* ws, const int32_t* radii, const float* out_alpha, const float* dL_dc,
                  const float* dL_dd, const float* dL_da, const float* extra, const float* dL_de, float* dL_dextra, const gsr_grads* g,
                  cudaStream_t st) {
    if (!f || !ws || !g) { set_error("gsr_backward: null argument"); return GSR_ERR_INVALID; }
    const bool has_extra = extra != nullptr;
    if (has_extra != (dL_de != nullptr) || has_extra != (dL_dextra != nullptr)) {
        set_error("gsr_backward_multi: extra_colors, dL_dout_extra and dL_dextra_colors must all be set or all be NULL");
        return GSR_ERR_INVALID;
    }
    const bool debug = f->debug != 0;
    const size_t P = (size_t)f->P;
    if (!g->dL_dmeans2D || !g->dL_dconic || !g->dL_dopacity || !g->dL_dcolors || !g->dL_ddepths || !g->dL_dmeans3D || !g->dL_dcov3D) {
        set_error("gsr_backward: null gradient buffer");
        return GSR_ERR_INVALID;
    }
    if (f->shs && !g->dL_dsh) { set_error("gsr_backward: dL_dsh missing"); return GSR_ERR_INVALID; }
    if (f->scales && (!g->dL_dscales || !g->dL_drotations)) { set_error("gsr_backward: dL_dscales/dL_drotations missing"); return GSR_ERR_INVALID; }
    // accumulated gradients start from zero
    cudaMemsetAsync(g->dL_dmeans2D, 0, 12 * P, st);
    cudaMemsetAsync(g->dL_dconic, 0, 16 * P, st);
    cudaMemsetAsync(g->dL_dopacity, 0, 4 * P, st);
    cudaMemsetAsync(g->dL_dcolors, 0, 12 * P, st);
    cudaMemsetAsync(g->dL_ddepths, 0, 4 * P, st);
    if (has_extra) cudaMemsetAsync(dL_dextra, 0, 12 * P, st);
    if (P == 0) return check_launch("gsr_backward(P=0)", debug, st);
    if (!radii || !out_alpha || !dL_dc || !dL_dd || !dL_da) { set_error("gsr_backward: null input"); return GSR_ERR_INVALID; }
    const ImageLayout il(f->W, f->H);
    const GeomLayout gl(P);
    if (ws->image_bytes < il.total || ws->geom_bytes < gl.total || !ws->binning) { set_error("gsr_backward: workspace too small"); return GSR_ERR_WORKSPACE; }
    const BinLayout bl(BinLayout::capacity_of(ws->binning_bytes));
    char* img = (char*)ws->image; char* geo = (char*)ws->geom; char* bin = (char*)ws->binning;
    const int D = f->D < 0 ? 0 : (f->D > 3 ? 3 : f->D);

    BwdArgs ba;
    ba.ranges = (const uint2*)(img + il.ranges); ba.point_list = (const uint32_t*)(bin + bl.point_list); ba.records = (const float4*)(geo + gl.records);
    ba.bal = (const uint32_t*)(bin + bl.bal);
    ba.W = f->W; ba.H = f->H; ba.gx = il.gx; ba.bg = f->bg; ba.accum_alphas = out_alpha; ba.n_contrib = (const uint32_t*)(img + il.n_contrib);
    ba.dL_dpixels = dL_dc; ba.dL_dpixel_depths = dL_dd; ba.dL_dpixel_alphas = dL_da;
    ba.dL_dmean2D = g->dL_dmeans2D; ba.dL_dconic = g->dL_dconic; ba.dL_dopacity = g->dL_dopacity; ba.dL_dcolors = g->dL_dcolors; ba.dL_ddepths = g->dL_ddepths;
    ba.extra = extra; ba.dL_dpixel_extras = dL_de; ba.dL_dextra = dL_dextra;
    {
        const dim3 grid(il.gx * (GSR_FOOTS / BWL_WARPS), il.gy);
        static int occ = -1;  // GSR_BWD_OCC=8|6|5: resident CTAs per SM the kernel is compiled for (64 / 80 / 96 registers), an experiment knob
        if (occ < 0) { const char* e = getenv("GSR_BWD_OCC"); occ = e ? atoi(e) : 6; }
        // EXTRA is compiled for 5 CTAs per SM (96 registers, 0 spills, 30 KiB shared memory per CTA): its three more pixel
        // gradients, staged colours and moments do not fit the 80 registers of 6 CTAs per SM (60 bytes of spills, sm_100a ptxas)
        if (has_extra) k_blend_backward<5, true><<<grid, BWL_WARPS * 32, 0, st>>>(ba);
        else if (occ == 8) k_blend_backward<8><<<grid, BWL_WARPS * 32, 0, st>>>(ba);
        else if (occ == 5) k_blend_backward<5><<<grid, BWL_WARPS * 32, 0, st>>>(ba);
        else k_blend_backward<6><<<grid, BWL_WARPS * 32, 0, st>>>(ba);
    }
    int rc = check_launch("gsr_backward/blend", debug, st);
    if (rc) return rc;

    GBParams gp;
    gp.P = f->P; gp.D = D; gp.M = f->M; gp.W = f->W; gp.H = f->H;
    gp.scale_modifier = f->scale_modifier; gp.tanfovx = f->tanfovx; gp.tanfovy = f->tanfovy;
    gp.h_y = f->H / (2.0f * f->tanfovy); gp.h_x = f->W / (2.0f * f->tanfovx);
    gp.means3D = f->means3D; gp.shs = f->shs; gp.scales = f->scales; gp.rotations = f->rotations;
    gp.cov3Ds = f->cov3D_precomp ? f->cov3D_precomp : (const float*)(geo + gl.cov3D);
    gp.view = f->viewmatrix; gp.proj = f->projmatrix; gp.campos = f->campos;
    gp.radii = radii; gp.clamped = (const uint8_t*)(geo + gl.clamped);
    gp.dL_dmean2D = g->dL_dmeans2D; gp.dL_dconic = g->dL_dconic; gp.dL_dcolor = g->dL_dcolors; gp.dL_ddepth = g->dL_ddepths;
    gp.dL_dmeans3D = g->dL_dmeans3D; gp.dL_dcov3D = g->dL_dcov3D; gp.dL_dsh = g->dL_dsh;
    gp.dL_dscale = f->scales ? g->dL_dscales : nullptr; gp.dL_drot = f->scales ? g->dL_drotations : nullptr;
    const bool m16 = f->shs && f->M == 16 && (((uintptr_t)f->shs | (uintptr_t)g->dL_dsh) & 15) == 0;
    if (m16) k_gaussian_backward<true><<<(f->P + GB_THREADS - 1) / GB_THREADS, GB_THREADS, 0, st>>>(gp);
    else k_gaussian_backward<false><<<(f->P + GB_THREADS - 1) / GB_THREADS, GB_THREADS, 0, st>>>(gp);
    // gradient buffers the reference leaves at zero for the absent parametrisation
    if (!f->scales) {
        if (g->dL_dscales) cudaMemsetAsync(g->dL_dscales, 0, 12 * P, st);
        if (g->dL_drotations) cudaMemsetAsync(g->dL_drotations, 0, 16 * P, st);
    }
    return check_launch("gsr_backward/gaussian", debug, st);
}

}  // namespace gsr
