// Convolution engine, tensor-core path: implicit GEMM on tcgen05 (5th-gen tensor cores) for sm_100a.
//
//   D[128 pixels x Cout] (fp32, TMEM)  +=  A[128 pixels x 32 ch] (smem, TMA)  x  B[Cout x 32 ch]^T (smem, TMA)     kind::tf32
//
// One CTA owns an 8x16 tile of output pixels (UMMA M = 128) and all Cout (UMMA N = Cout padded to 16, <= 256).  The K
// loop runs over (filter tap, concatenated source, 32-channel chunk):
//   * the A operand of a tap is the NHWC input tile shifted by the tap offset, fetched by ONE 4-D TMA box
//     {32 ch, 16 px, 8 px, 1 img} (traversal stride = conv stride).  Out-of-bounds elements are zero-filled by the TMA unit,
//     which IS the reference's PadSameConv2d (model/layers.py:220-252); channel concatenation (torch.cat,
//     monorec_model.py:372-380, :541-545) is just one tensor map per source;
//   * the B operand is the matching [Cout x 32] slice of the packed weights (2-D TMA);
//   * both land in 128-byte-swizzled K-major shared-memory tiles that tcgen05.mma consumes through smem descriptors.
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = epilogue (tcgen05.ld ->
// bias -> activation -> NHWC store, optional sub-pixel placement).  The producer and issuer loops run on CONVERGED warps with
// elect-predicated instructions (see umma_elect): their operands stay in uniform registers, ~7 SASS instructions per MMA.
// Pipelines: smem full/empty mbarrier ring between TMA and MMA; tmem full/empty mbarriers between MMA and epilogue (the
// accumulator is double-buffered in TMEM, the kernels are persistent over output tiles).
// Two kernels, chosen by the host code at the bottom of this file:
//   conv_tc_halo_kernel  stride-1 layers: ONE input box per (tile, K chunk) with its halo, every filter tap a shifted
//                        shared-memory descriptor into it; weights resident in shared memory, or -- when they do not fit
//                        next to two input stages -- streamed slice by slice through a second ring; 64- or 128-byte rows;
//   conv_tc_kernel       everything else (strided layers, the sub-pixel phases of Refine / Upconv -- up to four phases share
//                        one launch): one input box and one weight slice per (tap, K chunk).
// The epilogue is staged through shared memory (8 pixels x 64 contiguous bytes per store instruction); one-channel heads take
// a single accumulator column.  K steps that hold only the zero padding behind a source's channels are skipped.
//
// Reference being replaced: nn.Conv2d / nn.ConvTranspose2d + bias + LeakyReLU of model/layers.py:289-400 as used by
// MaskModule / DepthModule (model/monorec/monorec_model.py:287-385, :476-557).
#include "mr_common.cuh"
#include <cuda.h>
#include <cstdint>
#include <type_traits>
#include <cstdlib>
#include <cuda_fp16.h>

namespace {

constexpr int kTcThreads = 192;
constexpr int kKC = 32;                 // fp32 channels per K chunk = one 128-byte swizzle row
constexpr int kTileH = 8, kTileW = 16;  // 128 output pixels per CTA

struct TcArgs {
    int n_src;
    int chunks[MR_CONV_MAX_SRC];   // K chunks per source
    int tail_ksteps[MR_CONV_MAX_SRC];   // MMA K steps (32 bytes of channels each) that hold data in the LAST chunk of each source: the
                                        // zero padding behind a source's channels is neither multiplied nor read from shared memory
    int kh, kw, sy, sx, pad_t, pad_l;
    int Ho, Wo, Cout, n_pad, tiles_x, tiles_per_img, total_tiles, stages;
    uint32_t tmem_cols;
    const float* bias;
    float* dst;
    int dst_H, dst_W, dst_c, dst_coff, oy_step, ox_step, oy_off, ox_off;
    int act;
    float act_a, act_b;
    int round_out;                 // 1: round stored activations to TF32 (nearest) so the next layer's truncation is exact
    int kc;                        // channels per K chunk: 32 (fp32 sources, kind::tf32) or 64 (half sources, kind::f16)
    int f16, out_f16;              // half sources+weights / half destination
    uint32_t idesc;                // UMMA instruction descriptor
    int row_bytes;                 // bytes of one K chunk row in shared memory = swizzle span: 128, or 64 (half sources, 32-channel chunks)
    // tap-refetch kernel: up to 4 "phases" (the sub-pixel convolutions of one Refine / Upconv layer) share one launch; tile
    // index = spatial tile * n_phase + phase, so the phases of a spatial tile run side by side and its input boxes are L2 hits
    int n_phase;
    int ph_kh[4], ph_kw[4], ph_pad_t[4], ph_pad_l[4], ph_oy_off[4], ph_ox_off[4];
    int b_stream;                  // halo kernel: 0 = the layer's weights stay resident in shared memory; n > 0 = they do not fit: the
                                   // [n_pad x chunk] slice of every (chunk, tap) streams through a ring of n stages instead
    int halo_pitch;                // halo kernel: pixels per input row of the shared-memory box (8 outputs + kw - 1 taps to the right)
    uint32_t halo_a_bytes;         // halo kernel: bytes of one input stage (box rounded up to 1 KB)
    int epi;                       // MR_TC_EPI_*: the epilogue the host plan chose
};

// ---- PTX wrappers -------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
// K-major swizzled shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (1: unused for swizzled K-major) |
//   [32,46) stride byte offset >> 4 (distance between 8-row groups) | [46,48) version = 1 | [49,52) base offset |
//   [61,64) layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B.  Everything but the start address is layer-constant (desc_hi()).
// ---- single-lane instructions issued from CONVERGED warp code ---------------------------------------------------------------
// The producer and MMA warps used to run their loops under `if (lane == 0)`.  Every operand of UTMALDG / UTCHMMA / UTCBAR lives
// in a uniform register, and inside a divergent region ptxas cannot keep values there: the SASS of the tap loop had ~20
// instructions (R2UR.BROADCAST, ELECT, a waterfall branch) around every MMA, and that single-thread instruction stream -- not
// the tensor pipe, shared memory or HBM -- paced the kernels.  Here all 32 lanes execute the loops (uniform arithmetic only) and
// the instruction itself is predicated on elect.sync.
template <bool F16>
__device__ __forceinline__ void umma_elect(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                           uint32_t accumulate) {
    if (F16)
        asm volatile(
            "{\n\t"
            ".reg .pred p, pe;\n\t"
            ".reg .b64 da, db;\n\t"
            "mov.b64 da, {%1, %2};\n\t"
            "mov.b64 db, {%3, %4};\n\t"
            "setp.ne.b32 p, %6, 0;\n\t"
            "elect.sync _|pe, 0xffffffff;\n\t"
            "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
            "}\n" ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t"
            ".reg .pred p, pe;\n\t"
            ".reg .b64 da, db;\n\t"
            "mov.b64 da, {%1, %2};\n\t"
            "mov.b64 db, {%3, %4};\n\t"
            "setp.ne.b32 p, %6, 0;\n\t"
            "elect.sync _|pe, 0xffffffff;\n\t"
            "@pe tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t"
            "}\n" ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
            : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint32_t bar) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
        "}\n" ::"r"(bar)
        : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_elect(uint32_t bar, uint32_t bytes) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t"
        "}\n" ::"r"(bar), "r"(bytes)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_elect(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t"
        "}\n" ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_elect(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t"
        "}\n" ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
// shared-memory descriptor halves: low word = start address >> 4 | LBO (1, unused) << 16; high word = SBO >> 4 | version 1 << 14 |
// layout << 29 (the K-major swizzled descriptor's bit layout is in the comment further up)
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes, uint32_t row_bytes) {
    return (sbo_bytes >> 4) | (1u << 14) | ((row_bytes == 128 ? 2u : 4u) << 29);
}

__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float act_fn(float v, int act, float a, float b) {
    switch (act) {
        case MR_ACT_LEAKY: return v >= 0.f ? v : a * v;
        case MR_ACT_SIGMOID: return 1.0f / (1.0f + expf(-v));
        case MR_ACT_ABSTANH: return fmaf(b, fabsf(tanhf(v)), a);
        default: return v;
    }
}

// LeakyReLU x >= 0 ? x : s*x for any slope as one min / max: max(x, s*x) when s <= 1, min(x, s*x) when s > 1.  `s_le1` is the
// same for the whole layer, so the choice costs no per-element predicate (FMNMX takes it as an operand).
__device__ __forceinline__ float leaky(float x, float s, bool s_le1) {
    const float y = s * x;
    return s_le1 ? fmaxf(x, y) : fminf(x, y);
}

// Epilogue of one accumulator row (= one output pixel): 32 columns per step (two x16 TMEM loads, one wait), bias from shared
// memory, activation, optional TF32 rounding, 16-byte NHWC stores.
__device__ __forceinline__ void epilogue_row(uint32_t trow, const TcArgs& a, const float* bias_s, float* op, bool live,
                                             bool vec_ok) {
    __half* oph = reinterpret_cast<__half*>(op);   // when a.out_f16 the caller computed `op` in half elements
    for (int n0 = 0; n0 < a.n_pad; n0 += 32) {
        uint32_t r0[16], r1[16];
        const bool second = n0 + 16 < a.n_pad;
        tmem_ld16_nowait(trow + (uint32_t)n0, r0);
        if (second) tmem_ld16_nowait(trow + (uint32_t)(n0 + 16), r1);
        tmem_ld_wait();
        if (!live) continue;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (h == 1 && !second) break;
            const int nb = n0 + 16 * h;
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float x = __uint_as_float(h ? r1[j] : r0[j]) + bias_s[nb + j];
                if (a.act != MR_ACT_NONE) x = act_fn(x, a.act, a.act_a, a.act_b);
                if (a.round_out) x = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
                v[j] = x;
            }
            if (a.out_f16) {
                if (vec_ok && nb + 16 <= a.Cout) {
                    uint4 q0, q1;
                    __half2* h0 = reinterpret_cast<__half2*>(&q0);
                    __half2* h1 = reinterpret_cast<__half2*>(&q1);
#pragma unroll
                    for (int j = 0; j < 4; ++j) { h0[j] = __floats2half2_rn(v[2 * j], v[2 * j + 1]); h1[j] = __floats2half2_rn(v[8 + 2 * j], v[9 + 2 * j]); }
                    *reinterpret_cast<uint4*>(oph + nb) = q0;
                    *reinterpret_cast<uint4*>(oph + nb + 8) = q1;
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (nb + j < a.Cout) oph[nb + j] = __float2half_rn(v[j]);
                }
            } else if (vec_ok && nb + 16 <= a.Cout) {
#pragma unroll
                for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(op + nb + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (nb + j < a.Cout) op[nb + j] = v[j];
            }
        }
    }
}

// out-of-line copy of the generic epilogue for the staged kernel's rare fallback (keeps its hot code small)
// (`a` by value: a reference would force the kernel's parameter block onto the local stack for the hot path as well)
__device__ __noinline__ void epilogue_row_outofline(uint32_t trow, const TcArgs a, const float* bias_s, float* op, bool live, bool vec_ok) {
    epilogue_row(trow, a, bias_s, op, live, vec_ok);
}

// ---- staged epilogue -----------------------------------------------------------------------------------------------------------
// The source-level profile of round 1's register epilogue (profiles/r01_k2_fullres_f16_quad_ncu_details.txt and the source page of
// the same capture) shows ~900 executed instructions per warp and tile spread over a 12 700-instruction kernel body
// (23 % of the stall samples are instruction-fetch misses) -- per-element activation switches, predicates and 48 SEL + 16
// SHFL per quad transpose.  This variant keeps the per-tile decisions out of the element loop (LeakyReLU through leaky()
// with slope = 1 for "no activation", rounding as a template parameter) and transposes through a 2 KB per-warp staging
// buffer in shared memory instead of shuffles: every thread writes the 64 bytes of its pixel (4 x STS.128, XOR-swizzled,
// conflict-free), then lane l reads chunk l%4 of pixel l/4 + 8k and stores it, so that one store instruction covers 8
// pixels x 64 contiguous bytes.  One step = 16 fp32 or 32 half output channels.
template <bool OUT_F16, bool ROUND>
__device__ __forceinline__ void epilogue_staged(uint32_t trow, const TcArgs& a, const float* bias_s, uint32_t stg, uint8_t* const (&qptr)[4],
                                                const bool (&qlive)[4], int lane, float slope) {
    constexpr int kCols = OUT_F16 ? 32 : 16;        // output channels per 64-byte step
    constexpr int kChunk = OUT_F16 ? 8 : 4;         // channels per 16-byte chunk
    const bool s_le1 = slope <= 1.f;
    const uint32_t wrow = stg + (uint32_t)lane * 64u;
    const uint32_t wsw = ((uint32_t)lane >> 1) & 3u;
    const uint32_t c = (uint32_t)lane & 3u;
    uint32_t raddr[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t q = ((uint32_t)lane >> 2) + 8u * k;
        raddr[k] = stg + q * 64u + ((c ^ ((q >> 1) & 3u)) << 4);
    }
    for (int n0 = 0; n0 < a.n_pad; n0 += kCols) {
        uint32_t r0[16], r1[16];
        tmem_ld16_nowait(trow + (uint32_t)n0, r0);
        const bool second = OUT_F16 && (n0 + 16 < a.n_pad);
        if (second) tmem_ld16_nowait(trow + (uint32_t)(n0 + 16), r1);
        tmem_ld_wait();
        uint4 e[4];
        if (OUT_F16) {
            __half2* h = reinterpret_cast<__half2*>(e);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float x0 = __uint_as_float(r0[2 * j]) + bias_s[n0 + 2 * j], x1 = __uint_as_float(r0[2 * j + 1]) + bias_s[n0 + 2 * j + 1];
                h[j] = __floats2half2_rn(leaky(x0, slope, s_le1), leaky(x1, slope, s_le1));
            }
            if (second) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float x0 = __uint_as_float(r1[2 * j]) + bias_s[n0 + 16 + 2 * j], x1 = __uint_as_float(r1[2 * j + 1]) + bias_s[n0 + 17 + 2 * j];
                    h[8 + j] = __floats2half2_rn(leaky(x0, slope, s_le1), leaky(x1, slope, s_le1));
                }
            } else {
                e[2] = make_uint4(0u, 0u, 0u, 0u);
                e[3] = make_uint4(0u, 0u, 0u, 0u);
            }
        } else {
            uint32_t* w = reinterpret_cast<uint32_t*>(e);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float x = __uint_as_float(r0[j]) + bias_s[n0 + j];
                x = leaky(x, slope, s_le1);
                w[j] = ROUND ? ((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u) : __float_as_uint(x);
            }
        }
#pragma unroll
        for (uint32_t cc = 0; cc < 4; ++cc)
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(wrow + ((cc ^ wsw) << 4)), "r"(e[cc].x), "r"(e[cc].y),
                         "r"(e[cc].z), "r"(e[cc].w)
                         : "memory");
        __syncwarp();
        const bool col_ok = n0 + (int)c * kChunk + kChunk <= a.Cout;
        const size_t boff = ((size_t)n0 * (OUT_F16 ? 2 : 4)) + (size_t)c * 16;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint4 v;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(raddr[k]) : "memory");
            if (qlive[k] && col_ok) *reinterpret_cast<uint4*>(qptr[k] + boff) = v;
        }
        __syncwarp();
    }
}

// One tile of the staged epilogue for a warp (TMEM lane quadrant q): output pointers / liveness of the 4 pixels each lane
// stores for, then the 64-byte steps; tiles are kTW x kTH pixels with accumulator row p = y * kTW + x.  Layers the staged
// path cannot take (unaligned channel slices, the rare activations) go through the generic out-of-line epilogue.
template <int kTW, int kTH>
__device__ __forceinline__ void staged_tile(const TcArgs& a, const float* bias_s, uint32_t stg, int q, int lane, int b, int tile_y,
                                            int tile_x, uint32_t trow, bool lean_ok, bool vec_ok, float slope, int oy_off, int ox_off) {
    if (lean_ok) {
        const size_t esize = a.out_f16 ? 2 : 4;
        uint8_t* qptr[4];
        bool qlive[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {       // accumulator rows 32q + lane/4 + 8k
            const int pq = 32 * q + (lane >> 2) + 8 * k;
            const int qy = tile_y * kTH + pq / kTW, qx = tile_x * kTW + pq % kTW;
            qlive[k] = (qy < a.Ho) && (qx < a.Wo);
            const size_t qidx = (((size_t)b * a.dst_H + (qy * a.oy_step + oy_off)) * a.dst_W + (qx * a.ox_step + ox_off)) *
                                    a.dst_c + a.dst_coff;
            qptr[k] = reinterpret_cast<uint8_t*>(a.dst) + qidx * esize;
        }
        if (a.out_f16) epilogue_staged<true, false>(trow, a, bias_s, stg, qptr, qlive, lane, slope);
        else if (a.round_out) epilogue_staged<false, true>(trow, a, bias_s, stg, qptr, qlive, lane, slope);
        else epilogue_staged<false, false>(trow, a, bias_s, stg, qptr, qlive, lane, slope);
    } else {
        const int p = 32 * q + lane;
        const int oy = tile_y * kTH + p / kTW, ox = tile_x * kTW + p % kTW;
        const size_t oidx = (((size_t)b * a.dst_H + (oy * a.oy_step + oy_off)) * a.dst_W + (ox * a.ox_step + ox_off)) *
                                a.dst_c + a.dst_coff;
        const bool live = (oy < a.Ho) && (ox < a.Wo);
        if (a.epi == MR_TC_EPI_ONE_COLUMN) {
            // single-channel heads (sigmoid / a + b |tanh|): one accumulator column per pixel instead of the generic path's 16
            // activations per pixel (measured: 24->1 3x3 at full resolution 123 us with the generic epilogue)
            uint32_t r;
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(trow));
            tmem_ld_wait();
            float x = act_fn(__uint_as_float(r) + bias_s[0], a.act, a.act_a, a.act_b);
            if (a.round_out) x = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
            if (live) {
                if (a.out_f16) reinterpret_cast<__half*>(a.dst)[oidx] = __float2half_rn(x);
                else a.dst[oidx] = x;
            }
        } else {
            float* op = a.out_f16 ? reinterpret_cast<float*>(reinterpret_cast<__half*>(a.dst) + oidx) : a.dst + oidx;
            epilogue_row_outofline(trow, a, bias_s, op, live, vec_ok);
        }
    }
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// Persistent: each CTA loops over output tiles (tile = blockIdx.x, += gridDim.x).  The TMA->MMA shared-memory ring keeps
// flowing across tile boundaries and the accumulator is double-buffered in TMEM, so the epilogue of tile i overlaps the
// main loop of tile i+1.
__global__ void __launch_bounds__(kTcThreads)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
               const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmB1,
               const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ CUtensorMap tmB3, const TcArgs a) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * 8 + 4];   // full[8], empty[8], tmem_full[2], tmem_empty[2]
    __shared__ uint32_t tmem_base_s;
    __shared__ float bias_s[256];

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // (the broadcast tells ptxas the role branches are warp-uniform)
    const uint32_t tile_base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B tiles need 1024-byte alignment
    const uint32_t a_bytes = 128u * (uint32_t)a.row_bytes, b_bytes = (uint32_t)a.n_pad * (uint32_t)a.row_bytes;
    const uint32_t stage_bytes = a_bytes + b_bytes;
    const int stages = a.stages;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[8]);
    const uint32_t tfull0 = smem_u32(&bars[16]), tempty0 = smem_u32(&bars[18]);
    const int chunks_per_tap = a.chunks[0] + a.chunks[1] + a.chunks[2];
    const int n_phase = a.n_phase;

    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull0 + 8 * s, 1); mbar_init(tempty0 + 8 * s, 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = threadIdx.x; i < 256; i += kTcThreads) bias_s[i] = (a.bias != nullptr && i < a.Cout) ? __ldg(a.bias + i) : 0.f;
    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmA0);
        if (a.n_src > 1) prefetch_tmap(&tmA1);
        if (a.n_src > 2) prefetch_tmap(&tmA2);
        prefetch_tmap(&tmB);
        if (n_phase > 1) { prefetch_tmap(&tmB1); prefetch_tmap(&tmB2); prefetch_tmap(&tmB3); }
    }
    if (warp == 1) {   // TMEM allocation (power of two >= 32 columns), address published through shared memory
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                     "r"(a.tmem_cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = tmem_base_s;

    if (warp == 0) {
        // ===================== TMA producer (whole warp, converged; the copies are issued by an elected lane) =====================
        int st = 0;
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
            const int sp = tile / n_phase, phs = tile - sp * n_phase;
            const int b = sp / a.tiles_per_img, t = sp - b * a.tiles_per_img;
            const int tile_y = t / a.tiles_x, tile_x = t - tile_y * a.tiles_x;
            const int oy0 = tile_y * kTileH, ox0 = tile_x * kTileW;
            const int kh = a.ph_kh[phs], kw = a.ph_kw[phs], pad_t = a.ph_pad_t[phs], pad_l = a.ph_pad_l[phs];
            const CUtensorMap* tb = (phs == 0) ? &tmB : ((phs == 1) ? &tmB1 : ((phs == 2) ? &tmB2 : &tmB3));
            int brow = 0;
            for (int ky = 0; ky < kh; ++ky)
                for (int kx = 0; kx < kw; ++kx, brow += a.n_pad) {
                    const int ix0 = ox0 * a.sx - pad_l + kx, iy0 = oy0 * a.sy - pad_t + ky;
                    int kbase = 0;
                    for (int s = 0; s < a.n_src; ++s) {
                        const CUtensorMap* tm = (s == 0) ? &tmA0 : ((s == 1) ? &tmA1 : &tmA2);
                        for (int j = 0; j < a.chunks[s]; ++j, kbase += a.kc) {
                            mbar_wait(empty0 + 8 * st, ph ^ 1u);
                            const uint32_t sa = tile_base + st * stage_bytes, sb = sa + a_bytes;
                            mbar_expect_tx_elect(full0 + 8 * st, stage_bytes);
                            tma_load_4d_elect(sa, tm, full0 + 8 * st, j * a.kc, ix0, iy0, b);
                            tma_load_2d_elect(sb, tb, full0 + 8 * st, kbase, brow);
                            if (++st == stages) { st = 0; ph ^= 1u; }
                        }
                    }
                }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (whole warp, converged; the MMAs are issued by an elected lane) =====================
        // instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 = 1 @[4,6), a/b format TF32 = 2 @[7,10)/[10,13),
        // K-major A and B, N >> 3 @[17,23), M >> 4 @[24,29)
        const uint32_t idesc = a.idesc;
        const uint32_t dhi = desc_hi(8u * (uint32_t)a.row_bytes, (uint32_t)a.row_bytes);
        const int ksteps = a.row_bytes / 32;   // UMMA K = 32 bytes (8 tf32 / 16 half): 4 (2) steps inside the 128 (64)-byte swizzle row
        auto run = [&](auto f16tag) {
        constexpr bool kF16 = decltype(f16tag)::value;
        int st = 0, lt = 0;
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++lt) {
            const int buf = lt & 1;
            mbar_wait(tempty0 + 8 * buf, (((uint32_t)lt >> 1) & 1u) ^ 1u);   // epilogue has drained this accumulator
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t acc = tmem_d + (uint32_t)(buf * a.n_pad);
            const int phs = tile % n_phase;
            const int total = a.ph_kh[phs] * a.ph_kw[phs] * chunks_per_tap;
            uint32_t accf = 0;
            int src = 0, jc = 0;                                             // source / chunk inside the source of step c
            for (int c = 0; c < total; ++c) {
                mbar_wait(full0 + 8 * st, ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = tile_base + st * stage_bytes;
                const uint32_t alo = desc_lo(sa), blo = desc_lo(sa + a_bytes);
                const int ks = (jc == a.chunks[src] - 1) ? a.tail_ksteps[src] : ksteps;
                umma_elect<kF16>(acc, alo, dhi, blo, dhi, idesc, accf);
                if (ks > 1) umma_elect<kF16>(acc, alo + 2, dhi, blo + 2, dhi, idesc, 1u);
                if (ks > 2) umma_elect<kF16>(acc, alo + 4, dhi, blo + 4, dhi, idesc, 1u);
                if (ks > 3) umma_elect<kF16>(acc, alo + 6, dhi, blo + 6, dhi, idesc, 1u);
                if (++jc == a.chunks[src]) { jc = 0; if (++src == a.n_src) src = 0; }
                accf = 1u;
                umma_commit_elect(empty0 + 8 * st);                          // frees the smem stage once these MMAs have read it
                if (c == total - 1) umma_commit_elect(tfull0 + 8 * buf);     // accumulator complete
                if (++st == stages) { st = 0; ph ^= 1u; }
            }
        }
        };
        if (a.f16) run(std::true_type{}); else run(std::false_type{});
    } else {
        // ===================== epilogue, staged through shared memory (see epilogue_staged) =====================
        __shared__ __align__(16) uint8_t stage_s[4][2048];
        const int q = warp & 3;                 // TMEM lane quadrant this warp may read (the 4 epilogue warps have distinct ones)
        const uint32_t stg = smem_u32(&stage_s[q][0]);
        const bool vec_ok = ((a.dst_c | a.dst_coff) & (a.out_f16 ? 7 : 3)) == 0;
        const bool lean_ok = a.epi == MR_TC_EPI_STAGED;
        const float slope = a.act == MR_ACT_LEAKY ? a.act_a : 1.0f;
        int lt = 0;
        for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++lt) {
            const int sp = tile / n_phase, phs = tile - sp * n_phase;
            const int b = sp / a.tiles_per_img, t = sp - b * a.tiles_per_img;
            const int tile_y = t / a.tiles_x, tile_x = t - tile_y * a.tiles_x;
            const int buf = lt & 1;
            mbar_wait(tfull0 + 8 * buf, ((uint32_t)lt >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t trow = tmem_d + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * a.n_pad);
            staged_tile<kTileW, kTileH>(a, bias_s, stg, q, lane, b, tile_y, tile_x, trow, lean_ok, vec_ok, slope, a.ph_oy_off[phs],
                                        a.ph_ox_off[phs]);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8 * buf);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(a.tmem_cols));
    }
}

// -------------------------------------------------------------------------------------------------------------------------
// Stride-1 layers with small weights (the full-resolution 24..64-channel layers that dominate the stacks): "halo" variant.
//   * the whole packed weight tensor of the layer is loaded into shared memory ONCE per CTA (resident B);
//   * per (tile, source, K chunk) ONE TMA box {chunk, P px, 16 + kh - 1 px}, P = 8 + kw - 1, brings the input tile with its halo
//     (exactly the pixels the taps touch: a (k x 1) layer loads 8-px rows, a 3 x 3 layer 10-px rows);
//     every filter tap is then just a different shared-memory descriptor into that box: start address shifted by
//     (ky * P + kx) rows of 128 / 64 B, stride between 8-row groups = one halo row (P rows); the swizzle is a function of the
//     absolute shared-memory address, so neither shift needs to be a multiple of the 8-row swizzle atom.
//     L2->SM traffic drops from kh*kw boxes per tile to one.
// Output tile = 16 rows x 8 columns (an 8-row MMA group = 8 adjacent pixels of one output row).
// -------------------------------------------------------------------------------------------------------------------------
// ROWB: bytes per shared-memory row, 128 or 64 (half sources of <= 32 channels)
template <int ROWB>
__global__ void __launch_bounds__(kTcThreads)
conv_tc_halo_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                    const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB, const TcArgs a) {
    extern __shared__ uint8_t smem_raw[];
    constexpr int kBufs = 2;                                     // TMEM accumulators (double-buffered)
    // afull[4], aempty[4], tmem_full[kBufs], tmem_empty[kBufs], bfull, streamed weights: bsfull[8], bsempty[8]
    __shared__ __align__(8) uint64_t bars[2 * 4 + 2 * kBufs + 1 + 16];
    __shared__ uint32_t tmem_base_s;
    __shared__ float bias_s[256];

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // (the broadcast tells ptxas the role branches are warp-uniform)
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    constexpr uint32_t row_bytes = (uint32_t)ROWB;
    const uint32_t b_bytes = (uint32_t)a.n_pad * row_bytes;
    const int chunks_per_tap = a.chunks[0] + a.chunks[1] + a.chunks[2];
    const int taps = a.kh * a.kw;
    const int nbs = a.b_stream;                                                    // weight ring stages (0: resident)
    // bytes in front of the input stages: all weights, or the ring (multiple of 1024: n_pad % 16 == 0)
    const uint32_t bres_bytes = (uint32_t)(nbs > 0 ? nbs : taps * chunks_per_tap) * b_bytes;
    const uint32_t a_bytes = a.halo_a_bytes;                                       // multiple of 1024
    const uint32_t pitch = (uint32_t)a.halo_pitch;
    const uint32_t a_tx = (uint32_t)(16 + a.kh - 1) * pitch * row_bytes;           // bytes one box delivers
    const uint32_t a_base = base + ((bres_bytes + 1023u) & ~1023u);
    const int stages = a.stages;
    const uint32_t afull0 = smem_u32(&bars[0]), aempty0 = smem_u32(&bars[4]);
    const uint32_t tfull0 = smem_u32(&bars[8]), tempty0 = smem_u32(&bars[8 + kBufs]), bfull = smem_u32(&bars[8 + 2 * kBufs]);
    const uint32_t bsfull0 = smem_u32(&bars[9 + 2 * kBufs]), bsempty0 = smem_u32(&bars[17 + 2 * kBufs]);

    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(afull0 + 8 * s, 1); mbar_init(aempty0 + 8 * s, 1); }
        for (int s = 0; s < kBufs; ++s) { mbar_init(tfull0 + 8 * s, 1); mbar_init(tempty0 + 8 * s, 4); }
        mbar_init(bfull, 1);
        for (int s = 0; s < nbs; ++s) { mbar_init(bsfull0 + 8 * s, 1); mbar_init(bsempty0 + 8 * s, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = threadIdx.x; i < 256; i += kTcThreads) bias_s[i] = (a.bias != nullptr && i < a.Cout) ? __ldg(a.bias + i) : 0.f;
    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmA0);
        if (a.n_src > 1) prefetch_tmap(&tmA1);
        if (a.n_src > 2) prefetch_tmap(&tmA2);
        prefetch_tmap(&tmB);
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                     "r"(a.tmem_cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = tmem_base_s;

    if (warp == 0) {
        // ===================== TMA producer (whole warp, converged; the copies are issued by an elected lane) =====================
        // resident weights: every (tap, chunk) slice [n_pad x chunk] once
        if (nbs == 0) {
            mbar_expect_tx_elect(bfull, bres_bytes);
            for (int tp = 0; tp < taps; ++tp)
                for (int cg = 0; cg < chunks_per_tap; ++cg)
                    tma_load_2d_elect(base + (uint32_t)(tp * chunks_per_tap + cg) * b_bytes, &tmB, bfull, cg * a.kc, tp * a.n_pad);
        }
        int st = 0, bs = 0;
        uint32_t ph = 0, bph = 0;
        for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
            const int b = tile / a.tiles_per_img, t = tile - b * a.tiles_per_img;
            const int tile_y = t / a.tiles_x, tile_x = t - tile_y * a.tiles_x;
            const int ix0 = tile_x * 8 - a.pad_l, iy0 = tile_y * 16 - a.pad_t;
            int kbase = 0;
            for (int s = 0; s < a.n_src; ++s) {
                const CUtensorMap* tm = (s == 0) ? &tmA0 : ((s == 1) ? &tmA1 : &tmA2);
                for (int j = 0; j < a.chunks[s]; ++j, kbase += a.kc) {
                    mbar_wait(aempty0 + 8 * st, ph ^ 1u);
                    mbar_expect_tx_elect(afull0 + 8 * st, a_tx);
                    tma_load_4d_elect(a_base + st * a_bytes, tm, afull0 + 8 * st, j * a.kc, ix0, iy0, b);
                    if (++st == stages) { st = 0; ph ^= 1u; }
                    if (nbs > 0) {   // streamed weights: the slices of this chunk, tap by tap, behind its input box
                        int brow = 0;
                        for (int tp = 0; tp < taps; ++tp, brow += a.n_pad) {
                            mbar_wait(bsempty0 + 8 * bs, bph ^ 1u);
                            mbar_expect_tx_elect(bsfull0 + 8 * bs, b_bytes);
                            tma_load_2d_elect(base + (uint32_t)bs * b_bytes, &tmB, bsfull0 + 8 * bs, kbase, brow);
                            if (++bs == nbs) { bs = 0; bph ^= 1u; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (whole warp, converged; the MMAs are issued by an elected lane) =====================
        const uint32_t idesc = a.idesc;
        const uint32_t dhi_a = desc_hi(pitch * row_bytes, row_bytes);      // stride between 8-row groups = one halo row
        const uint32_t dhi_b = desc_hi(8u * row_bytes, row_bytes);
        const uint32_t tap_dx = row_bytes >> 4, tap_dy = (pitch * row_bytes) >> 4;   // descriptor steps of one tap to the right / down
        const uint32_t b_step = b_bytes >> 4;
        if (nbs == 0) mbar_wait(bfull, 0);
        auto run = [&](auto f16tag) {
        constexpr bool kF16 = decltype(f16tag)::value;
        int st = 0, bs = 0, lt = 0;
        uint32_t ph = 0, bph = 0;
        for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++lt) {
            const int buf = lt & (kBufs - 1);
            mbar_wait(tempty0 + 8 * buf, (((uint32_t)lt >> 1) & 1u) ^ 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t acc = tmem_d + (uint32_t)(buf * a.n_pad);
            uint32_t accf = 0;
            int src = 0, jc = 0;                                             // source / chunk inside the source of chunk cg
            for (int cg = 0; cg < chunks_per_tap; ++cg) {
                const int ks = (jc == a.chunks[src] - 1) ? a.tail_ksteps[src] : ROWB / 32;
                if (++jc == a.chunks[src]) { jc = 0; ++src; }
                mbar_wait(afull0 + 8 * st, ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                uint32_t alo_row = desc_lo(a_base + st * a_bytes);
                uint32_t blo = desc_lo(base) + (uint32_t)cg * b_step;                 // resident: slice (tap 0, chunk cg)
                for (int ky = 0; ky < a.kh; ++ky, alo_row += tap_dy) {
                    uint32_t alo = alo_row;
                    for (int kx = 0; kx < a.kw; ++kx, alo += tap_dx) {
                        if (nbs > 0) {
                            mbar_wait(bsfull0 + 8 * bs, bph);
                            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                            blo = desc_lo(base + (uint32_t)bs * b_bytes);
                        }
#pragma unroll
                        for (int k = 0; k < ROWB / 32; ++k) {   // 32 bytes of K per MMA (8 tf32 / 16 half): 4 per 128-byte row, 2 per 64-byte row
                            if (k < ks) umma_elect<kF16>(acc, alo + 2 * k, dhi_a, blo + 2 * k, dhi_b, idesc, accf);
                            accf = 1u;
                        }
                        if (nbs > 0) {
                            umma_commit_elect(bsempty0 + 8 * bs);   // frees the weight stage once these MMAs have read it
                            if (++bs == nbs) { bs = 0; bph ^= 1u; }
                        } else {
                            blo += (uint32_t)chunks_per_tap * b_step;   // next tap, same chunk
                        }
                    }
                }
                umma_commit_elect(aempty0 + 8 * st);
                if (cg == chunks_per_tap - 1) umma_commit_elect(tfull0 + 8 * buf);
                if (++st == stages) { st = 0; ph ^= 1u; }
            }
        }
        };
        if (a.f16) run(std::true_type{}); else run(std::false_type{});
    } else {
        // ===================== epilogue, staged through shared memory (tile = 16 rows x 8 columns) =====================
        __shared__ __align__(16) uint8_t stage_s[4][2048];
        const int q = warp & 3;                 // TMEM lane quadrant
        const uint32_t stg = smem_u32(&stage_s[warp - 2][0]);
        const bool vec_ok = ((a.dst_c | a.dst_coff) & (a.out_f16 ? 7 : 3)) == 0;
        const bool lean_ok = a.epi == MR_TC_EPI_STAGED;
        const float slope = a.act == MR_ACT_LEAKY ? a.act_a : 1.0f;
        int lt = 0;
        for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++lt) {
            const int b = tile / a.tiles_per_img, t = tile - b * a.tiles_per_img;
            const int tile_y = t / a.tiles_x, tile_x = t - tile_y * a.tiles_x;
            const int buf = lt & (kBufs - 1);
            mbar_wait(tfull0 + 8 * buf, ((uint32_t)lt >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t trow = tmem_d + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * a.n_pad);
            staged_tile<8, 16>(a, bias_s, stg, q, lane, b, tile_y, tile_x, trow, lean_ok, vec_ok, slope, a.oy_off, a.ox_off);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8 * buf);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(a.tmem_cols));
    }
}

// ---- host side: tensor maps ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;   // benign race: every thread resolves the same pointer
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

}  // namespace

// The launch plan: argument checks, kernel choice, ring depths, grid and epilogue of one call, on the host without the driver.
// `a` receives the kernel arguments (everything but the tensor maps, which need the driver).
static int conv2d_nhwc_tc_plan_impl(const mr_conv_desc* desc, int n_phases, int n_pad, int k_pad, int round_out, int sms,
                                    mr_conv_tc_plan* plan, TcArgs& a) {
    MR_REQUIRE(desc != nullptr, "mr_conv2d_nhwc_tc: null descriptor");
    MR_REQUIRE(n_phases >= 1 && n_phases <= 4, "mr_conv2d_nhwc_tc_phases: 1..4 phases (got %d)", n_phases);
    MR_REQUIRE(sms >= 1, "mr_conv2d_nhwc_tc_plan: sms=%d", sms);
    const mr_conv_desc& d = desc[0];
    for (int p = 1; p < n_phases; ++p) {   // phases share everything but the filter (size, padding, weights) and the output offset
        const mr_conv_desc& e = desc[p];
        bool same = e.n_src == d.n_src && e.B == d.B && e.Hs == d.Hs && e.Ws == d.Ws && e.upsample2 == d.upsample2 && e.sy == d.sy &&
                    e.sx == d.sx && e.Ho == d.Ho && e.Wo == d.Wo && e.Cout == d.Cout && e.bias == d.bias && e.dst == d.dst &&
                    e.dst_H == d.dst_H && e.dst_W == d.dst_W && e.dst_c == d.dst_c && e.dst_coff == d.dst_coff &&
                    e.oy_step == d.oy_step && e.ox_step == d.ox_step && e.act == d.act && e.act_a == d.act_a && e.act_b == d.act_b &&
                    e.src_dtype == d.src_dtype && e.dst_dtype == d.dst_dtype;
        for (int s = 0; same && s < d.n_src && s < MR_CONV_MAX_SRC; ++s) same = e.src[s] == d.src[s] && e.src_c[s] == d.src_c[s];
        MR_REQUIRE(same, "mr_conv2d_nhwc_tc_phases: phase %d differs from phase 0 in more than filter size, padding, weights and output offset", p);
        MR_REQUIRE(e.weight && e.kh >= 1 && e.kw >= 1 && (e.Ho - 1) * e.oy_step + e.oy_off < e.dst_H && (e.Wo - 1) * e.ox_step + e.ox_off < e.dst_W,
                   "mr_conv2d_nhwc_tc_phases: phase %d: bad filter / output placement", p);
        MR_REQUIRE((reinterpret_cast<uintptr_t>(e.weight) & 15) == 0, "mr_conv2d_nhwc_tc_phases: weights are not 16-byte aligned");
    }
    MR_REQUIRE(d.n_src >= 1 && d.n_src <= MR_CONV_MAX_SRC, "mr_conv2d_nhwc_tc: n_src=%d out of range", d.n_src);
    MR_REQUIRE(d.upsample2 == 0, "mr_conv2d_nhwc_tc: upsample-on-read is expressed as sub-pixel convolutions on this path");
    MR_REQUIRE(d.weight && d.dst, "mr_conv2d_nhwc_tc: null weight/dst");
    MR_REQUIRE(d.Cout >= 1 && d.Cout <= 256 && n_pad >= d.Cout && n_pad <= 256 && (n_pad % 16) == 0,
               "mr_conv2d_nhwc_tc: Cout=%d n_pad=%d unsupported (Cout <= 256, n_pad multiple of 16)", d.Cout, n_pad);
    MR_REQUIRE(d.B >= 1 && d.B <= 65535 && d.Hs >= 1 && d.Ws >= 1 && d.Ho >= 1 && d.Wo >= 1, "mr_conv2d_nhwc_tc: bad shape");
    MR_REQUIRE(d.kh >= 1 && d.kw >= 1 && d.sy >= 1 && d.sx >= 1 && d.sy <= 4 && d.sx <= 4, "mr_conv2d_nhwc_tc: bad kernel/stride");
    MR_REQUIRE(d.dst_coff >= 0 && d.dst_coff + d.Cout <= d.dst_c, "mr_conv2d_nhwc_tc: channel slice out of range");
    MR_REQUIRE((d.Ho - 1) * d.oy_step + d.oy_off < d.dst_H && (d.Wo - 1) * d.ox_step + d.ox_off < d.dst_W,
               "mr_conv2d_nhwc_tc: output placement out of range");
    MR_REQUIRE(d.act >= MR_ACT_NONE && d.act <= MR_ACT_ABSTANH, "mr_conv2d_nhwc_tc: unknown activation %d", d.act);
    MR_REQUIRE(d.src_dtype == MR_DT_F32 || d.src_dtype == MR_DT_F16, "mr_conv2d_nhwc_tc: bad src_dtype %d", d.src_dtype);
    MR_REQUIRE(d.dst_dtype == MR_DT_F32 || d.dst_dtype == MR_DT_F16, "mr_conv2d_nhwc_tc: bad dst_dtype %d", d.dst_dtype);
    a.n_src = d.n_src;
    const bool f16 = d.src_dtype == MR_DT_F16;
    // K chunk = one swizzle row of channels: 32 fp32 or 64 half (128 bytes).  Half sources whose channel counts waste less
    // with 32-channel chunks (32, 96, ... channels) are packed that way by the caller (k_pad tells): 64-byte rows, SWIZZLE_64B,
    // so that neither TMA nor the MMA spends time on the zero half of a 128-byte row.
    int kc = f16 ? 64 : kKC;
    if (f16) {
        int k64 = 0, k32 = 0;
        for (int s = 0; s < d.n_src; ++s) { k64 += (d.src_c[s] + 63) / 64 * 64; k32 += (d.src_c[s] + 31) / 32 * 32; }
        if (k_pad != k64 && k_pad == k32) kc = 32;
    }
    const int esize = f16 ? 2 : 4;
    const int cmult = f16 ? 8 : 4;            // pixel stride must be a multiple of 16 bytes for TMA
    a.row_bytes = kc * (f16 ? 2 : 4);
    a.kc = kc; a.f16 = f16 ? 1 : 0; a.out_f16 = (d.dst_dtype == MR_DT_F16) ? 1 : 0;
    // UMMA instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 = 1 @[4,6); a/b format @[7,10)/[10,13): TF32 = 2,
    // F16 = 0; K-major A and B; N >> 3 @[17,23); M >> 4 @[24,29)
    a.idesc = (1u << 4) | ((f16 ? 0u : 2u) << 7) | ((f16 ? 0u : 2u) << 10) | ((uint32_t)(n_pad >> 3) << 17) | ((128u >> 4) << 24);
    int ksum = 0;
    for (int s = 0; s < d.n_src; ++s) {
        const int C = d.src_c[s];
        MR_REQUIRE(d.src[s] != nullptr && C >= cmult && (C % cmult) == 0,
                   "mr_conv2d_nhwc_tc: source %d needs a channel count that is a multiple of %d (got %d)", s, cmult, C);
        MR_REQUIRE((reinterpret_cast<uintptr_t>(d.src[s]) & 15) == 0, "mr_conv2d_nhwc_tc: source %d is not 16-byte aligned", s);
        a.chunks[s] = (C + kc - 1) / kc;
        a.tail_ksteps[s] = ((C - (a.chunks[s] - 1) * kc) * esize + 31) / 32;
        ksum += a.chunks[s] * kc;
    }
    MR_REQUIRE(ksum == k_pad, "mr_conv2d_nhwc_tc: packed weight K (%d) does not match the sources (%d)", k_pad, ksum);
    MR_REQUIRE((reinterpret_cast<uintptr_t>(d.weight) & 15) == 0, "mr_conv2d_nhwc_tc: weights are not 16-byte aligned");
    // "halo" variant (one input box per tile, resident weights): stride 1, taps reach at most 8 px to the right, weights fit
    int chunks_all = 0;
    for (int s = 0; s < d.n_src; ++s) chunks_all += (d.src_c[s] + kc - 1) / kc;
    const size_t bres = (size_t)d.kh * d.kw * chunks_all * n_pad * a.row_bytes;
    // MONOREC_B200_TC_HALO: unset = automatic, 0 = never, n = 1..4: at most n CTAs per SM (1: also layers that only fit once).
    // History of the rule: with 16-px box rows only the 32-channel layers fitted twice per SM (32->32 3x3 over the single-frame
    // volumes: 631 -> 452 us in TF32, 489 -> 203 us in half) and one CTA per SM lost to the tap-refetch kernel (48->48 3x3:
    // 300 -> 335 us); with (8 + kw - 1)-px rows the 48-channel full-resolution layers fit twice as well (profiles/r02_k2_pitch.txt).
    static const int halo_env = getenv("MONOREC_B200_TC_HALO") ? atoi(getenv("MONOREC_B200_TC_HALO")) : -1;
    static const bool halo_f16 = getenv("MONOREC_B200_TC_HALO_F16") ? (atoi(getenv("MONOREC_B200_TC_HALO_F16")) != 0) : true;
    // (64-byte rows are fine inside the halo box too: half sources of <= 32 channels packed with 32-channel chunks; measured
    // 429 -> 203 us on the 32->32 3x3 layer over the single-frame volumes, profiles/r02_k2_variants.txt)
    // MONOREC_B200_TC_HALO_PITCH=16: the fixed 16-px rows of the first halo kernel (A/B measurements)
    static const int pitch_env = getenv("MONOREC_B200_TC_HALO_PITCH") ? atoi(getenv("MONOREC_B200_TC_HALO_PITCH")) : 0;
    const int halo_pitch = (pitch_env >= 8 + d.kw - 1) ? pitch_env : 8 + d.kw - 1;
    const size_t halo_a_bytes = ((size_t)(16 + d.kh - 1) * halo_pitch * a.row_bytes + 1023) & ~size_t(1023);
    const size_t bres_al = (bres + 1023) & ~size_t(1023);
    uint32_t halo_cols = 32;               // TMEM columns one CTA allocates (two accumulators)
    while (halo_cols < (uint32_t)(2 * n_pad)) halo_cols <<= 1;
    auto halo_fit = [&](int ctas) {   // A stages that fit next to the resident weights with `ctas` CTAs per SM
        if ((uint32_t)ctas * halo_cols > 512) return 0;
        // 228 KB per SM, 1 KB reserved per CTA; static per CTA: 8 KB epilogue staging + 1 KB bias + barriers; 1 KB alignment slack
        const size_t budget = (size_t)(ctas == 1 ? 210 : 228) * 1024 / ctas - (1 + 8 + 1 + 1) * 1024 - 512;
        int st = bres_al + 1024 < budget ? (int)((budget - 1024 - bres_al) / halo_a_bytes) : 0;
        return st > 4 ? 4 : st;
    };
    // CTAs per SM: up to three, each with at least two input stages (up to 4).  Measured after the issue loops moved to the
    // uniform datapath (profiles/r02_k2_ctas2.txt): cap 2 / 3 / 4 -> half-mode forward 3.98 / 3.94 / 4.06 ms, 32->32 3x3 over
    // the single-frame volumes 159 / 143 / 193 us (before that change 3-4 CTAs were slower than 2: profiles/r02_k2_ctas.txt).
    // MONOREC_B200_TC_HALO=n (1..4) caps / forces the count for measurements (1: also layers that only fit once).
    int halo_ctas = 0;
    if (n_phases == 1 && halo_env != 0 && (!f16 || halo_f16) && d.sy == 1 && d.sx == 1 && d.kw <= 9 && d.kh <= 7) {
        const int cap = (halo_env >= 1 && halo_env <= 4) ? halo_env : 3;
        for (int c = cap; c >= (halo_env == 1 ? 1 : 2) && halo_ctas == 0; --c)
            if (halo_fit(c) >= 2) halo_ctas = c;
    }
    // Weights that do not fit next to two input stages stream instead: the [n_pad x chunk] slice of each (chunk, tap) goes through
    // a ring of 3..8 stages behind the chunk's input box.  Per tile that is all the weights once (L2 hits) plus ONE input box per
    // chunk, against kh*kw input boxes + the same weights in the tap-refetch kernel -- the multi-source decoder layers were bound
    // by that L2->SM traffic (~12.7 TB/s aggregate on the 32+64->48 3x3 layer).  MONOREC_B200_TC_STREAM=0 disables it (A/B).
    static const bool stream_on = getenv("MONOREC_B200_TC_STREAM") ? (atoi(getenv("MONOREC_B200_TC_STREAM")) != 0) : true;
    int b_stream = 0, stream_stages = 0;
    const size_t b_slice = (size_t)n_pad * a.row_bytes;
    if (halo_ctas == 0 && stream_on && n_phases == 1 && halo_env != 0 && (!f16 || halo_f16) && d.sy == 1 && d.sx == 1 && d.kw <= 9 &&
        d.kh <= 7 && d.kh * d.kw > 1 && 2 * halo_cols <= 512) {
        const size_t budget = (size_t)228 * 1024 / 2 - (1 + 8 + 1 + 1) * 1024 - 512 - 1024;
        if (budget > 2 * halo_a_bytes + 3 * b_slice) {
            int nb = (int)((budget - 2 * halo_a_bytes) / b_slice);
            if (nb > 8) nb = 8;
            int st = (int)((budget - (size_t)nb * b_slice) / halo_a_bytes);
            b_stream = nb;
            stream_stages = st > 4 ? 4 : st;
            halo_ctas = 2;
        }
    }
    const bool halo = halo_ctas > 0;
    a.n_phase = n_phases;
    for (int p = 0; p < 4; ++p) {
        const mr_conv_desc& e = desc[p < n_phases ? p : 0];
        a.ph_kh[p] = e.kh; a.ph_kw[p] = e.kw; a.ph_pad_t[p] = e.pad_t; a.ph_pad_l[p] = e.pad_l; a.ph_oy_off[p] = e.oy_off; a.ph_ox_off[p] = e.ox_off;
    }
    a.kh = d.kh; a.kw = d.kw; a.sy = d.sy; a.sx = d.sx; a.pad_t = d.pad_t; a.pad_l = d.pad_l;
    a.Ho = d.Ho; a.Wo = d.Wo; a.Cout = d.Cout; a.n_pad = n_pad;
    a.tiles_x = halo ? (d.Wo + 7) / 8 : (d.Wo + kTileW - 1) / kTileW;
    const int tiles = a.tiles_x * (halo ? (d.Ho + 15) / 16 : (d.Ho + kTileH - 1) / kTileH);
    a.tiles_per_img = tiles;
    a.total_tiles = tiles * d.B * n_phases;
    // tap-refetch kernel, persistent grid: resident CTAs per SM bounded by TMEM (each CTA holds a power-of-two >= 2 * n_pad columns
    // of the 512) and capped at 4; with UMMA N = 32..64 one CTA cannot keep the tensor pipe busy, so several CTAs interleave
    // their MMA chains; the ring takes what shared memory is left
    static const int kForceCtas = getenv("MONOREC_B200_TC_CTAS") ? atoi(getenv("MONOREC_B200_TC_CTAS")) : 0;   // tuning knob
    uint32_t cols = 32;
    while (cols < (uint32_t)(2 * n_pad)) cols <<= 1;
    a.tmem_cols = cols;
    int ctas_per_sm = (int)(512 / cols);
    if (ctas_per_sm > 4) ctas_per_sm = 4;
    if (kForceCtas > 0 && (uint32_t)kForceCtas * cols <= 512) ctas_per_sm = kForceCtas;
    const size_t stage_bytes = (size_t)(128 + n_pad) * a.row_bytes;
    int stages = (int)(((size_t)(200 * 1024) / ctas_per_sm - 8 * 1024) / stage_bytes);
    if (stages > 8) stages = 8;
    if (stages < 2) stages = 2;
    size_t smem = (size_t)stages * stage_bytes + 1024;
    if (halo) {
        ctas_per_sm = halo_ctas;
        stages = b_stream ? stream_stages : halo_fit(halo_ctas);
        const size_t halo_front = b_stream ? (size_t)b_stream * b_slice : bres_al;   // bytes in front of the input stages
        smem = halo_front + (size_t)stages * halo_a_bytes + 1024;
        a.halo_pitch = halo_pitch;
        a.halo_a_bytes = (uint32_t)halo_a_bytes;
        a.b_stream = b_stream;
    }
    a.stages = stages;
    a.bias = d.bias; a.dst = d.dst;
    a.dst_H = d.dst_H; a.dst_W = d.dst_W; a.dst_c = d.dst_c; a.dst_coff = d.dst_coff;
    a.oy_step = d.oy_step; a.ox_step = d.ox_step; a.oy_off = d.oy_off; a.ox_off = d.ox_off;
    a.act = d.act; a.act_a = d.act_a; a.act_b = d.act_b; a.round_out = round_out;
    // staged epilogue: 16-byte stores of whole channel groups, no activation or LeakyReLU; one-channel heads take one accumulator
    // column; anything else (unaligned channel slices, Cout not a multiple of 4 / 8, sigmoid / |tanh| with Cout > 1) is generic
    const int vmask = a.out_f16 ? 7 : 3;
    if (((d.dst_c | d.dst_coff | d.Cout) & vmask) == 0 && !(a.out_f16 && round_out) && (d.act == MR_ACT_NONE || d.act == MR_ACT_LEAKY))
        a.epi = MR_TC_EPI_STAGED;
    else
        a.epi = d.Cout == 1 ? MR_TC_EPI_ONE_COLUMN : MR_TC_EPI_GENERIC;
    int grid = sms * ctas_per_sm;
    if (grid > a.total_tiles) grid = a.total_tiles;
    plan->kernel = !halo ? MR_TC_REFETCH : (b_stream ? MR_TC_HALO_STREAM : MR_TC_HALO);
    plan->ctas_per_sm = ctas_per_sm;
    plan->stages = stages;
    plan->b_stream = b_stream;
    plan->row_bytes = a.row_bytes;
    plan->kc = kc;
    plan->tmem_cols = (int)cols;
    plan->smem_bytes = (int)smem;
    plan->total_tiles = a.total_tiles;
    plan->grid = grid;
    plan->epilogue = a.epi;
    return MR_OK;
}

extern "C" int mr_conv2d_nhwc_tc_plan(const mr_conv_desc* descs, int n_phases, int n_pad, int k_pad, int round_out, int sms,
                                      mr_conv_tc_plan* out) {
    MR_REQUIRE(out != nullptr, "mr_conv2d_nhwc_tc_plan: null plan");
    TcArgs a{};
    return conv2d_nhwc_tc_plan_impl(descs, n_phases, n_pad, k_pad, round_out, sms, out, a);
}

static int conv2d_nhwc_tc_impl(const mr_conv_desc* desc, int n_phases, int n_pad, int k_pad, int round_out, void* stream) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    TcArgs a{};
    mr_conv_tc_plan plan{};
    const int prc = conv2d_nhwc_tc_plan_impl(desc, n_phases, n_pad, k_pad, round_out, sms, &plan, a);
    if (prc != MR_OK) return prc;
    EncodeTiledFn encode = get_encode_fn();
    if (encode == nullptr) {
        mr::set_error("mr_conv2d_nhwc_tc: cuTensorMapEncodeTiled is not available from this driver");
        return MR_ENOSUPPORT;
    }
    const mr_conv_desc& d = desc[0];
    const bool halo = plan.kernel != MR_TC_REFETCH;
    const int esize = a.f16 ? 2 : 4;
    const CUtensorMapDataType dtype = a.f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    const CUtensorMapSwizzle swizzle = a.row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    CUtensorMap tmA[MR_CONV_MAX_SRC];
    for (int s = 0; s < d.n_src; ++s) {
        const int C = d.src_c[s];
        const cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)d.Ws, (cuuint64_t)d.Hs, (cuuint64_t)d.B};
        const cuuint64_t gstr[3] = {(cuuint64_t)C * esize, (cuuint64_t)d.Ws * C * esize, (cuuint64_t)d.Hs * d.Ws * C * esize};
        // with a traversal stride s the box spans box/s loaded elements: 16 (8) output pixels need a span of 16*s (8*s)
        cuuint32_t box[4] = {(cuuint32_t)a.kc, (cuuint32_t)(kTileW * d.sx), (cuuint32_t)(kTileH * d.sy), 1};
        if (halo) { box[1] = (cuuint32_t)a.halo_pitch; box[2] = (cuuint32_t)(16 + d.kh - 1); }
        const cuuint32_t estr[4] = {1, (cuuint32_t)d.sx, (cuuint32_t)d.sy, 1};
        CUresult r = encode(&tmA[s], dtype, 4, const_cast<float*>(d.src[s]), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            mr::set_error("mr_conv2d_nhwc_tc: cuTensorMapEncodeTiled(A%d) failed with CUresult %d", s, (int)r);
            return MR_EINVAL;
        }
    }
    for (int s = d.n_src; s < MR_CONV_MAX_SRC; ++s) tmA[s] = tmA[0];
    CUtensorMap tmBs[4];
    for (int p = 0; p < n_phases; ++p) {
        const mr_conv_desc& e = desc[p];
        const cuuint64_t gdim[2] = {(cuuint64_t)k_pad, (cuuint64_t)e.kh * e.kw * n_pad};
        const cuuint64_t gstr[1] = {(cuuint64_t)k_pad * esize};
        const cuuint32_t box[2] = {(cuuint32_t)a.kc, (cuuint32_t)n_pad};
        const cuuint32_t estr[2] = {1, 1};
        CUresult r = encode(&tmBs[p], dtype, 2, const_cast<float*>(e.weight), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            mr::set_error("mr_conv2d_nhwc_tc: cuTensorMapEncodeTiled(B) failed with CUresult %d", (int)r);
            return MR_EINVAL;
        }
    }
    for (int p = n_phases; p < 4; ++p) tmBs[p] = tmBs[0];
    const size_t smem = (size_t)plan.smem_bytes;
    if (halo) {
        auto launch_halo = [&](auto kernel) -> int {
            MR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(212 * 1024)));
            kernel<<<plan.grid, kTcThreads, smem, (cudaStream_t)stream>>>(tmA[0], tmA[1], tmA[2], tmBs[0], a);
            return MR_OK;
        };
        const int lrc = a.row_bytes == 128 ? launch_halo(conv_tc_halo_kernel<128>) : launch_halo(conv_tc_halo_kernel<64>);
        if (lrc != MR_OK) return lrc;
        MR_LAUNCH_CHECK("conv_tc_halo_kernel");
        return MR_OK;
    }
    MR_CUDA(cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(212 * 1024)));
    conv_tc_kernel<<<plan.grid, kTcThreads, smem, (cudaStream_t)stream>>>(tmA[0], tmA[1], tmA[2], tmBs[0], tmBs[1], tmBs[2], tmBs[3], a);
    MR_LAUNCH_CHECK("conv_tc_kernel");
    return MR_OK;
}

extern "C" int mr_conv2d_nhwc_tc(const mr_conv_desc* desc, int n_pad, int k_pad, int round_out, void* stream) {
    return conv2d_nhwc_tc_impl(desc, 1, n_pad, k_pad, round_out, stream);
}

extern "C" int mr_conv2d_nhwc_tc_phases(const mr_conv_desc* descs, int n_phases, int n_pad, int k_pad, int round_out, void* stream) {
    return conv2d_nhwc_tc_impl(descs, n_phases, n_pad, k_pad, round_out, stream);
}
