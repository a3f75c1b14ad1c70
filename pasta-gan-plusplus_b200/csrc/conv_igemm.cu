// Implicit-GEMM convolution for sm_100a: tcgen05.mma with TMEM accumulators, TMA operand loads,
// mbarrier pipeline, warp-specialised persistent CTAs, fused modulated-conv epilogue.
//
//   GEMM view      D[pixel, g] = sum_{tap, c} A[pixel shifted by tap, c] * B[tap][g][c]
//   M (TMEM lanes) 128 output pixels: a TN x TH x TW block of (sample, row, column)
//   N (columns)    block_n GEMM columns g = phase * O + oc
//   K              taps x c_pad, walked in blocks of kb channels (kb * 2 bytes = one swizzle row)
//
// The A tile of a K step is one TMA box {kb, TW, TH, TN, 1} of the channels-innermost activation
// tensor at the tap's (dx, dy) offset; rows outside the image come back as zeros (TMA out-of-bounds
// fill), which is exactly the convolution's zero padding - no im2col buffer exists anywhere.
// The split-precision ("fp32 parity") mode runs the same loop over products (a_part, b_part) of
// the bf16 expansions of both operands, all accumulated in the same fp32 TMEM tile.
//
// Operand traffic (the C<=128 layers are bounded by L2->SM bandwidth, not by the tensor pipe, unless tiles are reused):
//   * ky reuse: for stride-1 convs the producer loads one activation slab of (TH + kh - 1) image rows per (kx, channel
//     block) and the kh vertical taps are issued from row-shifted views of it (descriptor start + ky*TW rows; the
//     shift is a multiple of the 8-row swizzle atom, so no re-swizzling is involved);
//   * product sharing: all bf16 parts of A (slabs) and B (tiles) are loaded once per K group and every product
//     (a_part, b_part) of the split-precision mode is issued from them;
//   * resident weights: when all weight tiles of a column tile fit next to the activation ring (64->64 3x3, ToRGB)
//     they are loaded once per CTA and stay in shared memory for every pixel tile the CTA processes.
//
// Warp roles (320 threads, 1 CTA per SM):
//   warp 0      TMA producer        (one elected lane)
//   warp 1      TMEM owner + tcgen05.mma issuer (one elected lane)
//   warps 2-9   epilogue (two warps per TMEM lane quarter, each half of the columns): tcgen05.ld -> demod / noise /
//               bias / activation / clamp -> global store
// Accumulators are double-buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// Replaces the cuDNN calls of torch_utils/ops/conv2d_gradfix.py:38,43,112-114 and the grouped-conv
// formulation of training/networks.py:85-93 (algebraically the non-fused form, networks.py:73-82).
#include <cuda.h>
#include <stdlib.h>
#include <atomic>
#include <type_traits>
#include "act.cuh"
#include "tc_ptx.cuh"

namespace pgpp {

constexpr int kThreads = 320;      // 2 control warps + 8 epilogue warps

constexpr int kTileM = 128;

struct IgemmParams {
    int n, h, w;
    int conv_h, conv_w;
    int kh, kw, pad_y, pad_x, stride;
    int num_cb, kb;
    int parts;                          // bf16 parts used of each operand (1, 2, 3)
    unsigned pa_mask[3];                // pa_mask[pb]: which A parts multiply B part pb
    int n_groups, inner;                // K groups per channel block (kw with ky reuse, kh*kw without) and taps per group (kh or 1)
    int reuse;                          // 1: one activation slab per (kx, cb), vertical taps are row-shifted views;
                                        // 2: ONE slab with an x halo per (cb, part), every tap is a row-shifted view (mma_role_slab)
    unsigned short tap_off16[64];       // reuse == 2: descriptor start offset of tap j inside the slab, in 16-byte units
    unsigned sbo_a;                     // reuse == 2: 8-row group stride of the A operand = slab row pitch in bytes
    int o, phases, phase_stride, o_rows, block_n;
    int tw, th, tn;
    int tiles_x, tiles_y, tiles_n, tiles_col;
    long long total_tiles;
    int a_stages, b_stages, b_resident;
    unsigned slab_bytes;                // one A part of one stage (= bytes of one activation TMA box)
    unsigned a_stage_bytes;             // stage pitch: parts * slab_bytes rounded up to 1024
    unsigned a_tx_bytes;                // parts * slab_bytes: bytes the activation TMA boxes of one stage deliver
    unsigned b_bytes, b_pitch;          // bytes of one weight TMA box, slot pitch (1024-byte multiple)
    unsigned ky_step_bytes;             // TW * row_bytes: shift of the slab view per vertical tap
    unsigned layout_type, sbo_bytes;
    unsigned idesc;
    unsigned tmem_cols;
    const float* dcoef; const float* noise; long long noise_stride_n; const float* bias;
    int act_fn; float alpha, gain, clamp;
    void* out; int out_dtype; int out_h, out_w; long long os_n, os_c, os_h, os_w;
    int accumulate;
    int up;     // 1, or 2 when phases == 4
    int wgt_per_sample;                 // weights carry a leading sample dimension
    int out_parts; long long out_part_stride;
    const float* spade_x; const float* spade_mean; const float* spade_rstd; float spade_pre_gain;   // SPADE epilogue (see epilogue_spade)
    int stack;                          // 1: split-precision products a0 x [b0; b1] issued as ONE N = 2 * block_n MMA (see mma_role)
    int acc_cols;                       // TMEM columns per accumulator buffer (block_n, or 2 * block_n when stack)
    unsigned idesc_stack;               // instruction descriptor with N = 2 * block_n
    int fold_gain;                      // activation is positively homogeneous and gain > 0: gain is folded into scale/shift/noise
    unsigned div_col_m, div_col_s, div_x_m, div_x_s, div_y_m, div_y_s;   // magic numbers for t / tiles_col, / tiles_x, / tiles_y
    float* stats_ws; long long stats_plane;    // instance-norm partials of the output: [3][stats_plane / o][o] (see pgpp_conv_desc.stats_ws)
    int slab9;                          // reuse == 2 with a 3 x 3 filter, 64-channel rows and 64-column weight tiles: mma_role_slab9 (compile-time descriptor offsets)
    int dbg;                            // PGPP_IGEMM_DEBUG ablation bits (timing experiments only, results are wrong): 1 epilogue without
                                        // arithmetic / stores, 2 without TMEM loads, 4 no MMAs issued, 8 arithmetic but no stores, 16 stores go to one
                                        // tile-sized region (no DRAM write traffic), 32 128-bit instead of 256-bit stores of the operand format, 64 no activation loads (the MMA warp
                                        // does not wait for them: MMA issue + tensor time alone)
    const float* wscale;                // e4m3 operands: per-GEMM-column weight scale [o_rows] (per sample: [n][o_rows]), folded into the epilogue scale
};

// column scale of the e4m3 weights (fp8 inference precision) for sample n, GEMM column g
__device__ __forceinline__ float weight_scale(const IgemmParams& p, int n, int g) {
    return __ldg(p.wscale + (p.wgt_per_sample ? (long long)n * p.o_rows : 0ll) + g);
}


// ------------------------------------------------------------------------------------------------

struct TileCoord { int n0, y0, x0, col0; };

// n / d for n < 2^31 with host-computed m = ceil(2^(31+s) / d), s = ceil(log2 d)
__device__ __forceinline__ unsigned fast_div(unsigned n, unsigned m, unsigned s) {
    return (unsigned)(((unsigned long long)n * m) >> (31 + s));
}

__device__ __forceinline__ TileCoord decode_tile(const IgemmParams& p, long long tt) {
    TileCoord c;
    unsigned t = (unsigned)tt, q;
    q = fast_div(t, p.div_col_m, p.div_col_s); c.col0 = (int)(t - q * p.tiles_col) * p.block_n; t = q;   // column tiles fastest: neighbours share A in L2
    q = fast_div(t, p.div_x_m, p.div_x_s);     c.x0 = (int)(t - q * p.tiles_x) * p.tw; t = q;
    q = fast_div(t, p.div_y_m, p.div_y_s);     c.y0 = (int)(t - q * p.tiles_y) * p.th; t = q;
    c.n0 = (int)t * p.tn;
    return c;
}

struct PixelCoord { int px, py, pn; };

template <class OT> struct IsBf16 { static constexpr bool value = false; };
template <> struct IsBf16<__nv_bfloat16> { static constexpr bool value = true; };
template <class OT> __device__ __forceinline__ OT cvt_out(float v);
template <> __device__ __forceinline__ float cvt_out<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 cvt_out<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half cvt_out<__half>(float v) { return __float2half_rn(v); }
template <class OT> __device__ __forceinline__ float cvt_in(OT v);
template <> __device__ __forceinline__ float cvt_in<float>(float v) { return v; }
template <> __device__ __forceinline__ float cvt_in<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float cvt_in<__half>(__half v) { return __half2float(v); }

// General epilogue of one accumulator tile for the calling warp: its 32 TMEM lanes (pixels) x columns
// [col_begin, col_end).  Handles every option (several samples per tile, accumulate, partial chunks, any activation).
template <int A, class OT, bool F8>
__device__ __forceinline__ void epilogue_general(const IgemmParams& p, const TileCoord tc, uint32_t tmem_tile, const PixelCoord pc,
                                                 int col_begin, int col_end) {
    const int x = tc.x0 + pc.px, y = tc.y0 + pc.py, n = tc.n0 + pc.pn;
    const bool pix_ok = x < p.conv_w && y < p.conv_h && n < p.n;
    const int total_cols = p.phases * p.phase_stride;
    OT* const out = (OT*)p.out;
    const float alpha = p.alpha, gain = p.gain, clamp = p.clamp;
    const long long cs = p.os_c;

    for (int c0 = col_begin; c0 < col_end; c0 += 16) {
        float v[16];
        tmem_ld16(tmem_tile + c0, v);       // warp-collective: executed by all lanes, valid pixel or not
        const int g0 = tc.col0 + c0;
        if (!pix_ok || g0 >= total_cols) continue;
        const int phase = (g0 >= p.phase_stride) + (g0 >= 2 * p.phase_stride) + (g0 >= 3 * p.phase_stride);
        const int oc0 = g0 - phase * p.phase_stride;        // a 16-column chunk never straddles phases (phase_stride % 16 == 0)
        if (oc0 >= p.o) continue;                           // padding columns between phases
        const int oy = y * p.up + (phase >> 1), ox = x * p.up + (phase & 1);
        float nz = 0.f;
        if (p.noise) nz = __ldg(p.noise + n * p.noise_stride_n + (long long)oy * p.out_w + ox);
        const long long base = n * p.os_n + oy * p.os_h + ox * p.os_w;
        const int valid = min(16, p.o - oc0);
        #pragma unroll
        for (int j = 0; j < 16; j++) {
            if (j < valid) {
                const int oc = oc0 + j;
                float r = v[j];
                if (p.dcoef) r *= __ldg(p.dcoef + (long long)n * p.o + oc);
                if (F8) r *= weight_scale(p, n, g0 + j);
                r += nz;
                if (p.bias) r += __ldg(p.bias + oc);
                r = act_forward<A, float>(r, alpha) * gain;
                if (clamp >= 0.f) r = fminf(fmaxf(r, -clamp), clamp);
                v[j] = r;
            }
        }
        if (cs == 1 && valid == 16 && !p.accumulate && ((base + oc0) * sizeof(OT)) % 16 == 0 && ((uintptr_t)out & 15) == 0) {
            for (int part = 0; part < p.out_parts; part++) {
                __align__(16) OT tmp[16];
                #pragma unroll
                for (int j = 0; j < 16; j++) { tmp[j] = cvt_out<OT>(v[j]); v[j] -= cvt_in<OT>(tmp[j]); }
                int4* dst = reinterpret_cast<int4*>(out + part * p.out_part_stride + base + oc0);
                const int4* src = reinterpret_cast<const int4*>(tmp);
                #pragma unroll
                for (int q = 0; q < (int)(16 * sizeof(OT) / 16); q++) dst[q] = src[q];
            }
        } else {
            OT* dst = out + base + (long long)oc0 * cs;
            #pragma unroll
            for (int j = 0; j < 16; j++) {
                if (j < valid) {
                    float r = v[j];
                    if (p.accumulate) r += cvt_in<OT>(*dst);
                    *dst = cvt_out<OT>(r);
                }
                dst += cs;
            }
        }
    }
}

// Sum over the 32 lanes of a warp of 16 values per lane in 16 shuffles (butterfly that halves the values per lane at every step):
// returns, in every lane, the total of value index (lane >> 1).
__device__ __forceinline__ float warp_sum16(const float (&a)[16], int lane) {
    const bool h4 = lane & 16, h3 = lane & 8, h2 = lane & 4, h1 = lane & 2;
    float b[8], c[4], e[2];
    #pragma unroll
    for (int i = 0; i < 8; i++) b[i] = (h4 ? a[i + 8] : a[i]) + __shfl_xor_sync(0xffffffffu, h4 ? a[i] : a[i + 8], 16);
    #pragma unroll
    for (int i = 0; i < 4; i++) c[i] = (h3 ? b[i + 4] : b[i]) + __shfl_xor_sync(0xffffffffu, h3 ? b[i] : b[i + 4], 8);
    #pragma unroll
    for (int i = 0; i < 2; i++) e[i] = (h2 ? c[i + 2] : c[i]) + __shfl_xor_sync(0xffffffffu, h2 ? c[i] : c[i + 2], 4);
    float r = (h1 ? e[1] : e[0]) + __shfl_xor_sync(0xffffffffu, h1 ? e[0] : e[1], 2);
    r += __shfl_xor_sync(0xffffffffu, r, 1);
    return r;
}

// Fast epilogue: one sample per tile, per-column (scale, shift) staged in shared memory with the gain already folded in
// (linear / relu / lrelu are positively homogeneous).
template <int A, class OT, bool CLAMP, bool ACC>
__device__ __forceinline__ void epilogue_fast(const IgemmParams& p, const TileCoord tc, uint32_t tmem_tile, const PixelCoord pc,
                                              int col_begin, int col_end, const float2* s_cs, float nz_pre, float* stats_row) {
    const int x = tc.x0 + pc.px, y = tc.y0 + pc.py, n = tc.n0;
    const bool pix_ok = x < p.conv_w && y < p.conv_h;
    OT* const out = (OT*)p.out;
    const float alpha = p.alpha, clamp = p.clamp, gain = p.gain;
    const unsigned cs = (unsigned)p.os_c;
    const bool nhwc = p.os_c == 1;
    const int nchunks = (p.dbg & 2) ? 0 : (col_end - col_begin) >> 4;
    // 256-bit stores need 32-byte aligned pixels and parts
    const bool v8_ok = IsBf16<OT>::value && !(p.dbg & 32) && ((uintptr_t)out & 31) == 0 && p.os_w % 16 == 0 && p.os_h % 16 == 0 && p.os_n % 16 == 0 &&
                       p.out_part_stride % 16 == 0;
    auto process = [&](const uint32_t (&acc)[16], int c0) {
        const int g0 = tc.col0 + c0;
        const int phase = (g0 >= p.phase_stride) + (g0 >= 2 * p.phase_stride) + (g0 >= 3 * p.phase_stride);
        const int oc0 = g0 - phase * p.phase_stride;
        if (!pix_ok || oc0 >= p.o || phase >= p.phases || (p.dbg & 1)) return;
        const int oy = y * p.up + (phase >> 1), ox = x * p.up + (phase & 1);
        // up = 1: the pixel's noise value was fetched before the accumulator wait (nz_pre); up = 2: it depends on the phase
        float nz = nz_pre;
        if (p.noise && p.phases != 1) nz = __ldg(p.noise + n * p.noise_stride_n + (long long)oy * p.out_w + ox) * gain;
        const long long base = (p.dbg & 16) ? pc.py * p.os_h + pc.px * p.os_w : n * p.os_n + oy * p.os_h + ox * p.os_w;
        const int valid = min(16, p.o - oc0);
        // out += result (ToRGB adding into the up-sampled skip image, the residual add of the SPADE block): all 16 loads
        // of the read-modify-write are issued before the arithmetic so that one memory round trip covers the chunk
        float prev[ACC ? 16 : 1];
        if (ACC) {
            const OT* src = out + base + (long long)oc0 * p.os_c;
            #pragma unroll
            for (int j = 0; j < 16; j++) prev[j] = j < valid ? cvt_in<OT>(src[(unsigned)j * cs]) : 0.f;
        }
        float v[16];
        const float4* s_cs4 = reinterpret_cast<const float4*>(s_cs + c0);      // (scale, shift) of two columns per 128-bit load
        #pragma unroll
        for (int j = 0; j < 16; j += 2) {
            const float4 q = s_cs4[j >> 1];
            float r0 = fmaf(__uint_as_float(acc[j]), q.x, nz) + q.y;
            float r1 = fmaf(__uint_as_float(acc[j + 1]), q.z, nz) + q.w;
            if (A == PGPP_ACT_RELU) { r0 = fmaxf(r0, 0.f); r1 = fmaxf(r1, 0.f); }
            if (A == PGPP_ACT_LRELU) { r0 = fmaxf(r0, r0 * alpha); r1 = fmaxf(r1, r1 * alpha); }    // 0 <= alpha <= 1 (checked on the host)
            if (CLAMP) { r0 = fminf(fmaxf(r0, -clamp), clamp); r1 = fminf(fmaxf(r1, -clamp), clamp); }
            v[j] = r0; v[j + 1] = r1;
        }
        if (p.dbg & 8) {
            float sum = 0.f;
            #pragma unroll
            for (int j = 0; j < 16; j++) sum += v[j];
            if (sum != 1.2345e38f) return;
        }
        if (!ACC && stats_row) {
            // instance-norm partials of this warp's 32 pixels (host guarantees full tiles, o % 16 == 0: the whole warp is here):
            // pivot = lane 0's value, so a locally constant channel leaves exactly zero deviations
            const int lane = threadIdx.x & 31;
            float pv[16], d1[16], d2[16];
            #pragma unroll
            for (int j = 0; j < 16; j++) {
                pv[j] = __shfl_sync(0xffffffffu, v[j], 0);
                d1[j] = v[j] - pv[j];
                d2[j] = d1[j] * d1[j];
            }
            const float s1 = warp_sum16(d1, lane), s2 = warp_sum16(d2, lane);
            float* row = stats_row + oc0;
            if (lane == 0) {
                #pragma unroll
                for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(row + j) = make_float4(pv[j], pv[j + 1], pv[j + 2], pv[j + 3]);
            }
            if (!(lane & 1)) {
                row[p.stats_plane + (lane >> 1)] = s1;
                row[2 * p.stats_plane + (lane >> 1)] = s2;
            }
        }
        if (ACC) {
            // lanes are consecutive pixels: coalesced along W for NCHW tensors
            OT* dst = out + base + (long long)oc0 * p.os_c;
            #pragma unroll
            for (int j = 0; j < 16; j++)
                if (j < valid) dst[(unsigned)j * cs] = cvt_out<OT>(v[j] + prev[j]);
        } else if (nhwc && valid == 16 && ((base + oc0) * sizeof(OT)) % 16 == 0 && ((uintptr_t)out & 15) == 0) {
            // channels-innermost output: 16 consecutive channels of one pixel, 128-bit stores; with out_parts > 1 the
            // bf16 expansion of the value is written (part q = bf16(v - earlier parts)): the next conv's operand format
            if (IsBf16<OT>::value) {
                // packed conversions (two values per cvt.rn.bf16x2.f32); the residual is formed only if another part follows
                for (int part = 0; part < p.out_parts; part++) {
                    const bool more = part + 1 < p.out_parts;
                    uint32_t w[8];
                    #pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
                        w[j] = *reinterpret_cast<const uint32_t*>(&h);
                        if (more) {
                            v[2 * j] -= __uint_as_float(w[j] << 16);
                            v[2 * j + 1] -= __uint_as_float(w[j] & 0xffff0000u);
                        }
                    }
                    OT* const dptr = out + part * p.out_part_stride + base + oc0;
                    if (v8_ok) {
                        // one 256-bit store: the lane's 16 channels are one full 32-byte sector
                        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dptr), "r"(w[0]), "r"(w[1]), "r"(w[2]),
                                     "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
                    } else {
                        int4* dst = reinterpret_cast<int4*>(dptr);
                        dst[0] = make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]);
                        dst[1] = make_int4((int)w[4], (int)w[5], (int)w[6], (int)w[7]);
                    }
                }
            } else
            for (int part = 0; part < p.out_parts; part++) {
                __align__(16) OT tmp[16];
                #pragma unroll
                for (int j = 0; j < 16; j++) { tmp[j] = cvt_out<OT>(v[j]); v[j] -= cvt_in<OT>(tmp[j]); }
                int4* dst = reinterpret_cast<int4*>(out + part * p.out_part_stride + base + oc0);
                const int4* src = reinterpret_cast<const int4*>(tmp);
                #pragma unroll
                for (int q = 0; q < (int)(16 * sizeof(OT) / 16); q++) dst[q] = src[q];
            }
        } else {
            OT* dst = out + base + (long long)oc0 * p.os_c;
            if (valid == 16) {
                #pragma unroll
                for (int j = 0; j < 16; j++) dst[(unsigned)j * cs] = cvt_out<OT>(v[j]);
            } else {
                #pragma unroll
                for (int j = 0; j < 16; j++) if (j < valid) dst[(unsigned)j * cs] = cvt_out<OT>(v[j]);
            }
        }
    };
    // two chunks of TMEM loads are kept in flight (one round trip per 32 columns); the second epilogue warp on the same scheduler
    // covers the rest of the latency
    int ch = 0;
    if (!p.stack) {
        for (; ch + 1 < nchunks; ch += 2) {
            const int c0 = col_begin + ch * 16;
            uint32_t ra[16], rb[16];
            tmem_ld16_issue(tmem_tile + c0, ra);
            tmem_ld16_issue(tmem_tile + c0 + 16, rb);
            tmem_ld_wait16(ra);
            tmem_ld_wait16(rb);
            process(ra, c0);
            process(rb, c0 + 16);
        }
    }
    for (; ch < nchunks; ch++) {
        const int c0 = col_begin + ch * 16;
        uint32_t ra[16];
        tmem_ld16_issue(tmem_tile + c0, ra);
        if (p.stack) {
            // stacked split-precision products: columns [block_n, 2 * block_n) hold a0 x b1, to be added to a0 x b0 + a1 x b0
            uint32_t rb[16];
            tmem_ld16_issue(tmem_tile + p.block_n + c0, rb);
            tmem_ld_wait16(ra);
            tmem_ld_wait16(rb);
            #pragma unroll
            for (int j = 0; j < 16; j++) ra[j] = __float_as_uint(__uint_as_float(ra[j]) + __uint_as_float(rb[j]));
        } else {
            tmem_ld_wait16(ra);
        }
        process(ra, c0);
    }
}

// SPADE epilogue (networks.py:1702-1723 fused into the gamma|beta GEMM): the accumulator tile holds gamma in columns [0, C)
// and beta in columns [C, 2C) of one pixel row per lane; the lane reads x[n, c, y, x] (float32 NCHW, coalesced across the
// lanes of a warp), applies the instance normalisation with the staged per-(sample, channel) statistics,
//   v = (x - mean) * rstd * (1 + gamma) + beta,   then the consumer's pre-activation relu(v) * pre_gain,
// and writes the bf16 expansion of v channels-innermost: the operand format of the next convolution.
// s_cs[c] = (rstd[n, c], bias_gamma[c]), s_cs[C + c] = (mean[n, c], bias_beta[c]).
// F8: e4m3 operands - gamma / beta are the accumulators times the weight column scales; the output is e4m3 when out_dtype says so.
template <bool F8>
__device__ __forceinline__ void epilogue_spade(const IgemmParams& p, const TileCoord tc, uint32_t tmem_tile, const PixelCoord pc,
                                               int half, const float2* s_cs) {
    const int C = p.o >> 1;
    const int chunks = C >> 4;
    const int ch_begin = (half * chunks) >> 1, ch_end = ((half + 1) * chunks) >> 1;
    const int x = tc.x0 + pc.px, y = tc.y0 + pc.py, n = tc.n0;
    const bool pix_ok = x < p.conv_w && y < p.conv_h;
    const long long plane = (long long)p.conv_h * p.conv_w;
    const float* xin = p.spade_x + (long long)n * C * plane + (long long)y * p.conv_w + x;
    __nv_bfloat16* const out = (__nv_bfloat16*)p.out + n * p.os_n + y * p.os_h + x * p.os_w;
    const float pre_gain = p.spade_pre_gain;
    for (int ch = ch_begin; ch < ch_end; ch++) {
        const int c0 = ch << 4;
        float xv[16];
        #pragma unroll
        for (int j = 0; j < 16; j++) xv[j] = pix_ok ? __ldg(xin + (long long)(c0 + j) * plane) : 0.f;
        uint32_t rg[16], rb[16];
        tmem_ld16_issue(tmem_tile + c0, rg);
        tmem_ld16_issue(tmem_tile + C + c0, rb);
        tmem_ld_wait16(rg);
        tmem_ld_wait16(rb);
        if (!pix_ok) continue;
        float v[16];
        #pragma unroll
        for (int j = 0; j < 16; j++) {
            const float2 qg = s_cs[c0 + j], qb = s_cs[C + c0 + j];
            float ag = __uint_as_float(rg[j]), ab = __uint_as_float(rb[j]);
            if (F8) { ag *= weight_scale(p, n, c0 + j); ab *= weight_scale(p, n, C + c0 + j); }
            const float g = ag + qg.y, b = ab + qb.y;
            float r = fmaf((xv[j] - qb.x) * qg.x, 1.f + g, b);
            if (pre_gain > 0.f) r = fmaxf(r, 0.f) * pre_gain;
            v[j] = r;
        }
        if (F8 && p.out_dtype == PGPP_E4M3) {
            uint8_t* const dst8 = (uint8_t*)p.out + n * p.os_n + y * p.os_h + x * p.os_w + c0;
            *reinterpret_cast<uint4*>(dst8) = make_uint4(e4m3x4(v[0], v[1], v[2], v[3]), e4m3x4(v[4], v[5], v[6], v[7]),
                                                         e4m3x4(v[8], v[9], v[10], v[11]), e4m3x4(v[12], v[13], v[14], v[15]));
            continue;
        }
        for (int part = 0; part < p.out_parts; part++) {
            __align__(16) __nv_bfloat16 tmp[16];
            #pragma unroll
            for (int j = 0; j < 16; j++) { tmp[j] = __float2bfloat16_rn(v[j]); v[j] -= __bfloat162float(tmp[j]); }
            int4* dst = reinterpret_cast<int4*>(out + part * p.out_part_stride + c0);
            const int4* src = reinterpret_cast<const int4*>(tmp);
            dst[0] = src[0];
            dst[1] = src[1];
        }
    }
}

template <class OT, bool F8>
__device__ __forceinline__ void epilogue_dispatch(const IgemmParams& p, const TileCoord tc, uint32_t tmem_tile, const PixelCoord pc,
                                                  int col_begin, int col_end, const float2* s_cs, bool fast, float nz_pre, float* stats_row) {
    if (fast) {
        // ACC: read-modify-write output (ToRGB into the skip image, residual adds)
#define PGPP_FAST(ACT) \
        if (p.accumulate) { if (cl) epilogue_fast<ACT, OT, true, true>(p, tc, tmem_tile, pc, col_begin, col_end, s_cs, nz_pre, stats_row);   \
                            else    epilogue_fast<ACT, OT, false, true>(p, tc, tmem_tile, pc, col_begin, col_end, s_cs, nz_pre, stats_row); } \
        else               { if (cl) epilogue_fast<ACT, OT, true, false>(p, tc, tmem_tile, pc, col_begin, col_end, s_cs, nz_pre, stats_row);  \
                            else    epilogue_fast<ACT, OT, false, false>(p, tc, tmem_tile, pc, col_begin, col_end, s_cs, nz_pre, stats_row); }
        const bool cl = p.clamp >= 0.f;
        switch (p.act_fn) {
            case PGPP_ACT_LINEAR: PGPP_FAST(PGPP_ACT_LINEAR) break;
            case PGPP_ACT_RELU:   PGPP_FAST(PGPP_ACT_RELU) break;
            default:              PGPP_FAST(PGPP_ACT_LRELU) break;
        }
#undef PGPP_FAST
        return;
    }
#define PGPP_EPI(ACT) epilogue_general<ACT, OT, F8>(p, tc, tmem_tile, pc, col_begin, col_end)
    switch (p.act_fn) {
        case PGPP_ACT_LINEAR: PGPP_EPI(PGPP_ACT_LINEAR); break;
        case PGPP_ACT_RELU: PGPP_EPI(PGPP_ACT_RELU); break;
        case PGPP_ACT_LRELU: PGPP_EPI(PGPP_ACT_LRELU); break;
        case PGPP_ACT_TANH: PGPP_EPI(PGPP_ACT_TANH); break;
        case PGPP_ACT_SIGMOID: PGPP_EPI(PGPP_ACT_SIGMOID); break;
        case PGPP_ACT_ELU: PGPP_EPI(PGPP_ACT_ELU); break;
        case PGPP_ACT_SELU: PGPP_EPI(PGPP_ACT_SELU); break;
        case PGPP_ACT_SOFTPLUS: PGPP_EPI(PGPP_ACT_SOFTPLUS); break;
        default: PGPP_EPI(PGPP_ACT_SWISH); break;
    }
#undef PGPP_EPI
}

// Lean epilogue for the operand-format hand-over, the configuration almost every large layer of the generator runs in: one sample
// per tile, gain folded into the staged (scale, shift), bf16 channels-innermost output in 1..3 parts (the next conv's TMA operand),
// phases == 1, no accumulate, linear / relu / lrelu.  Against the general path: everything tile-invariant is hoisted out of the tile
// loop, the pixel's noise value of the NEXT tile is fetched before this tile's accumulator wait (its latency was the largest single
// stall of the general epilogue), 32 columns per TMEM load, one 256-bit store per (16 channels, part).
// STK: columns [block_n, 2 * block_n) of the accumulator hold a0 x b1 and are added to a0 x b0 + a1 x b0 (see mma_role).
// ACC: out += result on the operand format (the residual adds y = skip + conv1(...) of ResBlock / Spade_ResBlockV4_512 without
// leaving the format): the parts already stored are summed, the result added and the bf16 expansion written back.
// F8: e4m3 operands (the column scale of the weights joins the staged scale) and e4m3 output, one part, one 128-bit store per 16 channels.
template <int A, bool STK, bool ACC, bool F8 = false>
__device__ __forceinline__ void epilogue_packed_role(const IgemmParams& p, uint32_t bar_base, uint32_t tmem_base, float2* s_params,
                                                     int warp, int lane) {
    const uint32_t tfull0 = bar_base + 8u * (2 * p.a_stages + 2 * p.b_stages), tempty0 = tfull0 + 16u;
    const int quarter = warp & 3, half = (warp - 2) >> 2;
    const int lane_row = quarter * 32 + lane;
    const int px = lane_row % p.tw, py = lane_row / p.tw;        // tn == 1
    const int etid = threadIdx.x - 64;
    const int block_n = p.block_n, cols_per = block_n >> 1, col_begin = half * cols_per;
    const float alpha = p.alpha, gain = p.gain;
    const float cl = p.clamp >= 0.f ? p.clamp : __int_as_float(0x7f800000);      // no clamp: +-inf bounds
    typedef typename std::conditional<F8, uint8_t, __nv_bfloat16>::type ET;
    ET* const out = (ET*)p.out;
    const long long part_stride = p.out_part_stride;
    const int nparts = p.out_parts;
    const float* const noise = p.noise;
    const int conv_w = p.conv_w, conv_h = p.conv_h;
    const long long total = p.total_tiles;
    auto noise_at = [&](const TileCoord& c) -> float {
        const int x = c.x0 + px, y = c.y0 + py;
        return (noise && x < conv_w && y < conv_h) ? __ldg(noise + c.n0 * p.noise_stride_n + (long long)y * p.out_w + x) : 0.f;
    };
    // one 16-column chunk: scale / noise / shift / activation / clamp, bf16 expansion, 256-bit stores
    auto chunk = [&](const uint32_t* acc, const float2* s_cs, float nz, ET* dst, bool store) {
        float v[16];
        const float4* s_cs4 = reinterpret_cast<const float4*>(s_cs);
        #pragma unroll
        for (int j = 0; j < 16; j += 2) {
            const float4 q = s_cs4[j >> 1];
            float r0 = fmaf(__uint_as_float(acc[j]), q.x, nz) + q.y;
            float r1 = fmaf(__uint_as_float(acc[j + 1]), q.z, nz) + q.w;
            if (A == PGPP_ACT_RELU) { r0 = fmaxf(r0, 0.f); r1 = fmaxf(r1, 0.f); }
            if (A == PGPP_ACT_LRELU) { r0 = fmaxf(r0, r0 * alpha); r1 = fmaxf(r1, r1 * alpha); }
            v[j] = fminf(fmaxf(r0, -cl), cl); v[j + 1] = fminf(fmaxf(r1, -cl), cl);
        }
        if (p.dbg & 8) {
            float sum = 0.f;
            #pragma unroll
            for (int j = 0; j < 16; j++) sum += v[j];
            store = store && sum == 1.2345e38f;
        }
        if (!store) return;
        if constexpr (F8) {
            if (ACC) {
                uint32_t prev[4];
                asm volatile("ld.global.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(prev[0]), "=r"(prev[1]), "=r"(prev[2]), "=r"(prev[3]) : "l"(dst) : "memory");
                #pragma unroll
                for (int j = 0; j < 8; j++) {
                    const float2 f = e4m3x2_to_float2(prev[j >> 1] >> (16 * (j & 1)));
                    v[2 * j] += f.x; v[2 * j + 1] += f.y;
                }
            }
            uint32_t w[4];
            #pragma unroll
            for (int j = 0; j < 4; j++) w[j] = e4m3x4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
            return;
        }
        if (ACC) {
            uint32_t prev[3][8];
            #pragma unroll
            for (int part = 0; part < 3; part++)
                if (part < nparts)
                asm volatile("ld.global.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];" : "=r"(prev[part][0]), "=r"(prev[part][1]), "=r"(prev[part][2]),
                             "=r"(prev[part][3]), "=r"(prev[part][4]), "=r"(prev[part][5]), "=r"(prev[part][6]), "=r"(prev[part][7])
                             : "l"(dst + part * part_stride) : "memory");
            #pragma unroll
            for (int part = 2; part >= 0; part--) {                 // smallest part first
                if (part >= nparts) continue;
                #pragma unroll
                for (int j = 0; j < 8; j++) {
                    v[2 * j] += __uint_as_float(prev[part][j] << 16);
                    v[2 * j + 1] += __uint_as_float(prev[part][j] & 0xffff0000u);
                }
            }
        }
        for (int part = 0; part < nparts; part++) {
            const bool more = part + 1 < nparts;
            uint32_t w[8];
            #pragma unroll
            for (int j = 0; j < 8; j++) {
                const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
                w[j] = *reinterpret_cast<const uint32_t*>(&h);
                if (more) {
                    v[2 * j] -= __uint_as_float(w[j] << 16);
                    v[2 * j + 1] -= __uint_as_float(w[j] & 0xffff0000u);
                }
            }
            asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + part * part_stride), "r"(w[0]), "r"(w[1]),
                         "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
        }
    };
    int buf = 0; uint32_t buf_phase = 0;
    int tag0 = -1, tag1 = -1;
    long long t = blockIdx.x;
    TileCoord tc = decode_tile(p, t);
    float nz_raw = noise_at(tc);
    while (t < total) {
        float2* const s_buf = s_params + buf * block_n;
        const int tag = tc.n0 * p.tiles_col + tc.col0 / block_n;
        if ((buf ? tag1 : tag0) != tag) {
            asm volatile("bar.sync 1, 256;" ::: "memory");      // every epilogue warp is done with the tile that last used this buffer
            if (etid < block_n) {
                const int oc = tc.col0 + etid;
                float sc = 1.f, sh = 0.f;
                if (oc < p.o) {
                    if (p.dcoef) sc = __ldg(p.dcoef + (long long)tc.n0 * p.o + oc);
                    if (F8) sc *= weight_scale(p, tc.n0, oc);
                    if (p.bias) sh = __ldg(p.bias + oc);
                }
                s_buf[etid] = make_float2(sc * gain, sh * gain);
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (buf) tag1 = tag; else tag0 = tag;
        }
        // next tile: coordinates and noise value, fetched while this tile's MMAs may still be running
        const long long t_next = t + gridDim.x;
        TileCoord tc_next = tc;
        float nz_next = 0.f;
        if (t_next < total) { tc_next = decode_tile(p, t_next); nz_next = noise_at(tc_next); }
        const int x = tc.x0 + px, y = tc.y0 + py;
        const bool pix_ok = x < conv_w && y < conv_h && !(p.dbg & 1);
        ET* const dst = out + tc.n0 * p.os_n + y * p.os_h + x * p.os_w + tc.col0 + col_begin;
        const float2* const s_cs = s_buf + col_begin;
        const int o_left = p.o - (tc.col0 + col_begin);                 // valid columns counted from this warp's first column
        const float nz = nz_raw * gain;
        mbar_wait(tfull0 + 8u * buf, buf_phase);
        tc_fence_after();
        const uint32_t tmem_tile = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * p.acc_cols + col_begin);
        if (!(p.dbg & 2)) {
            if (cols_per >= 32) {
                for (int c0 = 0; c0 < cols_per; c0 += 32) {
                    uint32_t ra[32];
                    tmem_ld32_issue(tmem_tile + c0, ra);
                    if (STK) {
                        uint32_t rb[32];
                        tmem_ld32_issue(tmem_tile + block_n + c0, rb);
                        tmem_ld_wait32(ra);
                        tmem_ld_wait32(rb);
                        #pragma unroll
                        for (int j = 0; j < 32; j++) ra[j] = __float_as_uint(__uint_as_float(ra[j]) + __uint_as_float(rb[j]));
                    } else {
                        tmem_ld_wait32(ra);
                    }
                    chunk(ra, s_cs + c0, nz, dst + c0, pix_ok && c0 + 16 <= o_left);
                    chunk(ra + 16, s_cs + c0 + 16, nz, dst + c0 + 16, pix_ok && c0 + 32 <= o_left);
                }
            } else {
                uint32_t ra[16];
                tmem_ld16_issue(tmem_tile, ra);
                tmem_ld_wait16(ra);
                chunk(ra, s_cs, nz, dst, pix_ok && 16 <= o_left);
            }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty0 + 8u * buf);
        if (++buf == 2) { buf = 0; buf_phase ^= 1; }
        t = t_next; tc = tc_next; nz_raw = nz_next;
    }
}

struct MmaCtx { uint32_t smem_base, b_base, bar_base, tmem_base; };

// MMA issuer role (warp 1).  The whole warp walks the warp-uniform loop so that descriptors live in uniform registers;
// one elected lane issues tcgen05.mma / tcgen05.commit.  PARTS / INNER / KS > 0 are compile-time copies of p.parts /
// p.inner / (kb / 16) for the common configurations (fully unrolled product / tap / K-step loops, a handful of
// instructions per MMA); <0, 0, 0> is the generic runtime-bounds version.
template <bool F8, int PARTS, int INNER, int KS, bool RES, bool STK = false>
__device__ __forceinline__ void mma_role(const IgemmParams& p, const MmaCtx mc) {
    const int SA = p.a_stages, SB = p.b_stages;
    auto afull_bar = [&](int s) { return mc.bar_base + 8u * s; };
    auto aempty_bar = [&](int s) { return mc.bar_base + 8u * (SA + s); };
    auto bfull_bar = [&](int s) { return mc.bar_base + 8u * (2 * SA + s); };
    auto bempty_bar = [&](int s) { return mc.bar_base + 8u * (2 * SA + SB + s); };
    auto tfull_bar = [&](int b) { return mc.bar_base + 8u * (2 * SA + 2 * SB + b); };
    auto tempty_bar = [&](int b) { return mc.bar_base + 8u * (2 * SA + 2 * SB + 2 + b); };
    const uint32_t bres_free_bar = mc.bar_base + 8u * (2 * SA + 2 * SB + 4);
    const int parts = PARTS ? PARTS : p.parts;
    const int inner = INNER ? INNER : p.inner;
    const int k_steps = KS ? KS : (F8 ? p.kb / 32 : p.kb / 16);     // K per tcgen05.mma: 16 (kind::f16), 32 (kind::f8f6f4) = 32 bytes
    const bool leader = elect_one();
    const bool mma_on = !(p.dbg & 4);
    const uint64_t desc_hi = make_smem_desc(0, p.layout_type, p.sbo_bytes);     // everything but the start address
    const uint32_t slab16 = p.slab_bytes >> 4, ky16 = p.ky_step_bytes >> 4, bpitch16 = p.b_pitch >> 4;
    const uint32_t idesc = p.idesc;
    int sa = 0; uint32_t pha = 0;
    int sb = 0; uint32_t phb = 0;
    int buf = 0; uint32_t buf_phase = 0;
    bool first_tile = true;
    int last_n = -1; uint32_t res_phase = 0;
    for (long long t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
        // resident weights: wait for the (re)load on the first tile and whenever the sample changed (per-sample weights)
        if (RES) {
            const int n0 = p.wgt_per_sample ? decode_tile(p, t).n0 : 0;
            if (first_tile || n0 != last_n) {
                if (!first_tile) res_phase ^= 1;
                for (int sl = 0; sl < SB; sl++) mbar_wait(bfull_bar(sl), res_phase);    // all resident weight tiles have landed
            }
            last_n = n0;
        }
        mbar_wait(tempty_bar(buf), buf_phase ^ 1);      // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = mc.tmem_base + (uint32_t)(buf * p.acc_cols);
        uint32_t acc = 0;
        uint32_t b_res16 = mc.b_base >> 4;              // resident weights: next tile in consumption order
        for (int g = 0; g < p.n_groups; g++) {
            for (int cb = 0; cb < p.num_cb; cb++) {
                mbar_wait(afull_bar(sa), pha);
                tc_fence_after();
                const uint32_t a16 = (mc.smem_base + sa * p.a_stage_bytes) >> 4;
                #pragma unroll
                for (int j = 0; j < (INNER ? INNER : 8); j++) {
                    if (j >= inner) break;
                    if (STK) {
                        // parts = 2, resident weights, block_n = 64: the tiles of b0 and b1 of a tap are adjacent in shared memory, so
                        // a0 x [b0; b1] is ONE MMA with N = 128 (a0 x b0 in columns [0, 64), a0 x b1 in [64, 128), summed by the
                        // epilogue) and a1 x b0 a second one with N = 64: two reads of the A tile per K step instead of three
                        const uint32_t b16 = b_res16;
                        b_res16 += 2 * bpitch16;
                        const uint64_t db = desc_hi | (uint64_t)(b16 & 0x3FFF);
                        const uint64_t da0 = desc_hi | (uint64_t)((a16 + j * ky16) & 0x3FFF);
                        const uint64_t da1 = desc_hi | (uint64_t)((a16 + slab16 + j * ky16) & 0x3FFF);
                        if (leader && mma_on) {
                            umma<F8>(tmem_d, da0, db, p.idesc_stack, acc);
                            umma<F8>(tmem_d, da0 + 2, db + 2, p.idesc_stack, 1);
                            umma<F8>(tmem_d, da0 + 4, db + 4, p.idesc_stack, 1);
                            umma<F8>(tmem_d, da0 + 6, db + 6, p.idesc_stack, 1);
                            umma<F8>(tmem_d, da1, db, idesc, 1);
                            umma<F8>(tmem_d, da1 + 2, db + 2, idesc, 1);
                            umma<F8>(tmem_d, da1 + 4, db + 4, idesc, 1);
                            umma<F8>(tmem_d, da1 + 6, db + 6, idesc, 1);
                        }
                        acc = 1;
                    }
                    if (!STK)
                    #pragma unroll
                    for (int pb = 0; pb < (PARTS ? PARTS : 3); pb++) {
                        if (pb >= parts) break;
                        uint32_t b16;
                        if (RES) {
                            b16 = b_res16;
                            b_res16 += bpitch16;
                        } else {
                            mbar_wait(bfull_bar(sb), phb);
                            tc_fence_after();
                            b16 = (mc.b_base + sb * p.b_pitch) >> 4;
                        }
                        const uint64_t db = desc_hi | (uint64_t)(b16 & 0x3FFF);
                        #pragma unroll
                        for (int pa = 0; pa < (PARTS ? PARTS : 3); pa++) {
                            if (pa + pb >= parts) break;                    // products a_pa * b_pb with pa + pb < parts
                            const uint64_t da = desc_hi | (uint64_t)((a16 + pa * slab16 + j * ky16) & 0x3FFF);
                            if (leader && mma_on) {
                                if (KS == 4) {
                                    // advance 16 elements (32 bytes) along K inside the swizzle row: +2 in the >>4 address field
                                    umma<F8>(tmem_d, da, db, idesc, acc);
                                    umma<F8>(tmem_d, da + 2, db + 2, idesc, 1);
                                    umma<F8>(tmem_d, da + 4, db + 4, idesc, 1);
                                    umma<F8>(tmem_d, da + 6, db + 6, idesc, 1);
                                } else {
                                    for (int k = 0; k < k_steps; k++)
                                        umma<F8>(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, acc | (uint32_t)k);
                                }
                            }
                            acc = 1;
                        }
                        if (!RES) {
                            if (leader) umma_commit(bempty_bar(sb));        // weight slot reusable once these MMAs retire
                            if (++sb == SB) { sb = 0; phb ^= 1; }
                        }
                    }
                }
                if (leader) umma_commit(aempty_bar(sa));                    // activation slab reusable
                if (++sa == SA) { sa = 0; pha ^= 1; }
            }
        }
        if (leader) umma_commit(tfull_bar(buf));                            // accumulator complete -> epilogue
        if (RES && p.wgt_per_sample) {
            // last tile of this sample on this CTA: once its MMAs retire the producer may overwrite the resident weights
            const long long tn = t + gridDim.x;
            if (tn < p.total_tiles && decode_tile(p, tn).n0 != last_n && leader) umma_commit(bres_free_bar);
        }
        if (++buf == 2) { buf = 0; buf_phase ^= 1; }
        first_tile = false;
    }
    __syncwarp();
}

// MMA issuer for the single-slab mode (p.reuse == 2): the activation ring holds one (channel block, part) slab per stage, the
// weights are resident, and tap j of the filter reads the slab through a descriptor whose start is shifted by whole pixel rows
// (tap_off16) with an 8-row group stride of one slab row (sbo_a) - the tensor core applies the 128-byte swizzle on the absolute
// shared-memory address, so such views are exact (tools/umma_probe.cu).  Product order: for every part a_pa of the slab, all taps,
// all weight parts b_pb with pa + pb < parts.  STK: parts == 2 and block_n == 64 -> a0 x [b0; b1] is one N = 128 MMA.
template <bool F8, int PARTS, int TAPS, bool STK>
__device__ __forceinline__ void mma_role_slab(const IgemmParams& p, const MmaCtx mc) {
    const int SA = p.a_stages, SB = p.b_stages;
    auto afull_bar = [&](int s) { return mc.bar_base + 8u * s; };
    auto aempty_bar = [&](int s) { return mc.bar_base + 8u * (SA + s); };
    auto bfull_bar = [&](int s) { return mc.bar_base + 8u * (2 * SA + s); };
    auto tfull_bar = [&](int b) { return mc.bar_base + 8u * (2 * SA + 2 * SB + b); };
    auto tempty_bar = [&](int b) { return mc.bar_base + 8u * (2 * SA + 2 * SB + 2 + b); };
    const uint32_t bres_free_bar = mc.bar_base + 8u * (2 * SA + 2 * SB + 4);
    const int parts = PARTS ? PARTS : p.parts;
    const int taps = TAPS ? TAPS : p.inner;
    const bool leader = elect_one();
    const bool mma_on = !(p.dbg & 4);
    const uint64_t desc_a_hi = make_smem_desc(0, p.layout_type, p.sbo_a);
    const uint64_t desc_b_hi = make_smem_desc(0, p.layout_type, p.sbo_bytes);
    const uint32_t bpitch16 = p.b_pitch >> 4;
    const uint32_t idesc = p.idesc;
    int sa = 0; uint32_t pha = 0;
    int buf = 0; uint32_t buf_phase = 0;
    bool first_tile = true;
    int last_n = -1; uint32_t res_phase = 0;
    for (long long t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
        const int n0 = p.wgt_per_sample ? decode_tile(p, t).n0 : 0;
        if (first_tile || n0 != last_n) {
            if (!first_tile) res_phase ^= 1;
            for (int sl = 0; sl < SB; sl++) mbar_wait(bfull_bar(sl), res_phase);
        }
        last_n = n0;
        mbar_wait(tempty_bar(buf), buf_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = mc.tmem_base + (uint32_t)(buf * p.acc_cols);
        uint32_t acc = 0;
        for (int cb = 0; cb < p.num_cb; cb++) {
            #pragma unroll
            for (int pa = 0; pa < (PARTS ? PARTS : 3); pa++) {
                if (pa >= parts) break;
                if (!(p.dbg & 64)) mbar_wait(afull_bar(sa), pha);
                tc_fence_after();
                const uint32_t a16 = (mc.smem_base + sa * p.a_stage_bytes) >> 4;
                const uint32_t b_cb16 = (mc.b_base >> 4) + (uint32_t)(cb * taps * parts) * bpitch16;
                #pragma unroll
                for (int j = 0; j < (TAPS ? TAPS : 64); j++) {
                    if (j >= taps) break;
                    const uint64_t da = desc_a_hi | (uint64_t)((a16 + p.tap_off16[j]) & 0x3FFF);
                    const uint32_t b_tap16 = b_cb16 + (uint32_t)(j * parts) * bpitch16;
                    if (STK) {
                        // pa == 0: a0 x [b0; b1] (N = 2 * block_n);  pa == 1: a1 x b0 (N = block_n)
                        const uint64_t db = desc_b_hi | (uint64_t)(b_tap16 & 0x3FFF);
                        const uint32_t id = pa == 0 ? p.idesc_stack : idesc;
                        if (leader && mma_on) {
                            umma<F8>(tmem_d, da, db, id, acc);
                            umma<F8>(tmem_d, da + 2, db + 2, id, 1);
                            umma<F8>(tmem_d, da + 4, db + 4, id, 1);
                            umma<F8>(tmem_d, da + 6, db + 6, id, 1);
                        }
                        acc = 1;
                    } else {
                        #pragma unroll
                        for (int pb = 0; pb < (PARTS ? PARTS : 3); pb++) {
                            if (pa + pb >= parts) break;
                            const uint64_t db = desc_b_hi | (uint64_t)((b_tap16 + pb * bpitch16) & 0x3FFF);
                            if (leader && mma_on) {
                                umma<F8>(tmem_d, da, db, idesc, acc);
                                umma<F8>(tmem_d, da + 2, db + 2, idesc, 1);
                                umma<F8>(tmem_d, da + 4, db + 4, idesc, 1);
                                umma<F8>(tmem_d, da + 6, db + 6, idesc, 1);
                            }
                            acc = 1;
                        }
                    }
                }
                if (leader) umma_commit(aempty_bar(sa));
                if (++sa == SA) { sa = 0; pha ^= 1; }
            }
        }
        if (leader) umma_commit(tfull_bar(buf));
        if (p.wgt_per_sample) {
            const long long tn = t + gridDim.x;
            if (tn < p.total_tiles && decode_tile(p, tn).n0 != last_n && leader) umma_commit(bres_free_bar);
        }
        if (++buf == 2) { buf = 0; buf_phase ^= 1; }
        first_tile = false;
    }
    __syncwarp();
}

// Experimental single-slab MMA issuer (PGPP_IGEMM_SLAB9=1) for 3 x 3 filters, 64-channel rows, 64-column resident weight tiles, 1 or 2 parts:
// every shared-memory descriptor of a tile differs from the stage's first one by a compile-time offset (tap (ky, kx) starts (ky * 10 + kx)
// 128-byte pixel rows into the slab, weight tile t starts t * 8 KB after the first, a K step is 32 bytes), so the elected lane issues the 36
// MMAs of a stage as straight-line code, ~4 instead of ~9 instructions per MMA.  Measured on 64->64 3x3 @512^2 n32 (profiles/
// r02_igemm64_issuer_ablation.md): with neither activation loads nor epilogue the fp32-parity tile loop runs in 1.23 ms against 1.40 ms for the
// generic issuer, but the complete kernel stays at 1.57 ms (bf16 mode: 0.83 vs 0.79 ms, uniform-register spills): the issuing warp is not what
// bounds these layers - the tensor pipe alone, fed from shared memory at N <= 128, already needs 1.23 ms.  Off by default.
template <bool F8, int PARTS, bool STK>
__device__ __forceinline__ void mma_role_slab9(const IgemmParams& p, const MmaCtx mc) {
    constexpr int TAPS = 9, PITCH = 10;
    constexpr uint32_t BP16 = 512;          // 64 rows x 128 bytes per weight tile, in 16-byte units
    const int SA = p.a_stages, SB = p.b_stages;
    auto afull_bar = [&](int s) { return mc.bar_base + 8u * s; };
    auto aempty_bar = [&](int s) { return mc.bar_base + 8u * (SA + s); };
    auto bfull_bar = [&](int s) { return mc.bar_base + 8u * (2 * SA + s); };
    auto tfull_bar = [&](int b) { return mc.bar_base + 8u * (2 * SA + 2 * SB + b); };
    auto tempty_bar = [&](int b) { return mc.bar_base + 8u * (2 * SA + 2 * SB + 2 + b); };
    const uint32_t bres_free_bar = mc.bar_base + 8u * (2 * SA + 2 * SB + 4);
    const bool leader = elect_one();
    const bool mma_on = !(p.dbg & 4), wait_a = !(p.dbg & 64);
    const uint64_t desc_a = make_smem_desc(0, p.layout_type, p.sbo_a), desc_b = make_smem_desc(0, p.layout_type, p.sbo_bytes);
    const uint32_t a_hi = (uint32_t)(desc_a >> 32), b_hi = (uint32_t)(desc_b >> 32), lo_flags = (uint32_t)desc_a;     // low word without the address
    const uint32_t idesc = p.idesc, idesc_stack = p.idesc_stack;
    const uint32_t a_stage16 = p.a_stage_bytes >> 4;
    int sa = 0; uint32_t pha = 0;
    int buf = 0; uint32_t buf_phase = 0;
    bool first_tile = true;
    int last_n = -1; uint32_t res_phase = 0;
    for (long long t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
        const int n0 = p.wgt_per_sample ? decode_tile(p, t).n0 : 0;
        if (first_tile || n0 != last_n) {
            if (!first_tile) res_phase ^= 1;
            for (int sl = 0; sl < SB; sl++) mbar_wait(bfull_bar(sl), res_phase);
        }
        last_n = n0;
        mbar_wait(tempty_bar(buf), buf_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = mc.tmem_base + (uint32_t)(buf * p.acc_cols);
        for (int cb = 0; cb < p.num_cb; cb++) {
            const uint32_t b_lo0 = lo_flags | (((mc.b_base >> 4) + (uint32_t)(cb * TAPS * PARTS) * BP16) & 0x3FFFu);
            #pragma unroll
            for (int pa = 0; pa < PARTS; pa++) {
                if (wait_a) mbar_wait(afull_bar(sa), pha);
                tc_fence_after();
                const uint32_t a_lo0 = lo_flags | (((mc.smem_base >> 4) + (uint32_t)sa * a_stage16) & 0x3FFFu);
                const uint32_t first = (cb == 0 && pa == 0) ? 0u : 1u;          // the first MMA of a tile overwrites the accumulator
                if (leader && mma_on) {
                    #pragma unroll
                    for (int j = 0; j < TAPS; j++) {
                        const uint32_t a_lo = a_lo0 + (uint32_t)(((j / 3) * PITCH + (j % 3)) * 8);
                        if (STK) {
                            // pa == 0: a0 x [b0; b1] (N = 128);  pa == 1: a1 x b0 (N = 64)
                            const uint32_t b_lo = b_lo0 + (uint32_t)(j * PARTS) * BP16;
                            const uint32_t id = pa == 0 ? idesc_stack : idesc;
                            umma_lh<F8>(tmem_d, a_lo, a_hi, b_lo, b_hi, id, j == 0 ? first : 1u);
                            umma_lh<F8>(tmem_d, a_lo + 2, a_hi, b_lo + 2, b_hi, id, 1u);
                            umma_lh<F8>(tmem_d, a_lo + 4, a_hi, b_lo + 4, b_hi, id, 1u);
                            umma_lh<F8>(tmem_d, a_lo + 6, a_hi, b_lo + 6, b_hi, id, 1u);
                        } else {
                            #pragma unroll
                            for (int pb = 0; pb < PARTS; pb++) {
                                if (pa + pb >= PARTS) break;
                                const uint32_t b_lo = b_lo0 + (uint32_t)(j * PARTS + pb) * BP16;
                                umma_lh<F8>(tmem_d, a_lo, a_hi, b_lo, b_hi, idesc, (j == 0 && pb == 0) ? first : 1u);
                                umma_lh<F8>(tmem_d, a_lo + 2, a_hi, b_lo + 2, b_hi, idesc, 1u);
                                umma_lh<F8>(tmem_d, a_lo + 4, a_hi, b_lo + 4, b_hi, idesc, 1u);
                                umma_lh<F8>(tmem_d, a_lo + 6, a_hi, b_lo + 6, b_hi, idesc, 1u);
                            }
                        }
                    }
                }
                if (leader) umma_commit(aempty_bar(sa));
                if (++sa == SA) { sa = 0; pha ^= 1; }
            }
        }
        if (leader) umma_commit(tfull_bar(buf));
        if (p.wgt_per_sample) {
            const long long tn = t + gridDim.x;
            if (tn < p.total_tiles && decode_tile(p, tn).n0 != last_n && leader) umma_commit(bres_free_bar);
        }
        if (++buf == 2) { buf = 0; buf_phase ^= 1; }
        first_tile = false;
    }
    __syncwarp();
}

// EPI 0: every epilogue option;  EPI 1: the lean operand-format epilogue only (epilogue_packed_role; smaller code and register footprint).
// F8: e4m3 operands (kind::f8f6f4; channel blocks of kb bytes = kb channels), weight column scales in the epilogue; EPI 1 writes e4m3.
template <int EPI, bool F8>
__global__ void __launch_bounds__(kThreads, 1)
igemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const IgemmParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // carve: [A ring: a_stages x parts slabs][B slots: b_stages x b_pitch] (1024-byte aligned), then barriers
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t b_base = smem_base + p.a_stages * p.a_stage_bytes;
    const uint32_t bar_base = b_base + p.b_stages * p.b_pitch;
    const int SA = p.a_stages, SB = p.b_stages;
    // barrier i at bar_base + 8*i
    auto afull_bar = [&](int s) { return bar_base + 8u * s; };
    auto aempty_bar = [&](int s) { return bar_base + 8u * (SA + s); };
    auto bfull_bar = [&](int s) { return bar_base + 8u * (2 * SA + s); };
    auto bempty_bar = [&](int s) { return bar_base + 8u * (2 * SA + SB + s); };
    auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * SA + 2 * SB + b); };
    auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * SA + 2 * SB + 2 + b); };
    const uint32_t bres_free_bar = bar_base + 8u * (2 * SA + 2 * SB + 4);     // resident weights may be overwritten (one completion per reload)
    const uint32_t tmem_slot = bar_base + 8u * (2 * SA + 2 * SB + 5);
    // per-column epilogue parameters (scale, shift), double-buffered with the accumulator: float2 [2][block_n]
    float2* const s_params = reinterpret_cast<float2*>(smem_raw + (((tmem_slot + 16u + 15u) & ~15u) - smem_u32(smem_raw)));   // 16-byte aligned: read as float4

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && elect_one()) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
        for (int s = 0; s < SA; s++) { mbar_init(afull_bar(s), 1); mbar_init(aempty_bar(s), 1); }
        for (int s = 0; s < SB; s++) { mbar_init(bfull_bar(s), 1); mbar_init(bempty_bar(s), 1); }
        for (int b = 0; b < 2; b++) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 8); }   // 8 epilogue warps arrive
        mbar_init(bres_free_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (elect_one()) {
            int sa = 0; uint32_t pha = 0;
            int sb = 0; uint32_t phb = 0;
            int k_tile = 0, last_n = -1;
            uint32_t reload_phase = 0;
            for (long long t = blockIdx.x; t < p.total_tiles; t += gridDim.x, k_tile++) {
                const TileCoord tc = decode_tile(p, t);
                const int wn = p.wgt_per_sample ? tc.n0 : 0;
                // resident weights are (re)loaded on the first tile and whenever the sample changes (per-sample weights)
                const bool load_res = p.b_resident && (k_tile == 0 || (p.wgt_per_sample && tc.n0 != last_n));
                if (load_res && k_tile > 0) {   // every MMA that reads the old weights must have retired: the MMA warp commits to
                    mbar_wait(bres_free_bar, reload_phase);     // this barrier after the last tile of each sample (waited in order,
                    reload_phase ^= 1;                          // one phase per reload, so the parity is never ambiguous)
                }
                last_n = tc.n0;
                if (load_res) {
                    // all resident weight tiles first (the MMA warp waits for the whole set before touching the activation
                    // ring, so they must not be queued behind activation stages it has not released yet)
                    int b_slot = 0;
                    for (int g = 0; g < p.n_groups; g++) {
                        const int ky0 = p.reuse ? 0 : g / p.kw;
                        const int kx = p.reuse ? g : g - ky0 * p.kw;
                        for (int cb = 0; cb < p.num_cb; cb++)
                            for (int j = 0; j < p.inner; j++)
                                for (int pb = 0; pb < p.parts; pb++, b_slot++) {
                                    mbar_expect_tx(bfull_bar(b_slot), p.b_bytes);
                                    tma_load_4d(b_base + b_slot * p.b_pitch, &map_b, bfull_bar(b_slot), cb * p.kb,
                                                (p.reuse == 2 ? j : (ky0 + j) * p.kw + kx) * p.o_rows + tc.col0, pb, wn);
                                }
                    }
                }
                if (p.reuse == 2) {
                    if (p.dbg & 64) continue;
                    // one slab (TW + kw - 1) x (TH + kh - 1) pixels per (channel block, part); stages are single parts
                    for (int cb = 0; cb < p.num_cb; cb++)
                        for (int pa = 0; pa < p.parts; pa++) {
                            mbar_wait(aempty_bar(sa), pha ^ 1);
                            mbar_expect_tx(afull_bar(sa), p.a_tx_bytes);
                            tma_load_5d(smem_base + sa * p.a_stage_bytes, &map_a, afull_bar(sa), cb * p.kb, tc.x0 - p.pad_x, tc.y0 - p.pad_y, tc.n0, pa);
                            if (++sa == SA) { sa = 0; pha ^= 1; }
                        }
                    continue;
                }
                for (int g = 0; g < p.n_groups; g++) {
                    // reuse: group = kx, the slab spans all ky;  no reuse: group = tap
                    const int ky0 = p.reuse ? 0 : g / p.kw;
                    const int kx = p.reuse ? g : g - ky0 * p.kw;
                    const int ix = tc.x0 * p.stride + kx - p.pad_x;
                    const int iy = tc.y0 * p.stride + ky0 - p.pad_y;
                    for (int cb = 0; cb < p.num_cb; cb++) {
                        mbar_wait(aempty_bar(sa), pha ^ 1);
                        mbar_expect_tx(afull_bar(sa), p.a_tx_bytes);
                        for (int pa = 0; pa < p.parts; pa++)
                            tma_load_5d(smem_base + sa * p.a_stage_bytes + pa * p.slab_bytes, &map_a, afull_bar(sa), cb * p.kb, ix, iy, tc.n0, pa);
                        if (++sa == SA) { sa = 0; pha ^= 1; }
                        if (p.b_resident) continue;
                        for (int j = 0; j < p.inner; j++) {
                            const int tap = (ky0 + j) * p.kw + kx;
                            for (int pb = 0; pb < p.parts; pb++) {
                                mbar_wait(bempty_bar(sb), phb ^ 1);
                                mbar_expect_tx(bfull_bar(sb), p.b_bytes);
                                tma_load_4d(b_base + sb * p.b_pitch, &map_b, bfull_bar(sb), cb * p.kb, tap * p.o_rows + tc.col0, pb, wn);
                                if (++sb == SB) { sb = 0; phb ^= 1; }
                            }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        const MmaCtx mc{smem_base, b_base, bar_base, tmem_base};
        const int ks = p.kb == (F8 ? 128 : 64) ? 4 : 0;     // 128-byte channel blocks
        const bool res = p.b_resident != 0;
        if constexpr (F8) {     // e4m3 operands are one part
            if (p.reuse == 2 && p.slab9) mma_role_slab9<F8, 1, false>(p, mc);
            else if (p.reuse == 2) { if (p.inner == 9) mma_role_slab<F8, 1, 9, false>(p, mc); else mma_role_slab<F8, 1, 0, false>(p, mc); }
            else if (ks == 4 && p.inner == 3) { if (res) mma_role<F8, 1, 3, 4, true>(p, mc); else mma_role<F8, 1, 3, 4, false>(p, mc); }
            else if (ks == 4 && p.inner == 7) mma_role<F8, 1, 7, 4, false>(p, mc);
            else if (ks == 4 && p.inner == 1) { if (res) mma_role<F8, 1, 1, 4, true>(p, mc); else mma_role<F8, 1, 1, 4, false>(p, mc); }
            else if (res) mma_role<F8, 1, 0, 0, true>(p, mc);
            else mma_role<F8, 1, 0, 0, false>(p, mc);
        }
        else if (p.reuse == 2 && p.slab9) {
            if (p.parts == 1) mma_role_slab9<F8, 1, false>(p, mc);
            else if (p.stack) mma_role_slab9<F8, 2, true>(p, mc);
            else mma_role_slab9<F8, 2, false>(p, mc);
        }
        else if (p.reuse == 2) {
            if (p.inner == 9 && p.parts == 1) mma_role_slab<F8, 1, 9, false>(p, mc);
            else if (p.inner == 9 && p.parts == 2 && p.stack) mma_role_slab<F8, 2, 9, true>(p, mc);
            else if (p.inner == 9 && p.parts == 2) mma_role_slab<F8, 2, 9, false>(p, mc);
            else if (p.stack) mma_role_slab<F8, 2, 0, true>(p, mc);
            else mma_role_slab<F8, 0, 0, false>(p, mc);
        }
        else if (ks == 4 && p.inner == 3 && p.parts == 1) { if (res) mma_role<F8, 1, 3, 4, true>(p, mc); else mma_role<F8, 1, 3, 4, false>(p, mc); }
        else if (ks == 4 && p.inner == 3 && p.parts == 2 && p.stack) mma_role<F8, 2, 3, 4, true, true>(p, mc);
        else if (ks == 4 && p.inner == 1 && p.parts == 2 && p.stack) mma_role<F8, 2, 1, 4, true, true>(p, mc);
        else if (ks == 4 && p.inner == 3 && p.parts == 2) { if (res) mma_role<F8, 2, 3, 4, true>(p, mc); else mma_role<F8, 2, 3, 4, false>(p, mc); }
        else if (ks == 4 && p.inner == 3 && p.parts == 3) mma_role<F8, 3, 3, 4, false>(p, mc);
        else if (ks == 4 && p.inner == 7 && p.parts == 1) mma_role<F8, 1, 7, 4, false>(p, mc);
        else if (ks == 4 && p.inner == 7 && p.parts == 2) mma_role<F8, 2, 7, 4, false>(p, mc);
        else if (ks == 4 && p.inner == 1 && p.parts == 1) { if (res) mma_role<F8, 1, 1, 4, true>(p, mc); else mma_role<F8, 1, 1, 4, false>(p, mc); }
        else if (ks == 4 && p.inner == 1 && p.parts == 2) { if (res) mma_role<F8, 2, 1, 4, true>(p, mc); else mma_role<F8, 2, 1, 4, false>(p, mc); }
        else if (res) mma_role<F8, 0, 0, 0, true>(p, mc);
        else mma_role<F8, 0, 0, 0, false>(p, mc);
    } else if (EPI == 1) {
        // ===================== epilogue warps, operand-format hand-over =====================
#define PGPP_PACKED(ACT) \
        if (p.accumulate) { if (p.stack) epilogue_packed_role<ACT, true, true>(p, bar_base, tmem_base, s_params, warp, lane);   \
                            else         epilogue_packed_role<ACT, false, true>(p, bar_base, tmem_base, s_params, warp, lane); } \
        else              { if (p.stack) epilogue_packed_role<ACT, true, false>(p, bar_base, tmem_base, s_params, warp, lane);  \
                            else         epilogue_packed_role<ACT, false, false>(p, bar_base, tmem_base, s_params, warp, lane); }
#define PGPP_PACKED_F8(ACT) \
        if (p.accumulate) epilogue_packed_role<ACT, false, true, true>(p, bar_base, tmem_base, s_params, warp, lane);  \
        else              epilogue_packed_role<ACT, false, false, true>(p, bar_base, tmem_base, s_params, warp, lane);
        if constexpr (F8) {     // one part: never stacked
            if (p.act_fn == PGPP_ACT_LINEAR) { PGPP_PACKED_F8(PGPP_ACT_LINEAR) }
            else if (p.act_fn == PGPP_ACT_RELU) { PGPP_PACKED_F8(PGPP_ACT_RELU) }
            else { PGPP_PACKED_F8(PGPP_ACT_LRELU) }
        } else {
        if (p.act_fn == PGPP_ACT_LINEAR) { PGPP_PACKED(PGPP_ACT_LINEAR) }
        else if (p.act_fn == PGPP_ACT_RELU) { PGPP_PACKED(PGPP_ACT_RELU) }
        else { PGPP_PACKED(PGPP_ACT_LRELU) }
        }
#undef PGPP_PACKED_F8
#undef PGPP_PACKED
    } else {
        // ===================== epilogue warps =====================
        const int quarter = warp & 3;                       // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;                   // which half of the columns
        const int lane_row = quarter * 32 + lane;
        PixelCoord pc;
        pc.px = lane_row % p.tw;
        pc.py = (lane_row / p.tw) % p.th;
        pc.pn = lane_row / (p.tw * p.th);
        const int etid = threadIdx.x - 64;                  // 0..255 among the epilogue threads
        const int cols_per = p.block_n >= 32 ? p.block_n / 2 : p.block_n;
        const int col_begin = half * cols_per;
        const int col_end = (p.block_n >= 32 || half == 0) ? col_begin + cols_per : col_begin;
        const bool fast = p.tn == 1 && p.fold_gain;
        int buf = 0; uint32_t buf_phase = 0;
        int tag0 = -1, tag1 = -1;                           // (sample, column tile) whose parameters each staging buffer holds
        for (long long t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
            const TileCoord tc = decode_tile(p, t);
            float2* s_cs = s_params + buf * p.block_n;
            if (fast) {
                const int tag = tc.n0 * p.tiles_col + tc.col0 / p.block_n;
                if ((buf ? tag1 : tag0) != tag) {
                    // every epilogue warp must be done with the tile that last used this buffer before it is rewritten
                    asm volatile("bar.sync 1, 256;" ::: "memory");
                    if (etid < p.block_n) {
                        const int g = tc.col0 + etid;
                        const int phase = (g >= p.phase_stride) + (g >= 2 * p.phase_stride) + (g >= 3 * p.phase_stride);
                        const int oc = g - phase * p.phase_stride;
                        float sc = 1.f, sh = 0.f;
                        if (oc < p.o && phase < p.phases) {
                            if (p.dcoef) sc = __ldg(p.dcoef + (long long)tc.n0 * p.o + oc);
                            if (F8) sc *= weight_scale(p, tc.n0, g);
                            if (p.bias) sh = __ldg(p.bias + oc);
                        }
                        if (p.spade_x) {        // (rstd | mean of the normalised tensor, bias of gamma | beta)
                            const int C = p.o >> 1;
                            const float st = etid < C ? __ldg(p.spade_rstd + (long long)tc.n0 * C + etid)
                                                      : (etid < p.o ? __ldg(p.spade_mean + (long long)tc.n0 * C + (etid - C)) : 0.f);
                            s_cs[etid] = make_float2(st, sh);
                        } else
                        s_cs[etid] = make_float2(sc * p.gain, sh * p.gain);
                    }
                    asm volatile("bar.sync 1, 256;" ::: "memory");
                    if (buf) tag1 = tag; else tag0 = tag;
                }
            }
            // the pixel's noise value does not depend on the accumulators: fetch it while the MMAs of this tile are still running
            float nz_pre = 0.f;
            if (fast && p.noise && p.phases == 1) {
                const int x = tc.x0 + pc.px, y = tc.y0 + pc.py;
                if (x < p.conv_w && y < p.conv_h) nz_pre = __ldg(p.noise + tc.n0 * p.noise_stride_n + (long long)y * p.out_w + x) * p.gain;
            }
            mbar_wait(tfull_bar(buf), buf_phase);
            tc_fence_after();
            const uint32_t tmem_tile = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * p.acc_cols);
            // instance-norm partials: row (pixel tile, lane quarter) of the workspace, pixel tiles numbered sample-major
            float* stats_row = nullptr;
            if (p.stats_ws) stats_row = p.stats_ws + ((long long)fast_div((unsigned)t, p.div_col_m, p.div_col_s) * 4 + quarter) * p.o;
            if (p.spade_x) epilogue_spade<F8>(p, tc, tmem_tile, pc, half, s_cs);
            else if (p.out_dtype == PGPP_F32) epilogue_dispatch<float, F8>(p, tc, tmem_tile, pc, col_begin, col_end, s_cs, fast, nz_pre, stats_row);
            else if (p.out_dtype == PGPP_BF16) epilogue_dispatch<__nv_bfloat16, F8>(p, tc, tmem_tile, pc, col_begin, col_end, s_cs, fast, nz_pre, nullptr);
            else epilogue_dispatch<__half, F8>(p, tc, tmem_tile, pc, col_begin, col_end, s_cs, fast, nz_pre, nullptr);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(buf));
            if (++buf == 2) { buf = 0; buf_phase ^= 1; }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// host side


} // namespace pgpp

namespace pgpp { static int igemm_launch(const pgpp_conv_desc* d, void* stream, long long* stats_rows_query); }

extern "C" int pgpp_conv2d_igemm(const pgpp_conv_desc* d, void* stream) { return pgpp::igemm_launch(d, stream, nullptr); }

extern "C" int64_t pgpp_conv2d_igemm_stats_rows(const pgpp_conv_desc* d) {
    long long rows = 0;
    const int rc = pgpp::igemm_launch(d, nullptr, &rows);
    return rc == PGPP_OK ? (int64_t)rows : (int64_t)rc;
}

// mean / rstd from the warp partials (pivot, sum of deviations, sum of squared deviations over 32 pixels each): all partials have the same
// count, so  mean = avg(mean_w),  M2 = sum M2_w + 32 * sum (mean_w - mean)^2  with  mean_w = pivot + s1 / 32,  M2_w = s2 - s1^2 / 32;
// accumulated in float64 (the between-partial term is formed from sums of mean_w and mean_w^2).
namespace pgpp {
__global__ void __launch_bounds__(512) instnorm_finalize_kernel(const float* ws, long long rows, long long rows_per_sample, int c, float eps,
                                                                 float* mean, float* rstd) {
    // 8 channels x 64 row slices per CTA (a warp reads four 32-byte row segments per load), 8 rows in flight per thread: also at batch 1
    // (a handful of CTAs) the walk over the 8192 partials of a 512 x 512 sample takes a few microseconds
    __shared__ double sh[3][64][9];
    const int chl = threadIdx.x & 7, slice = threadIdx.x >> 3;
    const int ch = blockIdx.x * 8 + chl, n = blockIdx.y;
    const long long plane = rows * c;
    double a = 0.0, b = 0.0, m2 = 0.0;
    if (ch < c) {
        const float* base = ws + (long long)n * rows_per_sample * c + ch;
        for (long long r0 = slice; r0 < rows_per_sample; r0 += 64 * 8) {
            float pv[8], s1[8], s2[8];
            #pragma unroll
            for (int k = 0; k < 8; k++) {
                const long long r = r0 + 64 * k;
                const bool ok = r < rows_per_sample;
                pv[k] = ok ? __ldg(base + r * c) : 0.f;
                s1[k] = ok ? __ldg(base + plane + r * c) : 0.f;
                s2[k] = ok ? __ldg(base + 2 * plane + r * c) : 0.f;
            }
            #pragma unroll
            for (int k = 0; k < 8; k++) {
                if (r0 + 64 * k >= rows_per_sample) break;
                const double mw = (double)pv[k] + (double)s1[k] * (1.0 / 32.0);
                a += mw; b += mw * mw;
                m2 += (double)s2[k] - (double)s1[k] * (double)s1[k] * (1.0 / 32.0);
            }
        }
    }
    sh[0][slice][chl] = a; sh[1][slice][chl] = b; sh[2][slice][chl] = m2;
    __syncthreads();
    // fixed-order tree over the 64 slices (deterministic)
    for (int step = 32; step > 0; step >>= 1) {
        if (slice < step) {
            sh[0][slice][chl] += sh[0][slice + step][chl]; sh[1][slice][chl] += sh[1][slice + step][chl]; sh[2][slice][chl] += sh[2][slice + step][chl];
        }
        __syncthreads();
    }
    if (slice == 0 && ch < c) {
        a = sh[0][0][chl]; b = sh[1][0][chl]; m2 = sh[2][0][chl];
        const double w = (double)rows_per_sample;
        const double mu = a / w;
        double var = (m2 + 32.0 * (b - a * a / w)) / (32.0 * w);
        if (var < 0.0) var = 0.0;
        mean[(long long)n * c + ch] = (float)mu;
        rstd[(long long)n * c + ch] = (float)(1.0 / sqrt(var + (double)eps));
    }
}
} // namespace pgpp

extern "C" int pgpp_instnorm_finalize(const float* ws, int64_t rows, int n, int c, float eps, float* mean, float* rstd, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(ws && mean && rstd, "ws, mean and rstd must be device pointers");
    PGPP_REQUIRE(n >= 1 && c >= 1 && rows >= n && rows % n == 0, "rows must be a positive multiple of n");
    dim3 grid((unsigned)((c + 7) / 8), (unsigned)n);
    instnorm_finalize_kernel<<<grid, 512, 0, (cudaStream_t)stream>>>(ws, rows, rows / n, c, eps, mean, rstd);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

static int pgpp::igemm_launch(const pgpp_conv_desc* d, void* stream, long long* stats_rows_query) {
    using namespace pgpp;
    PGPP_REQUIRE(d != nullptr, "desc is NULL");
    PGPP_REQUIRE(d->act && d->wgt && d->out, "act, wgt and out must be device pointers");
    PGPP_REQUIRE(d->n >= 1 && d->h >= 1 && d->w >= 1 && d->conv_h >= 1 && d->conv_w >= 1, "empty problem");
    PGPP_REQUIRE(d->c_pad >= 16 && d->c_pad % 16 == 0, "c_pad must be a positive multiple of 16");
    PGPP_REQUIRE(d->kh >= 1 && d->kw >= 1, "filter must be at least 1x1");
    PGPP_REQUIRE(d->stride == 1 || d->stride == 2, "stride must be 1 or 2");
    PGPP_REQUIRE(d->phases == 1 || d->phases == 4, "phases must be 1 or 4");
    PGPP_REQUIRE(d->phase_stride >= d->o && (d->phases == 1 ? d->phase_stride == d->o : d->phase_stride % 16 == 0),
                 "phase_stride must be o (phases == 1) or a multiple of 16 >= o (phases == 4)");
    PGPP_REQUIRE(d->block_n == 16 || d->block_n == 32 || d->block_n == 64 || d->block_n == 128 || d->block_n == 256,
                 "block_n must be 16, 32, 64, 128 or 256");
    PGPP_REQUIRE(d->o >= 1 && d->o_rows >= d->phases * d->phase_stride && d->o_rows % d->block_n == 0,
                 "o_rows must cover phases*phase_stride and be a multiple of block_n");
    PGPP_REQUIRE(d->products == 1 || d->products == 3 || d->products == 6, "products must be 1, 3 or 6");
    const int need_parts = d->products == 1 ? 1 : (d->products == 3 ? 2 : 3);
    PGPP_REQUIRE(d->a_parts >= need_parts && d->b_parts >= need_parts, "operand parts do not cover the requested products");
    const bool e4m3 = d->operand_e4m3 != 0;
    const int esize = e4m3 ? 1 : 2;             // bytes per operand element
    PGPP_REQUIRE(d->out_dtype == PGPP_F32 || d->out_dtype == PGPP_BF16 || d->out_dtype == PGPP_F16 || (e4m3 && d->out_dtype == PGPP_E4M3),
                 "unsupported output dtype (e4m3 output needs e4m3 operands)");
    if (e4m3) {
        PGPP_REQUIRE(d->products == 1 && !d->operand_f16, "e4m3 operands are one part (products must be 1)");
        PGPP_REQUIRE(d->wscale != nullptr, "e4m3 operands need the weight column scales (wscale)");
        PGPP_REQUIRE(d->c_pad % 32 == 0, "e4m3 operands: c_pad must be a multiple of 32");
    }
    PGPP_REQUIRE(d->act_fn >= 1 && d->act_fn <= 9, "no CUDA kernel found for the specified activation func");
    PGPP_REQUIRE(((uintptr_t)d->act & 15) == 0 && ((uintptr_t)d->wgt & 15) == 0, "packed operands must be 16-byte aligned");
    const int out_parts = d->out_parts <= 0 ? 1 : d->out_parts;
    PGPP_REQUIRE(out_parts <= 3, "out_parts must be 1, 2 or 3");
    PGPP_REQUIRE(out_parts == 1 || (d->out_dtype == PGPP_BF16 && d->out_stride[1] == 1 && d->o % 16 == 0 &&
                                    d->out_stride[3] % 8 == 0 && d->out_part_stride % 8 == 0 && ((uintptr_t)d->out & 15) == 0),
                 "split output needs bf16, channels-innermost, 16-byte aligned pixels, out channels % 16 == 0");
    const int pix_stride = d->act_pixel_stride > 0 ? d->act_pixel_stride : d->c_pad;
    PGPP_REQUIRE(pix_stride >= d->c_pad && (pix_stride * esize) % 16 == 0, "act_pixel_stride must be >= c_pad and a multiple of 16 bytes");
    const int up = d->phases == 4 ? 2 : 1;
    PGPP_REQUIRE(d->out_h == d->conv_h * up && d->out_w == d->conv_w * up, "output size does not match the conv grid");

    EncodeTiledFn encode = get_encode_fn();
    if (!encode) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return PGPP_ERR_CUDA; }

    IgemmParams p;
    p.n = d->n; p.h = d->h; p.w = d->w; p.conv_h = d->conv_h; p.conv_w = d->conv_w;
    p.kh = d->kh; p.kw = d->kw; p.pad_y = d->pad_y; p.pad_x = d->pad_x; p.stride = d->stride;
    if (e4m3) p.kb = (d->c_pad % 128 == 0) ? 128 : ((d->c_pad % 64 == 0) ? 64 : 32);      // channels = bytes
    else p.kb = (d->c_pad % 64 == 0) ? 64 : ((d->c_pad % 32 == 0) ? 32 : 16);
    p.num_cb = d->c_pad / p.kb;
    p.parts = need_parts;
    // products of the bf16 expansions: parts 1 -> a0b0; 2 -> a0b0 + a1b0 + a0b1; 3 -> + a2b0 + a1b1 + a0b2
    p.pa_mask[0] = (1u << need_parts) - 1u;
    p.pa_mask[1] = need_parts == 3 ? 3u : 1u;
    p.pa_mask[2] = 1u;
    p.o = d->o; p.phases = d->phases; p.phase_stride = d->phase_stride; p.o_rows = d->o_rows; p.block_n = d->block_n; p.up = up;
    // pixel tile TW x TH x TN = 128.  Stride-1 convs with kh > 1 on images of at least 16 x 8 use a 16 x 8 tile so that
    // one slab of TH + kh - 1 rows serves all vertical taps (ky reuse); everything else takes the widest tile.
    const int dil_y = d->dil_y > 1 ? d->dil_y : 1;
    PGPP_REQUIRE(dil_y == 1 || d->stride == 1, "dil_y > 1 needs stride 1");
    p.reuse = (d->stride == 1 && d->kh > 1 && d->conv_w >= 16 && d->conv_h >= 8 && (d->kh - 1) * dil_y <= 6) ? 1 : 0;
    PGPP_REQUIRE(dil_y == 1 || p.reuse, "dil_y > 1 is only supported on the slab-reuse path (images of at least 16 x 8, (kh-1)*dil_y <= 6)");
    const EnvFlags& env = env_flags();
    if (env.igemm_no_reuse) p.reuse = 0;
    // single-slab mode (reuse == 2): layers whose GEMM N is at most 64 are bound by the L2 -> shared-memory traffic of the three
    // filter-column slabs; an 8 x 16 pixel tile reads ONE (8 + kw - 1) x (16 + kh - 1) slab per (channel block, part) instead and
    // takes every tap as a row-shifted descriptor view of it (2.7x fewer activation bytes for 3 x 3).  Needs resident weights.
    const int slab_pitch = 8 + d->kw - 1, slab_rows2 = 16 + d->kh - 1;
    const int row_ch = e4m3 ? 128 : 64;         // channels of a 128-byte row
    const bool slab2_shape = d->stride == 1 && d->kh * d->kw > 1 && d->kh * d->kw <= 64 && dil_y == 1 && d->c_pad % row_ch == 0 && d->block_n <= 64 &&
                             d->phases * d->phase_stride <= d->block_n && d->conv_w >= 8 && d->conv_h >= 16 && need_parts <= 2 &&
                             !env.igemm_no_slab2 && !env.igemm_no_resident;
    if (slab2_shape) {
        const long long stage = ((long long)slab_pitch * slab_rows2 * 128 + 1023) & ~1023ll;
        const long long n_bt = (long long)(d->c_pad / row_ch) * d->kh * d->kw * need_parts;
        const long long b_pitch2 = ((long long)d->block_n * 128 + 1023) & ~1023ll;
        const long long need = 1024 + 2 * stage + n_bt * b_pitch2 + 8 * (2 * 2 + 2 * n_bt + 5) + 32 + 16ll * d->block_n;
        const long long tiles = (long long)((d->conv_w + 7) / 8) * ((d->conv_h + 15) / 16) * d->n;
        if (n_bt <= 64 && need <= 227 * 1024 && tiles > sm_count()) p.reuse = 2;
    }
    if (p.reuse == 2) { p.tw = 8; p.th = 16; p.tn = 1; }
    else if (p.reuse) { p.tw = 16; p.th = 8; p.tn = 1; }
    else {
        p.tw = pow2_ceil(d->conv_w); if (p.tw > kTileM) p.tw = kTileM;
        p.th = pow2_ceil(d->conv_h); if (p.th > kTileM / p.tw) p.th = kTileM / p.tw;
        p.tn = kTileM / (p.tw * p.th);
    }
    p.n_groups = p.reuse == 2 ? 1 : (p.reuse ? d->kw : d->kh * d->kw);
    p.inner = p.reuse == 2 ? d->kh * d->kw : (p.reuse ? d->kh : 1);
    p.tiles_x = (d->conv_w + p.tw - 1) / p.tw;
    p.tiles_y = (d->conv_h + p.th - 1) / p.th;
    p.tiles_n = (d->n + p.tn - 1) / p.tn;
    p.tiles_col = (d->phases * d->phase_stride + d->block_n - 1) / d->block_n;
    p.total_tiles = (long long)p.tiles_x * p.tiles_y * p.tiles_n * p.tiles_col;
    const unsigned row_bytes = (unsigned)(p.kb * esize);
    const int slab_rows = p.tn * (p.th + (p.inner - 1) * dil_y) * p.tw;        // multiple of 8 (TW % 8 == 0 with reuse, 128 without)
    p.slab_bytes = (unsigned)slab_rows * row_bytes;
    p.a_tx_bytes = p.parts * p.slab_bytes;
    p.a_stage_bytes = (p.a_tx_bytes + 1023u) & ~1023u;
    p.sbo_a = 8 * row_bytes;
    for (int j = 0; j < 64; j++) p.tap_off16[j] = 0;
    if (p.reuse == 2) {             // one part per stage; tap (ky, kx) starts (ky * pitch + kx) pixel rows into the slab
        p.slab_bytes = (unsigned)(slab_pitch * slab_rows2) * row_bytes;
        p.a_tx_bytes = p.slab_bytes;
        p.a_stage_bytes = (p.slab_bytes + 1023u) & ~1023u;
        p.sbo_a = (unsigned)slab_pitch * row_bytes;
        for (int ky = 0; ky < d->kh; ky++)
            for (int kx = 0; kx < d->kw; kx++)
                p.tap_off16[ky * d->kw + kx] = (unsigned short)(((ky * slab_pitch + kx) * row_bytes) >> 4);
    }
    p.ky_step_bytes = (unsigned)(p.tw * dil_y) * row_bytes;
    p.b_bytes = (unsigned)d->block_n * row_bytes;
    p.b_pitch = (p.b_bytes + 1023u) & ~1023u;
    p.layout_type = row_bytes == 128 ? 2u : (row_bytes == 64 ? 4u : 6u);   // SWIZZLE_128B / 64B / 32B
    p.sbo_bytes = 8 * row_bytes;
    // instruction descriptor (cute/arch/mma_sm100_desc.hpp InstrDescriptor): fp32 accum, bf16 A/B, K-major, M = 128
    // a_format / b_format (bits 7-9 / 10-12): 1 = bf16, 0 = f16 (the fp16 layers of the discriminator run native f16 MMAs)
    // kind::f8f6f4: a_format / b_format 0 = E4M3
    const unsigned ab_fmt = (d->operand_f16 || e4m3) ? 0u : ((1u << 7) | (1u << 10));
    PGPP_REQUIRE(!d->operand_f16 || d->products == 1, "fp16 operands are a single part (products must be 1)");
    p.idesc = (1u << 4) | ab_fmt | ((unsigned)(d->block_n >> 3) << 17) | ((unsigned)(kTileM >> 4) << 24);
    unsigned cols = (unsigned)pow2_ceil(2 * d->block_n); if (cols < 32) cols = 32;
    p.tmem_cols = cols;
    // shared-memory plan (227 KB per CTA): weights resident if every tile of a column tile fits beside a 2-deep
    // activation ring, otherwise a weight ring of up to 8 slots and 2..4 activation stages
    auto smem_need = [&](long long a_st, long long b_st) -> long long {
        return 1024 + a_st * p.a_stage_bytes + b_st * p.b_pitch + 8 * (2 * a_st + 2 * b_st + 5) + 16 + 16 + 16ll * p.block_n;
    };
    const long long smem_max = 227 * 1024;
    const long long n_btiles = (long long)p.n_groups * p.num_cb * p.inner * p.parts;
    p.b_resident = 0;
    if (p.tiles_col == 1 && n_btiles <= 64 && !env.igemm_no_resident && smem_need(2, n_btiles) <= smem_max &&
        p.total_tiles > sm_count()) {
        p.b_resident = 1;
        p.b_stages = (int)n_btiles;
        p.a_stages = 2;
        while (p.a_stages < (p.reuse == 2 ? 8 : 6) && smem_need(p.a_stages + 1, n_btiles) <= smem_max) p.a_stages++;
    } else {
        PGPP_REQUIRE(p.reuse != 2, "internal: single-slab mode needs resident weights");
        p.a_stages = 2;
        p.b_stages = 2;
        if (smem_need(2, 2) > smem_max) { set_error("tile does not fit shared memory"); return PGPP_ERR_UNSUPPORTED; }
        while (p.b_stages < 8 && smem_need(p.a_stages, p.b_stages + 1) <= smem_max) p.b_stages++;
        while (p.a_stages < 4 && smem_need(p.a_stages + 1, p.b_stages) <= smem_max) p.a_stages++;
    }
    const size_t smem_bytes = (size_t)smem_need(p.a_stages, p.b_stages);
    p.dcoef = d->dcoef; p.noise = d->noise; p.noise_stride_n = d->noise_stride_n; p.bias = d->bias;
    p.act_fn = d->act_fn; p.alpha = d->alpha; p.gain = d->gain; p.clamp = d->clamp;
    p.out = d->out; p.out_dtype = d->out_dtype; p.out_h = d->out_h; p.out_w = d->out_w;
    p.os_n = d->out_stride[0]; p.os_c = d->out_stride[1]; p.os_h = d->out_stride[2]; p.os_w = d->out_stride[3];
    p.accumulate = d->accumulate;
    p.wgt_per_sample = d->wgt_per_sample ? 1 : 0;
    p.out_parts = out_parts; p.out_part_stride = d->out_part_stride;
    PGPP_REQUIRE(!p.wgt_per_sample || p.tn == 1, "per-sample weights need images of at least 128 pixels (one sample per tile)");
    p.spade_x = d->spade_x; p.spade_mean = d->spade_mean; p.spade_rstd = d->spade_rstd; p.spade_pre_gain = d->spade_pre_gain;
    if (d->spade_x) {
        PGPP_REQUIRE(d->spade_mean && d->spade_rstd, "SPADE epilogue needs mean and rstd");
        PGPP_REQUIRE(d->phases == 1 && d->o % 32 == 0 && d->block_n == d->o && d->stride == 1 && p.tn == 1,
                     "SPADE epilogue: o = 2C (gamma | beta) with C % 16 == 0 in ONE column tile (block_n == o), stride 1, images of at least 128 pixels");
        PGPP_REQUIRE((d->out_dtype == PGPP_BF16 || (e4m3 && d->out_dtype == PGPP_E4M3 && out_parts == 1 && d->out_stride[3] % 16 == 0)) &&
                     d->out_stride[1] == 1 && !d->accumulate && d->out_stride[3] % 8 == 0 && d->out_part_stride % 8 == 0 && ((uintptr_t)d->out & 15) == 0,
                     "SPADE epilogue writes the channels-innermost bf16 (or, from e4m3 operands, e4m3) operand format (16-byte aligned pixels)");
        PGPP_REQUIRE(d->act_fn == PGPP_ACT_LINEAR && d->gain == 1.f && d->clamp < 0.f && !d->noise && !d->dcoef,
                     "SPADE epilogue: the GEMM itself must be linear (no noise, demodulation, gain or clamp)");
    }
    p.fold_gain = (d->gain > 0.f && (d->act_fn == PGPP_ACT_LINEAR || d->act_fn == PGPP_ACT_RELU ||
                                     (d->act_fn == PGPP_ACT_LRELU && d->alpha >= 0.f && d->alpha <= 1.f))) ? 1 : 0;
    // stacked products (see mma_role): fp32-parity mode with 2 parts, resident 64-column weight tiles, fast epilogue
    p.stack = (need_parts == 2 && d->block_n == 64 && p.b_resident && p.kb == 64 && (p.inner == 3 || p.inner == 1 || p.reuse == 2) && p.tn == 1 && p.fold_gain &&
               !d->spade_x && !env.igemm_no_stack) ? 1 : 0;
    p.slab9 = (p.reuse == 2 && d->kh == 3 && d->kw == 3 && row_bytes == 128 && d->block_n == 64 && p.b_pitch == 8192 && need_parts <= 2 &&
               env.igemm_slab9) ? 1 : 0;       // opt-in (PGPP_IGEMM_SLAB9=1): measured neutral in fp32-parity mode, 5 % slower in bf16 mode
    p.acc_cols = p.stack ? 2 * d->block_n : d->block_n;
    p.idesc_stack = (1u << 4) | ab_fmt | ((unsigned)((2 * d->block_n) >> 3) << 17) | ((unsigned)(kTileM >> 4) << 24);
    if (p.stack) p.tmem_cols = 256;
    auto magic = [](unsigned dv, unsigned& m, unsigned& sft) {
        sft = 0; while ((1ull << sft) < dv) sft++;
        m = (unsigned)(((1ull << (31 + sft)) + dv - 1) / dv);
    };
    magic((unsigned)p.tiles_col, p.div_col_m, p.div_col_s);
    magic((unsigned)p.tiles_x, p.div_x_m, p.div_x_s);
    magic((unsigned)p.tiles_y, p.div_y_m, p.div_y_s);
    PGPP_REQUIRE(p.total_tiles < (1ll << 31), "too many tiles");
    p.dbg = env.igemm_debug;
    p.wscale = e4m3 ? d->wscale : nullptr;

    // instance-norm partials of the output (pgpp_conv_desc.stats_ws): fast float32 NCHW epilogue, full pixel tiles, whole 16-column chunks
    const bool stats_ok = p.tn == 1 && p.fold_gain && d->out_dtype == PGPP_F32 && d->phases == 1 && !d->accumulate && !d->spade_x && d->o % 16 == 0 &&
                          d->conv_w % p.tw == 0 && d->conv_h % p.th == 0 && out_parts == 1;
    const long long stats_rows = stats_ok ? (long long)p.tiles_x * p.tiles_y * p.tiles_n * 4 : 0;
    if (stats_rows_query) { *stats_rows_query = stats_rows; return PGPP_OK; }
    PGPP_REQUIRE(!d->stats_ws || stats_ok, "stats_ws: this launch cannot produce instance-norm statistics (see pgpp_conv2d_igemm_stats_rows)");
    PGPP_REQUIRE(((uintptr_t)d->stats_ws & 15) == 0, "stats_ws must be 16-byte aligned");
    p.stats_ws = d->stats_ws; p.stats_plane = stats_rows * d->o;

    // tensor maps
    CUtensorMap map_a, map_b;
    {
        const cuuint64_t dims[5] = {(cuuint64_t)d->c_pad, (cuuint64_t)d->w, (cuuint64_t)d->h, (cuuint64_t)d->n, (cuuint64_t)d->a_parts};
        const cuuint64_t pb = (cuuint64_t)pix_stride * esize;
        const cuuint64_t strides[4] = {pb, pb * d->w, pb * d->w * d->h, pb * d->w * d->h * d->n};
        cuuint32_t box[5] = {(cuuint32_t)p.kb, (cuuint32_t)(p.tw * d->stride), (cuuint32_t)((p.th + (p.inner - 1) * dil_y) * d->stride), (cuuint32_t)p.tn, 1};
        if (p.reuse == 2) { box[1] = (cuuint32_t)slab_pitch; box[2] = (cuuint32_t)slab_rows2; }
        const cuuint32_t estr[5] = {1, (cuuint32_t)d->stride, (cuuint32_t)d->stride, 1, 1};
        const CUtensorMapSwizzle sw = row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
        const CUtensorMapDataType el = e4m3 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
        CUresult r = encode(&map_a, el, 5, const_cast<void*>(d->act), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(activations) failed with CUresult %d", (int)r); return PGPP_ERR_CUDA; }
        const cuuint64_t wrows = (cuuint64_t)d->o_rows * d->kh * d->kw;
        const cuuint64_t wdims[4] = {(cuuint64_t)d->c_pad, wrows, (cuuint64_t)d->b_parts, (cuuint64_t)(d->wgt_per_sample ? d->n : 1)};
        const cuuint64_t rb = (cuuint64_t)d->c_pad * esize;
        const cuuint64_t wstrides[3] = {rb, rb * wrows, rb * wrows * d->b_parts};
        const cuuint32_t wbox[4] = {(cuuint32_t)p.kb, (cuuint32_t)d->block_n, 1, 1};
        const cuuint32_t westr[4] = {1, 1, 1, 1};
        r = encode(&map_b, el, 4, const_cast<void*>(d->wgt), wdims, wstrides, wbox, westr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(weights) failed with CUresult %d", (int)r); return PGPP_ERR_CUDA; }
    }
    // lean operand-format epilogue (EPI 1) when the launch needs nothing else
    // (e4m3 operands: the lean epilogue writes e4m3 - and is the only one that does)
    const bool epi_packed = p.tn == 1 && p.fold_gain && d->out_dtype == (e4m3 ? PGPP_E4M3 : PGPP_BF16) && p.os_c == 1 && d->phases == 1 && !d->spade_x &&
                            d->o % 16 == 0 && d->block_n >= 32 && ((uintptr_t)d->out & (e4m3 ? 15 : 31)) == 0 && p.os_w % 16 == 0 && p.os_h % 16 == 0 &&
                            p.os_n % 16 == 0 && p.out_part_stride % 16 == 0 && (!env.igemm_no_lean_epilogue || e4m3);
    PGPP_REQUIRE(d->out_dtype != PGPP_E4M3 || d->spade_x || (epi_packed && out_parts == 1 && !d->stats_ws),
                 "e4m3 output: one part, channels-innermost, 16-byte aligned pixels, o % 16 == 0, phases == 1, one sample per tile, "
                 "linear / relu / lrelu with gain > 0, block_n >= 32");
    {
        // once per device (the attribute is per function per context)
        static std::atomic<bool> done[64];
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64 || !done[dev].load(std::memory_order_acquire)) {
            PGPP_CUDA_OK(cudaFuncSetAttribute(igemm_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            PGPP_CUDA_OK(cudaFuncSetAttribute(igemm_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            PGPP_CUDA_OK(cudaFuncSetAttribute(igemm_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            PGPP_CUDA_OK(cudaFuncSetAttribute(igemm_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            if (dev >= 0 && dev < 64) done[dev].store(true, std::memory_order_release);
        }
    }
    long long grid = p.total_tiles;
    const int sms = sm_count();
    if (grid > sms) grid = sms;
    PGPP_REQUIRE(epi_packed || out_parts == 1 || !d->accumulate,
                 "accumulating into a split (operand-format) output needs the lean epilogue: one sample per tile, linear / relu / lrelu with gain > 0, "
                 "32-byte aligned pixels, block_n >= 32, phases == 1");
    if (e4m3) {
        if (epi_packed) igemm_kernel<1, true><<<(unsigned)grid, kThreads, smem_bytes, (cudaStream_t)stream>>>(map_a, map_b, p);
        else igemm_kernel<0, true><<<(unsigned)grid, kThreads, smem_bytes, (cudaStream_t)stream>>>(map_a, map_b, p);
    } else if (epi_packed) igemm_kernel<1, false><<<(unsigned)grid, kThreads, smem_bytes, (cudaStream_t)stream>>>(map_a, map_b, p);
    else igemm_kernel<0, false><<<(unsigned)grid, kThreads, smem_bytes, (cudaStream_t)stream>>>(map_a, map_b, p);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}
