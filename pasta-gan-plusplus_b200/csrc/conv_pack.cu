// Operand preparation for the tensor-core convolution (sm_100a).
//   pgpp_pack_activations : any-layout x (* per-(n,c) scale) -> channels-innermost bf16 parts
//   pgpp_modconv_demod_coefs : d[n,o] = rsqrt(sum (w*s)^2 + eps)     (training/networks.py:64-68)
// Both are small HBM-bound helpers; the heavy lifting is conv_igemm.cu.
#include "common.cuh"

namespace pgpp {

struct PackArgs {
    const void* x; const float* scale; __nv_bfloat16* out;
    int n, c, h, w, c_pad, parts;
    int c_total, c_off;         // destination pixel stride and first channel
    long long s_n, s_c, s_h, s_w;
    long long part_stride;      // elements between parts = n*h*w*c_pad
    int f16;                    // 1: the operand is IEEE half (one part) instead of the bf16 expansion (fp16 layers, native f16 MMA)
    int e4m3;                   // 1: the operand is ONE part of e4m3 bytes (fp8 inference precision); out and the strides count bytes
    // gradient of a fused bias_act (pgpp_pack_act_gradient): x = dy, gate = the saved output y (same dtype and strides)
    const void* gate; int act; float alpha, gain, clamp;
    float* csum;                // [N][C][x_tiles * y_tiles] per-tile channel sums of the packed gradient (the bias gradient), or NULL
};

__device__ __forceinline__ void split_store(float v, __nv_bfloat16* dst, long long part_stride, int parts, int f16 = 0) {
    if (f16) { *reinterpret_cast<__half*>(dst) = __float2half_rn(v); return; }
    // part p = bf16(v - sum of earlier parts): 8, 16, 24 significand bits for 1, 2, 3 parts
    #pragma unroll 3
    for (int p = 0; p < parts; p++) {
        const __nv_bfloat16 q = __float2bfloat16_rn(v);
        dst[p * part_stride] = q;
        v -= __bfloat162float(q);
    }
}

// ---- 64-channel x 128-pixel transposing tile shared by pack_nchw_kernel and spade_pack_kernel -------------------------
// The source is pixel-contiguous (NCHW-like), the destination channel-contiguous.  A CTA of 256 threads owns 64 channels of
// 128 pixels (tw x rows block of one image, tw a power of two).  Thread (warp w, lane l) loads channels 8w..8w+7 of pixels
// 4l..4l+3 (one 128-bit load per channel: a warp reads 512 contiguous bytes of one channel row), converts them to the bf16
// expansion in registers - 8 consecutive channels of one pixel are one 16-byte packet of the destination - and parks the
// packets in shared memory (XOR-swizzled by the lane so both sides are bank-conflict free); after one barrier 8 consecutive
// threads write the 128-byte channel row of a pixel with one 128-bit store each.
struct TileGeom { int log_tw, x_tiles, y_tiles, c_tiles; };

// 8 consecutive channels of pixel k as one 16-byte packet of the current bf16 part; `more`: another part follows, so the residual
// v - bf16(v) is left in v (packed conversions: one cvt.rn.bf16x2.f32 per channel pair)
__device__ __forceinline__ uint4 split_packet(float (&v)[8][4], int k, int f16 = 0, bool more = true, int e4m3 = 0) {
    if (e4m3)       // 8 bytes in the low half of the packet
        return make_uint4(e4m3x4(v[0][k], v[1][k], v[2][k], v[3][k]), e4m3x4(v[4][k], v[5][k], v[6][k], v[7][k]), 0u, 0u);
    if (f16) {
        __align__(16) __half hq[8];
        #pragma unroll
        for (int j = 0; j < 8; j++) hq[j] = __float2half_rn(v[j][k]);
        return *reinterpret_cast<const uint4*>(hq);
    }
    uint32_t w[4];
    #pragma unroll
    for (int j = 0; j < 4; j++) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j][k], v[2 * j + 1][k]);
        w[j] = *reinterpret_cast<const uint32_t*>(&h);
        if (more) {
            v[2 * j][k] -= __uint_as_float(w[j] << 16);
            v[2 * j + 1][k] -= __uint_as_float(w[j] & 0xffff0000u);
        }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// writes the tile held in v (see above) to out[part][n][y][x][c_off + c0 ...]; sm = parts * 128 * 8 packets
__device__ __forceinline__ void emit_tile(float (&v)[8][4], uint4* sm, int parts, __nv_bfloat16* out, long long part_stride,
                                          int n, int h, int w, int y0, int x0, int log_tw, int c0, int c_lim, int c_total, int c_off,
                                          int f16 = 0, int e4m3 = 0) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int part = 0; part < parts; part++) {
        #pragma unroll
        for (int k = 0; k < 4; k++)
            sm[(part * 128 + 4 * lane + k) * 8 + (warp ^ (lane & 7))] = split_packet(v, k, f16, part + 1 < parts, e4m3);
    }
    __syncthreads();
    const int tw_mask = (1 << log_tw) - 1;
    for (int part = 0; part < parts; part++) {
        #pragma unroll
        for (int it = 0; it < 4; it++) {
            const int item = it * 256 + threadIdx.x;
            const int px = item >> 3, ch = item & 7;
            const int y = y0 + (px >> log_tw), x = x0 + (px & tw_mask);
            if (y < h && x < w && c0 + ch * 8 < c_lim) {
                const long long idx = part * part_stride + (((long long)n * h + y) * w + x) * c_total + c_off + c0 + ch * 8;
                const uint4 pk = sm[(part * 128 + px) * 8 + (ch ^ ((px >> 2) & 7))];
                if (e4m3) *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(out) + idx) = make_uint2(pk.x, pk.y);
                else *reinterpret_cast<uint4*>(out + idx) = pk;
            }
        }
    }
}

__device__ __forceinline__ void decode_tile_block(const TileGeom& g, int& xt, int& yt, int& ct, int& n) {
    long long b = blockIdx.x;
    xt = (int)(b % g.x_tiles); b /= g.x_tiles;
    ct = (int)(b % g.c_tiles); b /= g.c_tiles;
    yt = (int)(b % g.y_tiles);
    n = (int)(b / g.y_tiles);
}

static TileGeom tile_geometry(int h, int w, int c_pad) {
    int tw;
    if (w % 128 == 0) tw = 128; else if (w % 64 == 0) tw = 64; else if (w % 32 == 0) tw = 32; else if (w % 16 == 0) tw = 16;
    else { tw = 16; while (tw < w && tw < 128) tw <<= 1; }
    TileGeom g;
    g.log_tw = 0; while ((1 << g.log_tw) < tw) g.log_tw++;
    const int rows = 128 / tw;
    g.x_tiles = (w + tw - 1) / tw;
    g.y_tiles = (h + rows - 1) / rows;
    g.c_tiles = (c_pad + 63) / 64;
    return g;
}

// VEC: float source, W % 4 == 0, all strides and the base pointer 16-byte aligned -> one 128-bit load per channel
// the stored value of the stand-alone gradient kernel (rounded to the tensor's dtype), so that the fused pass is bit-identical to it
template <class T> __device__ __forceinline__ float round_through(float v) { return v; }
template <> __device__ __forceinline__ float round_through<__half>(float v) { return __half2float(__float2half_rn(v)); }
template <> __device__ __forceinline__ float round_through<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// dy -> dy * act'(.) * gain with the clamp gate, from the saved OUTPUT y (act.cuh, G == 1; linear / relu / lrelu), branch-free.
// neg_slope = 1 / 0 / alpha for linear / relu / lrelu.  The kernel's test `y / gain > 0` is taken from the signs of y and gain (no
// division per element; they differ only where y / gain underflows to zero).
struct GateConsts { float neg_slope, gain, clamp; bool gain_pos, gain_neg, clamped; };
__device__ __forceinline__ GateConsts gate_consts(int act, float alpha, float gain, float clamp) {
    GateConsts k;
    k.neg_slope = act == PGPP_ACT_RELU ? 0.f : (act == PGPP_ACT_LRELU ? alpha : 1.f);
    k.gain = gain; k.clamp = clamp; k.gain_pos = gain > 0.f; k.gain_neg = gain < 0.f; k.clamped = clamp >= 0.f;
    return k;
}
__device__ __forceinline__ float act_gradient_from_output(float dy, float y, const GateConsts& k) {
    const bool pos = k.gain_pos ? y > 0.f : (k.gain_neg && y < 0.f);
    float v = (pos ? dy : dy * k.neg_slope) * k.gain;
    const bool inside = !k.clamped || (y > -k.clamp && y < k.clamp);
    return inside ? v : 0.f;
}

template <class T> struct RawVec4 { typedef uint2 type; };          // 4 consecutive pixels of a 16-bit tensor
template <> struct RawVec4<float> { typedef float4 type; };
template <> struct RawVec4<double> { typedef float4 type; };        // never loaded (VEC is false for 64-bit sources)
template <class T> __device__ __forceinline__ float raw_get(const typename RawVec4<T>::type& q, int k) {
    return (float)to_acc<T>(reinterpret_cast<const T*>(&q)[k]);
}
template <> __device__ __forceinline__ float raw_get<float>(const float4& q, int k) { return reinterpret_cast<const float*>(&q)[k]; }
template <> __device__ __forceinline__ float raw_get<double>(const float4& q, int k) { return reinterpret_cast<const float*>(&q)[k]; }

template <class T, bool VEC, bool GATE = false>
__global__ void __launch_bounds__(256) pack_nchw_kernel(PackArgs p, TileGeom g) {
    extern __shared__ uint4 sm_packets[];
    int xt, yt, ct, n;
    decode_tile_block(g, xt, yt, ct, n);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tw_mask = (1 << g.log_tw) - 1;
    const int x0 = xt << g.log_tw, y0 = yt * (128 >> g.log_tw), c0 = ct * 64;
    const int y = y0 + ((4 * lane) >> g.log_tw), x = x0 + ((4 * lane) & tw_mask);
    const T* src = (const T*)p.x + n * p.s_n + y * p.s_h + x;
    float v[8][4];
    if constexpr (VEC) {
        // vector loads: ALL loads of a channel group are issued before the first use - no branch, no conversion and no store between them
        // (a load per basic block, converted on arrival, is eight dependent round trips per thread; with the gate operand sixteen) -
        // then, for the gradient pass, dy * act'(y) * gain without a branch
        typedef typename RawVec4<T>::type Raw;
        constexpr int GROUP = (GATE && sizeof(T) == 4) ? 4 : 8;         // channels per load phase (registers)
        const GateConsts gk = gate_consts(p.act, p.alpha, p.gain, p.clamp);
        const T* gsrc = GATE ? (const T*)p.gate + n * p.s_n + y * p.s_h + x : nullptr;
        const float* scp = p.scale ? p.scale + (long long)n * p.c : nullptr;
        const bool px_ok = y < p.h && x < p.w;
        #pragma unroll
        for (int i0 = 0; i0 < 8; i0 += GROUP) {
            Raw rd[GROUP], rg[GATE ? GROUP : 1];
            float sc[GROUP];
            #pragma unroll
            for (int i = 0; i < GROUP; i++) {
                const int c = c0 + warp * 8 + i0 + i;
                const bool ok = px_ok && c < p.c;
                const long long off = ok ? c * p.s_c : 0;
                rd[i] = *reinterpret_cast<const Raw*>(ok ? src + off : (const T*)p.x);       // always a valid address; masked below
                if constexpr (GATE) rg[i] = *reinterpret_cast<const Raw*>(ok ? gsrc + off : (const T*)p.gate);
                sc[i] = (scp != nullptr && ok) ? scp[c] : 1.f;
            }
            #pragma unroll
            for (int i = 0; i < GROUP; i++) {
                const bool ok = px_ok && c0 + warp * 8 + i0 + i < p.c;
                #pragma unroll
                for (int k = 0; k < 4; k++) {
                    float val = raw_get<T>(rd[i], k) * sc[i];
                    if constexpr (GATE) val = round_through<T>(act_gradient_from_output(val, raw_get<T>(rg[i], k), gk));
                    v[i0 + i][k] = ok ? val : 0.f;
                }
            }
        }
    } else {
        // rows that are not 16-byte aligned (the odd-width blurred images of the down = 2 layers): element loads, same two phases
        constexpr int GROUP = sizeof(T) == 8 ? 2 : (GATE ? 4 : 8);
        const GateConsts gk = gate_consts(p.act, p.alpha, p.gain, p.clamp);
        const T* gsrc = GATE ? (const T*)p.gate + n * p.s_n + y * p.s_h + x : nullptr;
        const float* scp = p.scale ? p.scale + (long long)n * p.c : nullptr;
        #pragma unroll
        for (int i0 = 0; i0 < 8; i0 += GROUP) {
            T rd[GROUP][4], rg[GATE ? GROUP : 1][4];
            float sc[GROUP];
            #pragma unroll
            for (int i = 0; i < GROUP; i++) {
                const int c = c0 + warp * 8 + i0 + i;
                const bool row_ok = y < p.h && c < p.c;
                #pragma unroll
                for (int k = 0; k < 4; k++) {
                    const bool ok = row_ok && x + k < p.w;
                    const long long off = ok ? c * p.s_c + k : 0;
                    rd[i][k] = ok ? src[off] : *(const T*)p.x;          // always a valid address; masked below
                    if constexpr (GATE) rg[i][k] = ok ? gsrc[off] : *(const T*)p.gate;
                }
                sc[i] = (scp != nullptr && row_ok) ? scp[c] : 1.f;
            }
            #pragma unroll
            for (int i = 0; i < GROUP; i++) {
                const bool row_ok = y < p.h && c0 + warp * 8 + i0 + i < p.c;
                #pragma unroll
                for (int k = 0; k < 4; k++) {
                    float val = (float)to_acc<T>(rd[i][k]) * sc[i];
                    if constexpr (GATE) val = round_through<T>(act_gradient_from_output(val, (float)to_acc<T>(rg[i][k]), gk));
                    v[i0 + i][k] = (row_ok && x + k < p.w) ? val : 0.f;
                }
            }
        }
    }
    if constexpr (GATE) {
        if (p.csum) {
            // per-channel sums of the tile (pixels outside the image and channels beyond C hold zeros), after ALL loads were issued (a store
            // inside the loop would order the loads behind it).  8 values x 32 lanes, transposed butterfly: 9 shuffles instead of 40;
            // lane l ends with the total of channel 4 * bit4(l) + 2 * bit3(l) + bit2(l)
            float s8[8];
            #pragma unroll
            for (int i = 0; i < 8; i++) s8[i] = (v[i][0] + v[i][1]) + (v[i][2] + v[i][3]);
            float s4[4], s2[2];
            #pragma unroll
            for (int j = 0; j < 4; j++) {
                const bool hi = lane & 16;
                s4[j] = (hi ? s8[j + 4] : s8[j]) + __shfl_xor_sync(0xffffffffu, hi ? s8[j] : s8[j + 4], 16);
            }
            #pragma unroll
            for (int j = 0; j < 2; j++) {
                const bool hi = lane & 8;
                s2[j] = (hi ? s4[j + 2] : s4[j]) + __shfl_xor_sync(0xffffffffu, hi ? s4[j] : s4[j + 2], 8);
            }
            const bool hi = lane & 4;
            float s1 = (hi ? s2[1] : s2[0]) + __shfl_xor_sync(0xffffffffu, hi ? s2[0] : s2[1], 4);
            s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
            s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
            const int c = c0 + warp * 8 + ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
            if ((lane & 3) == 0 && c < p.c)
                p.csum[((long long)n * p.c + c) * ((long long)g.x_tiles * g.y_tiles) + (long long)yt * g.x_tiles + xt] = s1;
        }
    }
    emit_tile(v, sm_packets, p.parts, p.out, p.part_stride, n, p.h, p.w, y0, x0, g.log_tw, c0, p.c_pad, p.c_total, p.c_off, p.f16, p.e4m3);
}

// any strides (channels_last inputs are coalesced here): one thread per (pixel, channel)
template <class T>
__global__ void __launch_bounds__(256) pack_generic_kernel(PackArgs p, long long total) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(e % p.c_pad);
        long long r = e / p.c_pad;
        const int x = (int)(r % p.w); r /= p.w;
        const int y = (int)(r % p.h);
        const int n = (int)(r / p.h);
        float v = 0.f;
        if (c < p.c) {
            v = (float)to_acc<T>(((const T*)p.x)[n * p.s_n + c * p.s_c + y * p.s_h + x * p.s_w]);
            if (p.scale) v *= p.scale[n * p.c + c];
        }
        const long long idx = (e / p.c_pad) * p.c_total + p.c_off + c;
        if (p.e4m3) reinterpret_cast<uint8_t*>(p.out)[idx] = (uint8_t)__nv_cvt_float_to_fp8(v, __NV_SATFINITE, __NV_E4M3);
        else split_store(v, p.out + idx, p.part_stride, p.parts, p.f16);
    }
}

template <class T>
static int launch_pack(const PackArgs& p, cudaStream_t stream) {
    if (p.s_w == 1 && p.s_c != 1) {
        const TileGeom g = tile_geometry(p.h, p.w, p.c_pad);
        const long long blocks = (long long)g.x_tiles * g.y_tiles * g.c_tiles * p.n;
        PGPP_REQUIRE(blocks <= 2147483647LL, "activation tensor too large to pack");
        const size_t smem = (size_t)p.parts * 128 * 8 * sizeof(uint4);
        // 128-bit loads: rows 16-byte aligned and either W % 4 == 0 or a row pitch that covers the last (partial) group of 4
        const bool vec = sizeof(T) <= 4 && (p.w % 4 == 0 || p.s_h >= (p.w + 3) / 4 * 4) && p.s_c % 4 == 0 && p.s_h % 4 == 0 && p.s_n % 4 == 0 &&
                         ((uintptr_t)p.x & (4 * sizeof(T) - 1)) == 0;
        if (p.gate) {
            if (vec) pack_nchw_kernel<T, true, true><<<(unsigned)blocks, 256, smem, stream>>>(p, g);
            else pack_nchw_kernel<T, false, true><<<(unsigned)blocks, 256, smem, stream>>>(p, g);
        } else if (vec) pack_nchw_kernel<T, true><<<(unsigned)blocks, 256, smem, stream>>>(p, g);
        else pack_nchw_kernel<T, false><<<(unsigned)blocks, 256, smem, stream>>>(p, g);
    } else {
        PGPP_REQUIRE(!p.gate, "pgpp_pack_act_gradient needs pixel-contiguous (NCHW) tensors");
        const long long total = (long long)p.n * p.h * p.w * p.c_pad;
        long long blocks = (total + 255) / 256;
        const long long cap = (long long)sm_count() * occupancy_of(pack_generic_kernel<T>, 256, 0);
        if (blocks > cap) blocks = cap;
        pack_generic_kernel<T><<<(unsigned)blocks, 256, 0, stream>>>(p, total);
    }
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

struct Im2colArgs {
    const void* x; const float* scale; __nv_bfloat16* out;
    int n, c, h, w, hp, kw, r, pad_x, pad_y, parts;
    long long s_n, s_c, s_h, s_w, part_stride;
};

// One CTA per 128-pixel segment of one packed row: the r * C source rows it needs (with the kw - 1 halo) are staged in
// shared memory with coalesced reads, then 8 consecutive threads assemble the 128-byte channel row of a pixel through a
// channel -> (row, column offset) table and write one 128-bit store per part.
constexpr int kIm2colTile = 128;

template <class T>
__global__ void __launch_bounds__(256) im2col_kernel(Im2colArgs p, int x_tiles) {
    extern __shared__ float sm_rows[];                       // [r * c][kIm2colTile + kw - 1], then the table
    const int pitch = kIm2colTile + p.kw - 1;
    const int n_rows = p.r * p.c;
    int* lut = reinterpret_cast<int*>(sm_rows + n_rows * pitch);
    long long b = blockIdx.x;
    const int xt = (int)(b % x_tiles); b /= x_tiles;
    const int yy = (int)(b % p.hp);
    const int n = (int)(b / p.hp);
    const int x0 = xt * kIm2colTile;
    if (threadIdx.x < 64) {
        const int ch = threadIdx.x;
        int off = -1;
        if (ch < p.r * p.kw * p.c) {
            const int c = ch % p.c, t = ch / p.c;
            const int kx = t % p.kw, ry = t / p.kw;
            off = (ry * p.c + c) * pitch + kx;
        }
        lut[ch] = off;
    }
    for (int idx = threadIdx.x; idx < n_rows * pitch; idx += 256) {
        const int row = idx / pitch, col = idx - row * pitch;
        const int ry = row / p.c, c = row - ry * p.c;
        const int iy = yy - p.pad_y + ry, ix = x0 + col - p.pad_x;
        float val = 0.f;
        if (iy >= 0 && iy < p.h && ix >= 0 && ix < p.w) {
            val = (float)to_acc<T>(((const T*)p.x)[n * p.s_n + c * p.s_c + iy * p.s_h + ix * p.s_w]);
            if (p.scale) val *= p.scale[n * p.c + c];
        }
        sm_rows[idx] = val;
    }
    __syncthreads();
    #pragma unroll
    for (int it = 0; it < kIm2colTile * 8 / 256; it++) {
        const int item = it * 256 + threadIdx.x;
        const int px = item >> 3, cg = item & 7;
        if (x0 + px >= p.w) continue;
        float v[8];
        #pragma unroll
        for (int j = 0; j < 8; j++) {
            const int off = lut[cg * 8 + j];
            v[j] = off >= 0 ? sm_rows[off + px] : 0.f;
        }
        __nv_bfloat16* dst = p.out + (((long long)n * p.hp + yy) * p.w + x0 + px) * 64 + cg * 8;
        for (int part = 0; part < p.parts; part++) {
            __align__(16) __nv_bfloat16 qv[8];
            #pragma unroll
            for (int j = 0; j < 8; j++) { qv[j] = __float2bfloat16_rn(v[j]); v[j] -= __bfloat162float(qv[j]); }
            *reinterpret_cast<int4*>(dst + part * p.part_stride) = *reinterpret_cast<const int4*>(qv);
        }
    }
}

struct SpadeArgs {
    const float* x; const float* mean; const float* rstd; const float* gamma; const float* beta; __nv_bfloat16* out;
    int n, c, h, w, c_pad, parts; long long gb_stride_n, part_stride; float pre_gain;
};

// same 64-channel x 128-pixel transposing tile as pack_nchw_kernel, with the SPADE arithmetic applied on the way in
template <bool VEC>
__global__ void __launch_bounds__(256) spade_pack_kernel(SpadeArgs p, TileGeom g) {
    extern __shared__ uint4 sm_packets[];
    int xt, yt, ct, n;
    decode_tile_block(g, xt, yt, ct, n);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tw_mask = (1 << g.log_tw) - 1;
    const int x0 = xt << g.log_tw, y0 = yt * (128 >> g.log_tw), c0 = ct * 64;
    const int y = y0 + ((4 * lane) >> g.log_tw), x = x0 + ((4 * lane) & tw_mask);
    const long long plane = (long long)p.h * p.w;
    float v[8][4];
    #pragma unroll
    for (int i = 0; i < 8; i++) {
        const int c = c0 + warp * 8 + i;
        #pragma unroll
        for (int k = 0; k < 4; k++) v[i][k] = 0.f;
        if (c < p.c && y < p.h && x < p.w) {
            const long long off = (long long)c * plane + (long long)y * p.w + x;
            const float* xp = p.x + (long long)n * p.c * plane + off;
            const float* gp = p.gamma + n * p.gb_stride_n + off;
            const float* bp = p.beta + n * p.gb_stride_n + off;
            float xv[4] = {0.f, 0.f, 0.f, 0.f}, gv[4] = {0.f, 0.f, 0.f, 0.f}, bv[4] = {0.f, 0.f, 0.f, 0.f};
            if (VEC) {
                const float4 a = *reinterpret_cast<const float4*>(xp), b = *reinterpret_cast<const float4*>(gp), d = *reinterpret_cast<const float4*>(bp);
                xv[0] = a.x; xv[1] = a.y; xv[2] = a.z; xv[3] = a.w;
                gv[0] = b.x; gv[1] = b.y; gv[2] = b.z; gv[3] = b.w;
                bv[0] = d.x; bv[1] = d.y; bv[2] = d.z; bv[3] = d.w;
            } else {
                #pragma unroll
                for (int k = 0; k < 4; k++)
                    if (x + k < p.w) { xv[k] = xp[k]; gv[k] = gp[k]; bv[k] = bp[k]; }
            }
            const float mu = p.mean[n * p.c + c], rs = p.rstd[n * p.c + c];
            #pragma unroll
            for (int k = 0; k < 4; k++) {
                float r = fmaf((xv[k] - mu) * rs, 1.f + gv[k], bv[k]);
                if (p.pre_gain > 0.f) r = fmaxf(r, 0.f) * p.pre_gain;
                v[i][k] = (VEC || x + k < p.w) ? r : 0.f;
            }
        }
    }
    emit_tile(v, sm_packets, p.parts, p.out, p.part_stride, n, p.h, p.w, y0, x0, g.log_tw, c0, p.c_pad, p.c_pad, 0);
}

struct DirectArgs {
    const float* x; const float* w; const float* bias; float* out_nchw; __nv_bfloat16* out_packed;
    int n, c, h, wd, o, kh, kw, pad_y, pad_x, taps;
    int act; float alpha, gain, clamp, wscale;
    int c_pad, c_total, c_off, parts; long long part_stride;
};

// Direct (CUDA-core, exact fp32) convolution for inputs with very few taps per output (C * kh * kw <= 16: the 3x3 conv_mlp on the
// 1-channel parsing map, the 1x1 stem on the 5-channel pose map).  Such layers are bound by writing their 64..128-channel output;
// expanding the input to 64-channel operand rows for the tensor-core path costs 3-4x their roofline time.  Same 64-channel x
// 128-pixel tile and thread mapping as pack_nchw_kernel: a thread accumulates 8 output channels x 4 pixels from a sliding window
// of the input rows, weights are broadcast from shared memory, and the result leaves either as NCHW float32 (128-bit stores) or
// through emit_tile as the bf16 operand format of the next convolution, with bias / activation / gain / clamp applied.
constexpr int kDirectMaxTaps = 16;

// KH, CIN > 0: compile-time filter height / input channels (fully unrolled tap loops); 0: runtime values.
// The 8 channels of a thread are accumulated as 4 packed float32 pairs (FFMA2): the kernel is bound by instruction issue, not by
// its 2 GB of output (ncu: profiles/r02_ncu_small_kernels.md).
// ACT > 0: compile-time activation (pgpp_act; then the clamp is compile-time too: CLAMP) - the epilogue is a large part of the issue-bound kernel
template <int KW, int KH, int CIN, int ACT = 0, bool CLAMP = true>
__global__ void __launch_bounds__(256) conv_direct_kernel(DirectArgs p, TileGeom g, long long total_tiles) {
    extern __shared__ uint4 sm_packets[];
    __shared__ __align__(16) float sw[kDirectMaxTaps * 64];      // [tap][channel of the 64-channel tile]
    __shared__ float sb[64];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tw_mask = (1 << g.log_tw) - 1;
    const long long plane = (long long)p.h * p.wd;
    const int kh = KH ? KH : p.kh, cin = CIN ? CIN : p.c;
    int loaded_ct = -1;
    // persistent over the tiles: the weights of a 64-channel tile are staged once (the channel tile is the slowest tile index)
    for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        unsigned b = (unsigned)tile;
        const int xt = divmod_u32(b, (unsigned)g.x_tiles);
        const int yt = divmod_u32(b, (unsigned)g.y_tiles);
        const int n = divmod_u32(b, (unsigned)p.n);
        const int ct = (int)b;
        const int x0 = xt << g.log_tw, y0 = yt * (128 >> g.log_tw), c0 = ct * 64;
        __syncthreads();                        // previous tile's packets fully written out; weights no longer in use
        if (ct != loaded_ct) {
            for (int i = threadIdx.x; i < 64 * p.taps; i += 256) {
                const int tap = i >> 6, oc = c0 + (i & 63);
                sw[i] = oc < p.o ? p.w[(long long)oc * p.taps + tap] * p.wscale : 0.f;
            }
            if (threadIdx.x < 64) sb[threadIdx.x] = (p.bias && c0 + threadIdx.x < p.o) ? p.bias[c0 + threadIdx.x] : 0.f;
            loaded_ct = ct;
            __syncthreads();
        }
        const int y = y0 + ((4 * lane) >> g.log_tw), x = x0 + ((4 * lane) & tw_mask);
        const int tile_rows = 128 >> g.log_tw, tile_w = 1 << g.log_tw;
        const bool interior = y0 - p.pad_y >= 0 && y0 + tile_rows - 1 + (kh - 1 - p.pad_y) < p.h && x0 - KW / 2 >= 0 && x0 + tile_w - 1 + KW / 2 < p.wd;
        f32x2 acc[4][4];                        // [channel pair][pixel]
        #pragma unroll
        for (int i = 0; i < 4; i++)
            #pragma unroll
            for (int k = 0; k < 4; k++) acc[i][k] = 0ull;
        if (y < p.h && x < p.wd) {
            const float* src = p.x + (long long)n * p.c * plane;
            const float* wrow = sw + warp * 8;
            #pragma unroll
            for (int ci = 0; ci < (CIN ? CIN : kDirectMaxTaps); ci++) {
                if (ci >= cin) break;
                #pragma unroll
                for (int ky = 0; ky < (KH ? KH : 1); ky++) {
                    for (int kyr = ky; kyr < kh; kyr += (KH ? KH : 1)) {           // KH == 0: runtime loop over the filter rows
                        const int iy = y + kyr - p.pad_y;
                        const bool row_ok = iy >= 0 && iy < p.h;
                        const float* row = src + (long long)ci * plane + (long long)iy * p.wd;
                        f32x2 in2[4 + KW - 1];
                        if (interior) {         // the tile's halo lies inside the image: no per-element bounds tests
                            #pragma unroll
                            for (int j = 0; j < 4 + KW - 1; j++) {
                                const float v = __ldg(row + x + j - KW / 2);
                                in2[j] = pack2(v, v);
                            }
                        } else {
                            #pragma unroll
                            for (int j = 0; j < 4 + KW - 1; j++) {
                                const int ix = x + j - KW / 2;
                                const float v = (row_ok && ix >= 0 && ix < p.wd) ? __ldg(row + ix) : 0.f;
                                in2[j] = pack2(v, v);
                            }
                        }
                        const float* wt = wrow + ((ci * kh + kyr) * KW) * 64;
                        #pragma unroll
                        for (int kx = 0; kx < KW; kx++) {
                            const float4 wa = *reinterpret_cast<const float4*>(wt + kx * 64);
                            const float4 wb = *reinterpret_cast<const float4*>(wt + kx * 64 + 4);
                            const f32x2 w2[4] = {pack2(wa.x, wa.y), pack2(wa.z, wa.w), pack2(wb.x, wb.y), pack2(wb.z, wb.w)};
                            #pragma unroll
                            for (int i = 0; i < 4; i++)
                                #pragma unroll
                                for (int k = 0; k < 4; k++) ffma2(acc[i][k], w2[i], in2[kx + k]);
                        }
                        if (KH) break;
                    }
                }
            }
        }
        float v[8][4];
        #pragma unroll
        for (int i = 0; i < 4; i++)
            #pragma unroll
            for (int k = 0; k < 4; k++) {
                v[2 * i][k] = __uint_as_float((uint32_t)acc[i][k]);
                v[2 * i + 1][k] = __uint_as_float((uint32_t)(acc[i][k] >> 32));
            }
        #pragma unroll
        for (int i = 0; i < 8; i++) {
            const float bb = sb[warp * 8 + i];
            #pragma unroll
            for (int k = 0; k < 4; k++) {
                float r = v[i][k] + bb;
                const int act = ACT ? ACT : p.act;
                if (act == PGPP_ACT_RELU) r = fmaxf(r, 0.f);
                else if (act == PGPP_ACT_LRELU) r = r > 0.f ? r : r * p.alpha;
                r *= p.gain;
                if ((ACT ? CLAMP : true) && p.clamp >= 0.f) r = fminf(fmaxf(r, -p.clamp), p.clamp);
                v[i][k] = r;
            }
        }
        if (p.out_packed) {
            emit_tile(v, sm_packets, p.parts, p.out_packed, p.part_stride, n, p.h, p.wd, y0, x0, g.log_tw, c0, p.c_pad, p.c_total, p.c_off);
        } else if (y < p.h && x < p.wd) {
            #pragma unroll
            for (int i = 0; i < 8; i++) {
                const int oc = c0 + warp * 8 + i;
                if (oc >= p.o) continue;
                float* dst = p.out_nchw + ((long long)n * p.o + oc) * plane + (long long)y * p.wd + x;
                if (x + 3 < p.wd && (p.wd & 3) == 0) __stcs(reinterpret_cast<float4*>(dst), make_float4(v[i][0], v[i][1], v[i][2], v[i][3]));
                else {
                    #pragma unroll
                    for (int k = 0; k < 4; k++) if (x + k < p.wd) dst[k] = v[i][k];
                }
            }
        }
    }
}

struct FirPackArgs {
    const float* x; __nv_bfloat16* out;
    int n, c, ih, iw, oh, ow, padx0, pady0, c_pad, parts;
    long long xs_n, xs_c, xs_h, part_stride;
    float k[4][4];              // taps, flipped / zero-padded to 4 x 4 and scaled by gain on the host
};

// FIR blur (up = down = 1, filter up to 4 x 4) of an NCHW float32 tensor written directly in the operand format: the
// "blur, then strided convolution" pair of conv2d_resample.py:119-122 without the float32 intermediate.  A CTA owns 64 channels
// of a 32 x 4 block of output pixels: the 35 x 7 input halo of every channel is staged in shared memory with coalesced loads,
// thread (warp w, lane l) filters channels 8w..8w+7 of 4 consecutive pixels from it, and the packets leave through emit_tile
// (which reuses the staging buffer).
constexpr int kFirTw = 32, kFirTh = 4, kFirPitch = 36, kFirRows = kFirTh + 3;

__global__ void __launch_bounds__(256) fir_pack_kernel(FirPackArgs p, int x_tiles, int y_tiles, int c_tiles) {
    extern __shared__ uint4 sm_packets[];
    float* stage = reinterpret_cast<float*>(sm_packets);                 // [64][kFirRows][kFirPitch]
    long long b = blockIdx.x;
    const int xt = (int)(b % x_tiles); b /= x_tiles;
    const int ct = (int)(b % c_tiles); b /= c_tiles;
    const int yt = (int)(b % y_tiles);
    const int n = (int)(b / y_tiles);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = xt * kFirTw, y0 = yt * kFirTh, c0 = ct * 64;
    const int ix0 = x0 - p.padx0, iy0 = y0 - p.pady0;
    // stage: one (channel, row) of 35 floats per warp and step, lanes along x; 8 steps are issued back to back so that 8..16 loads
    // per lane are in flight before the first shared-memory store
    for (int i0 = 0; i0 < 64 * kFirRows / 8; i0 += 8) {
        float va[8], vb[8];
        #pragma unroll
        for (int u = 0; u < 8; u++) {
            const int cr = warp + 8 * (i0 + u);
            const int ch = cr / kFirRows, r = cr - ch * kFirRows;
            const int c = c0 + ch, iy = iy0 + r;
            const bool ok = c < p.c && iy >= 0 && iy < p.ih;
            const float* row = p.x + n * p.xs_n + (long long)c * p.xs_c + (long long)iy * p.xs_h;
            const int ixa = ix0 + lane, ixb = ix0 + lane + 32;
            va[u] = (ok && ixa >= 0 && ixa < p.iw) ? __ldg(row + ixa) : 0.f;
            vb[u] = (ok && lane < kFirTw + 3 - 32 && ixb >= 0 && ixb < p.iw) ? __ldg(row + ixb) : 0.f;
        }
        #pragma unroll
        for (int u = 0; u < 8; u++) {
            const int cr = warp + 8 * (i0 + u);
            float* dst = stage + cr * kFirPitch;
            dst[lane] = va[u];
            if (lane < kFirPitch - 32) dst[lane + 32] = vb[u];
        }
    }
    __syncthreads();
    const int r = lane >> 3, cx = (lane & 7) * 4;                   // pixel row of the tile, first of the 4 columns
    float v[8][4];
    #pragma unroll
    for (int i = 0; i < 8; i++) {
        const float* src = stage + ((warp * 8 + i) * kFirRows + r) * kFirPitch + cx;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        #pragma unroll
        for (int jy = 0; jy < 4; jy++) {
            // 8 consecutive staged floats as two 128-bit loads (cx and the row pitch are multiples of 4): a quarter warp reads
            // 128 contiguous bytes, no bank conflicts
            const float4 lo = *reinterpret_cast<const float4*>(src + jy * kFirPitch);
            const float4 hi = *reinterpret_cast<const float4*>(src + jy * kFirPitch + 4);
            const float in[7] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z};
            #pragma unroll
            for (int jx = 0; jx < 4; jx++)
                #pragma unroll
                for (int k = 0; k < 4; k++) acc[k] = fmaf(in[k + jx], p.k[jy][jx], acc[k]);
        }
        #pragma unroll
        for (int k = 0; k < 4; k++) v[i][k] = acc[k];
    }
    __syncthreads();                                                // staging buffer becomes the packet buffer
    emit_tile(v, sm_packets, p.parts, p.out, p.part_stride, n, p.oh, p.ow, y0, x0, 5, c0, p.c_pad, p.c_pad, 0);
}

struct MixArgs {
    const float* x[2]; const float* m[2]; const float* a[2]; const float* b[2]; __nv_bfloat16* out;
    int n, c, h, w, c_pad, parts, terms; long long part_stride;
};

// v[n,c,p] = sum_t x_t[n,c,p] * a_t[n,p] + m_t[n,c] * b_t[n,p]  ->  packed operand (same transposing tile as pack_nchw_kernel).
// The masked feature composition of SynthesisNetworkFull_v18 (networks.py:2253-2276, 2307-2315): per branch
// x * (1 - res_mask) + mean * res_mask, times the branch's 256 x 256 mask, summed over the upper / lower branches.
template <bool VEC>
__global__ void __launch_bounds__(256) mix_pack_kernel(MixArgs p, TileGeom g) {
    extern __shared__ uint4 sm_packets[];
    int xt, yt, ct, n;
    decode_tile_block(g, xt, yt, ct, n);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tw_mask = (1 << g.log_tw) - 1;
    const int x0 = xt << g.log_tw, y0 = yt * (128 >> g.log_tw), c0 = ct * 64;
    const int y = y0 + ((4 * lane) >> g.log_tw), x = x0 + ((4 * lane) & tw_mask);
    const long long plane = (long long)p.h * p.w;
    const long long pix = (long long)y * p.w + x;
    float v[8][4];
    #pragma unroll
    for (int i = 0; i < 8; i++)
        #pragma unroll
        for (int k = 0; k < 4; k++) v[i][k] = 0.f;
    if (y < p.h && x < p.w) {
        for (int t = 0; t < p.terms; t++) {
            float av[4] = {0.f, 0.f, 0.f, 0.f}, bv[4] = {0.f, 0.f, 0.f, 0.f};
            const float* ap = p.a[t] + n * plane + pix;
            const float* bp = p.b[t] + n * plane + pix;
            if (VEC) {
                const float4 qa = *reinterpret_cast<const float4*>(ap), qb = *reinterpret_cast<const float4*>(bp);
                av[0] = qa.x; av[1] = qa.y; av[2] = qa.z; av[3] = qa.w;
                bv[0] = qb.x; bv[1] = qb.y; bv[2] = qb.z; bv[3] = qb.w;
            } else {
                #pragma unroll
                for (int k = 0; k < 4; k++) if (x + k < p.w) { av[k] = ap[k]; bv[k] = bp[k]; }
            }
            #pragma unroll
            for (int i = 0; i < 8; i++) {
                const int c = c0 + warp * 8 + i;
                if (c >= p.c) continue;
                const float* xp = p.x[t] + ((long long)n * p.c + c) * plane + pix;
                float xv[4] = {0.f, 0.f, 0.f, 0.f};
                if (VEC) {
                    const float4 q = *reinterpret_cast<const float4*>(xp);
                    xv[0] = q.x; xv[1] = q.y; xv[2] = q.z; xv[3] = q.w;
                } else {
                    #pragma unroll
                    for (int k = 0; k < 4; k++) if (x + k < p.w) xv[k] = xp[k];
                }
                const float mv = p.m[t][n * p.c + c];
                #pragma unroll
                for (int k = 0; k < 4; k++) v[i][k] += __fadd_rn(__fmul_rn(xv[k], av[k]), __fmul_rn(mv, bv[k]));
            }
        }
    }
    emit_tile(v, sm_packets, p.parts, p.out, p.part_stride, n, p.h, p.w, y0, x0, g.log_tw, c0, p.c_pad, p.c_pad, 0);
}

// one CTA per output channel: W2[i] = sum_t w[o,i,t]^2 in shared memory, then one warp per sample
__global__ void __launch_bounds__(256) demod_kernel(const float* __restrict__ w, const float* __restrict__ s,
                                                    float* __restrict__ d, int n, int o, int ic, int taps, float eps) {
    extern __shared__ float w2[];
    const int oc = blockIdx.x;
    const float* wp = w + (long long)oc * ic * taps;
    for (int i = threadIdx.x; i < ic; i += blockDim.x) {
        float a = 0.f;
        for (int t = 0; t < taps; t++) { const float v = wp[i * taps + t]; a = fmaf(v, v, a); }
        w2[i] = a;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = warp; b < n; b += blockDim.x / 32) {
        float a = 0.f;
        for (int i = lane; i < ic; i += 32) { const float sv = s[(long long)b * ic + i]; a = fmaf(sv * sv, w2[i], a); }
        #pragma unroll
        for (int m = 16; m > 0; m >>= 1) a += __shfl_xor_sync(0xffffffffu, a, m);
        if (lane == 0) d[(long long)b * o + oc] = rsqrtf(a + eps);
    }
}

} // namespace pgpp

extern "C" int pgpp_pack_activations(const void* x, const int64_t size[4], const int64_t stride[4], int dtype,
                                     const float* scale, void* out, int c_pad, int parts, void* stream) {
    return pgpp_pack_activations_slice(x, size, stride, dtype, scale, out, c_pad, c_pad, 0, parts, stream);
}

namespace pgpp {
__global__ void __launch_bounds__(256) modulate_weights_kernel(const float* __restrict__ master, const float* __restrict__ s,
                                                               __nv_bfloat16* __restrict__ out, long long rows, int c_pad, int c_in,
                                                               int parts, long long per_sample_part) {
    // one thread per 8 consecutive channels of one (sample, row): 128-bit stores per part
    const int groups = c_pad / 8;
    const long long total = rows * groups;
    const int n = blockIdx.y;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long row = e / groups;
        const int c0 = (int)(e - row * groups) * 8;
        float v[8];
        #pragma unroll
        for (int j = 0; j < 8; j++) {
            const int c = c0 + j;
            v[j] = c < c_in ? master[row * c_pad + c] * s[(long long)n * c_in + c] : 0.f;
        }
        __nv_bfloat16* dst = out + (long long)n * parts * per_sample_part + row * c_pad + c0;
        for (int part = 0; part < parts; part++) {
            __align__(16) __nv_bfloat16 q[8];
            #pragma unroll
            for (int j = 0; j < 8; j++) { q[j] = __float2bfloat16_rn(v[j]); v[j] -= __bfloat162float(q[j]); }
            *reinterpret_cast<int4*>(dst + part * per_sample_part) = *reinterpret_cast<const int4*>(q);
        }
    }
}
} // namespace pgpp

extern "C" int pgpp_modulate_weights(const float* master, const float* s, void* out, int n, int64_t rows, int c_pad, int c_in,
                                     int parts, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(master && s && out, "master, s and out must be device pointers");
    PGPP_REQUIRE(n >= 1 && n <= 65535 && rows >= 1 && c_pad % 16 == 0 && c_in >= 1 && c_in <= c_pad && parts >= 1 && parts <= 3, "bad modulate_weights arguments");
    const long long total = rows * (c_pad / 8);
    long long blocks = (total + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    modulate_weights_kernel<<<dim3((unsigned)blocks, (unsigned)n), 256, 0, (cudaStream_t)stream>>>(master, s, (__nv_bfloat16*)out, rows, c_pad, c_in,
                                                                                                  parts, rows * c_pad);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

namespace pgpp {
struct PackGate { const void* y; int act; float alpha, gain, clamp; float* csum; };
static int pack_slice(const void* x, const int64_t size[4], const int64_t stride[4], int dtype, const float* scale, void* out,
                      int c_pad, int c_total, int c_off, int parts, int f16, void* stream, const PackGate* gate = nullptr, int e4m3 = 0);
}

extern "C" int pgpp_pack_act_gradient_tiles(int h, int w) {
    const pgpp::TileGeom g = pgpp::tile_geometry(h, w, 64);
    return g.x_tiles * g.y_tiles;
}

extern "C" int pgpp_pack_act_gradient(const void* dy, const void* y, const int64_t size[4], const int64_t stride[4], int dtype,
                                      int act_fn, float alpha, float gain, float clamp, void* out, int c_pad, int parts, int f16,
                                      float* csum, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(dy && y, "dy and y must be device pointers");
    PGPP_REQUIRE(act_fn == PGPP_ACT_LINEAR || act_fn == PGPP_ACT_RELU || act_fn == PGPP_ACT_LRELU,
                 "pgpp_pack_act_gradient: the activation's derivative must depend on its output only (linear, relu, lrelu)");
    PGPP_REQUIRE(dtype == PGPP_F32 || dtype == PGPP_F16 || dtype == PGPP_BF16, "pgpp_pack_act_gradient: dtype must be f32, f16 or bf16");
    PGPP_REQUIRE(stride[3] == 1 && stride[1] != 1, "pgpp_pack_act_gradient needs pixel-contiguous (NCHW) tensors");
    PGPP_REQUIRE(!f16 || parts == 1, "fp16 operands are a single part");
    PackGate gate{y, act_fn, alpha, gain, clamp, csum};
    return pack_slice(dy, size, stride, dtype, nullptr, out, c_pad, c_pad, 0, parts, f16, stream, &gate);
}

extern "C" int pgpp_pack_activations_slice(const void* x, const int64_t size[4], const int64_t stride[4], int dtype,
                                           const float* scale, void* out, int c_pad, int c_total, int c_off, int parts, void* stream) {
    return pgpp::pack_slice(x, size, stride, dtype, scale, out, c_pad, c_total, c_off, parts, 0, stream);
}

extern "C" int pgpp_pack_activations_f16(const void* x, const int64_t size[4], const int64_t stride[4], int dtype,
                                         const float* scale, void* out, int c_pad, int c_total, int c_off, void* stream) {
    return pgpp::pack_slice(x, size, stride, dtype, scale, out, c_pad, c_total, c_off, 1, 1, stream);
}

extern "C" int pgpp_pack_activations_e4m3(const void* x, const int64_t size[4], const int64_t stride[4], int dtype,
                                          const float* scale, void* out, int c_pad, int c_total, int c_off, void* stream) {
    return pgpp::pack_slice(x, size, stride, dtype, scale, out, c_pad, c_total, c_off, 1, 0, stream, nullptr, 1);
}

int pgpp::pack_slice(const void* x, const int64_t size[4], const int64_t stride[4], int dtype, const float* scale, void* out,
                     int c_pad, int c_total, int c_off, int parts, int f16, void* stream, const PackGate* gate, int e4m3) {
    PGPP_REQUIRE(x && out, "x and out must be device pointers");
    PGPP_REQUIRE(parts >= 1 && parts <= 3, "parts must be 1, 2 or 3");
    PGPP_REQUIRE(c_pad >= size[1] && c_pad % 16 == 0, "c_pad must be a multiple of 16 and >= C");
    PGPP_REQUIRE(c_total >= c_off + c_pad && c_total % 8 == 0 && c_off % 8 == 0 && c_off >= 0, "bad destination channel slice");
    PackArgs p;
    p.c_total = c_total; p.c_off = c_off;
    p.x = x; p.scale = scale; p.out = (__nv_bfloat16*)out;
    p.n = (int)size[0]; p.c = (int)size[1]; p.h = (int)size[2]; p.w = (int)size[3];
    p.c_pad = c_pad; p.parts = parts; p.f16 = f16; p.e4m3 = e4m3;
    p.s_n = stride[0]; p.s_c = stride[1]; p.s_h = stride[2]; p.s_w = stride[3];
    p.part_stride = (long long)p.n * p.h * p.w * c_total;
    p.gate = nullptr; p.act = PGPP_ACT_LINEAR; p.alpha = 0.f; p.gain = 1.f; p.clamp = -1.f; p.csum = nullptr;
    if (gate) { p.gate = gate->y; p.act = gate->act; p.alpha = gate->alpha; p.gain = gate->gain; p.clamp = gate->clamp; p.csum = gate->csum; }
    if (p.part_stride == 0) return PGPP_OK;
    cudaStream_t s = (cudaStream_t)stream;
    switch (dtype) {
        case PGPP_F32:  return launch_pack<float>(p, s);
        case PGPP_F16:  return launch_pack<__half>(p, s);
        case PGPP_BF16: return launch_pack<__nv_bfloat16>(p, s);
        case PGPP_F64:  return launch_pack<double>(p, s);
    }
    set_error("unsupported dtype %d", dtype);
    return PGPP_ERR_UNSUPPORTED;
}

extern "C" int pgpp_pack_im2col(const void* x, const int64_t size[4], const int64_t stride[4], int dtype, const float* scale,
                                void* out, int kw, int r, int pad_x, int pad_y, int parts, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(x && out, "x and out must be device pointers");
    PGPP_REQUIRE(parts >= 1 && parts <= 3 && kw >= 1 && r >= 1 && pad_x >= 0 && pad_y >= 0, "bad im2col arguments");
    PGPP_REQUIRE((long long)r * kw * size[1] <= 64, "im2col packing needs r*kw*C <= 64");
    Im2colArgs p;
    p.x = x; p.scale = scale; p.out = (__nv_bfloat16*)out;
    p.n = (int)size[0]; p.c = (int)size[1]; p.h = (int)size[2]; p.w = (int)size[3]; p.hp = p.h + pad_y;
    p.kw = kw; p.r = r; p.pad_x = pad_x; p.pad_y = pad_y; p.parts = parts;
    p.s_n = stride[0]; p.s_c = stride[1]; p.s_h = stride[2]; p.s_w = stride[3];
    p.part_stride = (long long)p.n * p.hp * p.w * 64;
    if ((long long)p.n * p.hp * p.w == 0) return PGPP_OK;
    const int x_tiles = (p.w + kIm2colTile - 1) / kIm2colTile;
    const long long blocks = (long long)x_tiles * p.hp * p.n;
    PGPP_REQUIRE(blocks <= 2147483647LL, "tensor too large");
    const size_t smem = sizeof(float) * (size_t)(r * p.c) * (kIm2colTile + kw - 1) + 64 * sizeof(int);
    PGPP_REQUIRE(smem <= 48 * 1024, "im2col row staging does not fit shared memory");
    cudaStream_t s = (cudaStream_t)stream;
#define PGPP_IM2COL(T) im2col_kernel<T><<<(unsigned)blocks, 256, smem, s>>>(p, x_tiles);
    switch (dtype) {
        case PGPP_F32:  PGPP_IM2COL(float) break;
        case PGPP_F16:  PGPP_IM2COL(__half) break;
        case PGPP_BF16: PGPP_IM2COL(__nv_bfloat16) break;
        case PGPP_F64:  PGPP_IM2COL(double) break;
        default: set_error("unsupported dtype %d", dtype); return PGPP_ERR_UNSUPPORTED;
    }
#undef PGPP_IM2COL
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

extern "C" int pgpp_spade_modulate_pack(const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
                                        int64_t gb_stride_n, void* out, int n, int c, int h, int w, int c_pad, int parts, float pre_gain, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(x && mean && rstd && gamma && beta && out, "null pointer");
    PGPP_REQUIRE(n >= 1 && c >= 1 && h >= 1 && w >= 1 && c_pad >= c && c_pad % 16 == 0 && parts >= 1 && parts <= 3, "bad spade_modulate_pack arguments");
    SpadeArgs p;
    p.x = x; p.mean = mean; p.rstd = rstd; p.gamma = gamma; p.beta = beta; p.out = (__nv_bfloat16*)out;
    p.n = n; p.c = c; p.h = h; p.w = w; p.c_pad = c_pad; p.parts = parts; p.gb_stride_n = gb_stride_n;
    p.part_stride = (long long)n * h * w * c_pad; p.pre_gain = pre_gain;
    const TileGeom g = tile_geometry(h, w, c_pad);
    const long long blocks = (long long)g.x_tiles * g.y_tiles * g.c_tiles * n;
    PGPP_REQUIRE(blocks <= 2147483647LL, "tensor too large");
    const size_t smem = (size_t)parts * 128 * 8 * sizeof(uint4);
    const bool vec = w % 4 == 0 && gb_stride_n % 4 == 0 && (((uintptr_t)x | (uintptr_t)gamma | (uintptr_t)beta) & 15) == 0;
    if (vec) spade_pack_kernel<true><<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(p, g);
    else spade_pack_kernel<false><<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(p, g);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

extern "C" int pgpp_modconv_demod_coefs(const float* w, const float* s, float* d, int n, int o, int i, int taps,
                                        float eps, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(w && s && d, "w, s and d must be device pointers");
    PGPP_REQUIRE(n >= 1 && o >= 1 && i >= 1 && taps >= 1, "empty problem");
    PGPP_REQUIRE((size_t)i * sizeof(float) <= 200 * 1024, "too many input channels");
    const size_t smem = (size_t)i * sizeof(float);
    if (smem > 48 * 1024)
        PGPP_CUDA_OK(cudaFuncSetAttribute(demod_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    demod_kernel<<<o, 256, smem, (cudaStream_t)stream>>>(w, s, d, n, o, i, taps, eps);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

extern "C" int pgpp_mix_pack(const float* x1, const float* m1, const float* a1, const float* b1, const float* x2, const float* m2,
                             const float* a2, const float* b2, void* out, int n, int c, int h, int w, int c_pad, int parts, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(x1 && m1 && a1 && b1 && out, "null pointer");
    PGPP_REQUIRE((x2 == nullptr) == (m2 == nullptr) && (x2 == nullptr) == (a2 == nullptr) && (x2 == nullptr) == (b2 == nullptr),
                 "the second term needs all of x2, m2, a2, b2");
    PGPP_REQUIRE(n >= 1 && c >= 1 && h >= 1 && w >= 1 && c_pad >= c && c_pad % 16 == 0 && parts >= 1 && parts <= 3, "bad mix_pack arguments");
    MixArgs p;
    p.x[0] = x1; p.m[0] = m1; p.a[0] = a1; p.b[0] = b1; p.x[1] = x2; p.m[1] = m2; p.a[1] = a2; p.b[1] = b2;
    p.terms = x2 ? 2 : 1;
    p.out = (__nv_bfloat16*)out; p.n = n; p.c = c; p.h = h; p.w = w; p.c_pad = c_pad; p.parts = parts;
    p.part_stride = (long long)n * h * w * c_pad;
    const TileGeom g = tile_geometry(h, w, c_pad);
    const long long blocks = (long long)g.x_tiles * g.y_tiles * g.c_tiles * n;
    PGPP_REQUIRE(blocks <= 2147483647LL, "tensor too large");
    const size_t smem = (size_t)parts * 128 * 8 * sizeof(uint4);
    const uintptr_t al = (uintptr_t)x1 | (uintptr_t)a1 | (uintptr_t)b1 | (uintptr_t)x2 | (uintptr_t)a2 | (uintptr_t)b2;
    const bool vec = w % 4 == 0 && (al & 15) == 0;
    if (vec) mix_pack_kernel<true><<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(p, g);
    else mix_pack_kernel<false><<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(p, g);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

extern "C" int pgpp_conv2d_direct(const float* x, const float* w, const float* bias, int n, int c, int h, int wd, int o, int kh, int kw,
                                  int pad_y, int pad_x, float wscale, int act_fn, float alpha, float gain, float clamp,
                                  float* out_nchw, void* out_packed, int c_total, int c_off, int parts, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(x && w && (out_nchw != nullptr) != (out_packed != nullptr), "x, w and exactly one of out_nchw / out_packed are required");
    PGPP_REQUIRE(n >= 1 && c >= 1 && h >= 1 && wd >= 1 && o >= 1, "empty problem");
    PGPP_REQUIRE(kh >= 1 && (kw == 1 || kw == 3) && c * kh * kw <= kDirectMaxTaps, "direct convolution: C * kh * kw <= 16 and kw = 1 or 3");
    PGPP_REQUIRE(2 * pad_y == kh - 1 && 2 * pad_x == kw - 1, "direct convolution: 'same' padding only");
    PGPP_REQUIRE(act_fn == PGPP_ACT_LINEAR || act_fn == PGPP_ACT_RELU || act_fn == PGPP_ACT_LRELU, "direct convolution: linear, relu or lrelu");
    DirectArgs p;
    p.x = x; p.w = w; p.bias = bias; p.out_nchw = out_nchw; p.out_packed = (__nv_bfloat16*)out_packed;
    p.n = n; p.c = c; p.h = h; p.wd = wd; p.o = o; p.kh = kh; p.kw = kw; p.pad_y = pad_y; p.pad_x = pad_x; p.taps = c * kh * kw;
    p.act = act_fn; p.alpha = alpha; p.gain = gain; p.clamp = clamp; p.wscale = wscale;
    p.parts = parts; p.c_total = c_total; p.c_off = c_off; p.c_pad = (o + 7) / 8 * 8;
    p.part_stride = (long long)n * h * wd * c_total;
    size_t smem = 0;
    if (out_packed) {
        PGPP_REQUIRE(parts >= 1 && parts <= 3 && o % 8 == 0 && c_off % 8 == 0 && c_total % 8 == 0 && c_total >= c_off + o &&
                     ((uintptr_t)out_packed & 15) == 0, "bad packed destination");
        smem = (size_t)parts * 128 * 8 * sizeof(uint4);
    }
    TileGeom g = tile_geometry(h, wd, (o + 63) / 64 * 64);
    const long long total = (long long)g.x_tiles * g.y_tiles * g.c_tiles * n;
    PGPP_REQUIRE(total < (1ll << 31), "direct convolution: too many tiles");
    auto launch = [&](auto kernel) -> int {
        if (smem > 40 * 1024) PGPP_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        long long blocks = total;
        const long long cap = (long long)sm_count() * occupancy_of(kernel, 256, smem);
        if (blocks > cap) blocks = cap;
        kernel<<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(p, g, total);
        return PGPP_OK;
    };
    const int rc = (kw == 3 && kh == 3 && c == 1 && act_fn == PGPP_ACT_RELU && clamp < 0.f) ? launch(conv_direct_kernel<3, 3, 1, PGPP_ACT_RELU, false>)
                 : (kw == 3 && kh == 3 && c == 1) ? launch(conv_direct_kernel<3, 3, 1>)
                 : (kw == 1 && kh == 1) ? launch(conv_direct_kernel<1, 1, 0>)
                 : kw == 1 ? launch(conv_direct_kernel<1, 0, 0>) : launch(conv_direct_kernel<3, 0, 0>);
    if (rc != PGPP_OK) return rc;
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

extern "C" int pgpp_fir_pack(const float* x, const int64_t size[4], const int64_t stride[4], const float* f_host, int fw, int fh,
                             int padx0, int padx1, int pady0, int pady1, int flip, float gain, void* out, int c_pad, int parts, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(x && f_host && out, "x, f and out must be given (f is a HOST array of fh * fw taps)");
    PGPP_REQUIRE(fw >= 1 && fw <= 4 && fh >= 1 && fh <= 4, "fir_pack: filter up to 4 x 4");
    PGPP_REQUIRE(stride[3] == 1, "fir_pack: x must have unit stride along W");
    PGPP_REQUIRE(parts >= 1 && parts <= 3 && c_pad >= size[1] && c_pad % 8 == 0, "bad fir_pack destination");
    FirPackArgs p;
    p.x = x; p.out = (__nv_bfloat16*)out;
    p.n = (int)size[0]; p.c = (int)size[1]; p.ih = (int)size[2]; p.iw = (int)size[3];
    p.ow = p.iw + padx0 + padx1 - fw + 1; p.oh = p.ih + pady0 + pady1 - fh + 1;
    PGPP_REQUIRE(p.ow >= 1 && p.oh >= 1, "output must be at least 1x1");
    p.padx0 = padx0; p.pady0 = pady0; p.c_pad = c_pad; p.parts = parts;
    p.xs_n = stride[0]; p.xs_c = stride[1]; p.xs_h = stride[2];
    p.part_stride = (long long)p.n * p.oh * p.ow * c_pad;
    for (int jy = 0; jy < 4; jy++)
        for (int jx = 0; jx < 4; jx++) {
            float v = 0.f;
            if (jy < fh && jx < fw) {
                const int sy = flip ? jy : fh - 1 - jy, sx = flip ? jx : fw - 1 - jx;     // upfirdn2d correlates with the flipped filter
                v = f_host[sy * fw + sx] * gain;
            }
            p.k[jy][jx] = v;
        }
    if (p.n == 0 || p.c == 0) return PGPP_OK;
    const int x_tiles = (p.ow + kFirTw - 1) / kFirTw, y_tiles = (p.oh + kFirTh - 1) / kFirTh, c_tiles = (c_pad + 63) / 64;
    const long long blocks = (long long)x_tiles * y_tiles * c_tiles * p.n;
    PGPP_REQUIRE(blocks <= 2147483647LL, "tensor too large");
    size_t smem = sizeof(float) * 64 * kFirRows * kFirPitch;
    const size_t packets = (size_t)parts * 128 * 8 * sizeof(uint4);
    if (packets > smem) smem = packets;
    static bool attr_done = false;
    if (!attr_done) { PGPP_CUDA_OK(cudaFuncSetAttribute(fir_pack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)); attr_done = true; }
    fir_pack_kernel<<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(p, x_tiles, y_tiles, c_tiles);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}
