// Weight operand preparation for the tensor-core convolution (sm_100a): one launch turns a convolution weight tensor
// into the [parts][taps][o_rows][c_pad] 16-bit K-major operand the TMA weight map of conv_igemm.cu reads - scale, spatial
// flip, input/output transposition, zero padding of rows and channels, the bf16 expansion (or a plain fp16 copy), and for
// the StyleGAN2 up=2 layer the polyphase combination with the 4x4 FIR - and optionally keeps the fp32 "master" rows the
// per-sample (style-modulated) weight route starts from.
//
// Replaces the eager-PyTorch packing of round 1 (a 144-iteration Python loop of GPU ops for the polyphase form, torch.zeros /
// stack / cast chains for the plain form), which invalidated on every optimizer step and dominated the launch count of a
// training iteration.  A weight tensor is at most 512 x 512 x 3 x 3: the kernel is launch-latency sized, not bandwidth sized.
#include "common.cuh"

namespace pgpp {

struct WPackArgs {
    const void* w; int w_dtype;
    int o, ic, kh, kw;                 // logical [O, I, kh, kw] AFTER the optional transposition
    long long s_o, s_i, s_y, s_x;      // element strides of the logical dimensions in the source tensor
    int flip;                          // 1: spatially flipped kernel (true convolution); 0: correlation kernel as stored
    float scale;
    int phases, phase_stride;          // 4: polyphase up=2 form (kh = kw = 3, 4x4 FIR), rows = phase * phase_stride + o
    const float* fir; int flip_filter; // phases == 4: the FIR (device, 16 floats, row-major [fy][fx]); flipped unless flip_filter
    int taps, o_rows, o_off, c_pad, parts, f16;
    uint16_t* out; float* master;
    long long part_stride;             // taps * o_rows * c_pad
};

template <class T> __device__ __forceinline__ float wload(const void* p, long long i) { return (float)to_acc<T>(((const T*)p)[i]); }

__device__ __forceinline__ float wget(const WPackArgs& a, int o, int i, int ky, int kx) {
    if (a.flip) { ky = a.kh - 1 - ky; kx = a.kw - 1 - kx; }
    const long long idx = o * a.s_o + i * a.s_i + ky * a.s_y + kx * a.s_x;
    switch (a.w_dtype) {
        case PGPP_F32: return wload<float>(a.w, idx);
        case PGPP_F16: return wload<__half>(a.w, idx);
        case PGPP_BF16: return wload<__nv_bfloat16>(a.w, idx);
        default: return (float)((const double*)a.w)[idx];
    }
}

// one thread = 8 consecutive channels of one (tap, row): one 16-byte store per part
__global__ void __launch_bounds__(256) pack_weights_kernel(WPackArgs a, long long total8) {
    __shared__ float s_fir[16];
    if (a.phases == 4) {
        if (threadIdx.x < 16) {
            const int fy = threadIdx.x >> 2, fx = threadIdx.x & 3;
            // upfirdn2d correlates with the flipped filter unless flip_filter (upfirdn2d.py:193-196); the gain 4 = up^2 is folded in
            s_fir[threadIdx.x] = 4.f * (a.flip_filter ? a.fir[fy * 4 + fx] : a.fir[(3 - fy) * 4 + (3 - fx)]);
        }
        __syncthreads();
    }
    const int c8 = a.c_pad >> 3;
    const int rows = a.phases == 4 ? a.phases * a.phase_stride : a.o;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total8; e += (long long)gridDim.x * blockDim.x) {
        const int cg = (int)(e % c8);
        long long r = e / c8;
        const int row = (int)(r % rows);
        const int tap = (int)(r / rows);
        int o = row, phase = 0;
        if (a.phases == 4) { phase = row / a.phase_stride; o = row - phase * a.phase_stride; }
        float v[8];
        #pragma unroll
        for (int j = 0; j < 8; j++) {
            const int i = cg * 8 + j;
            float val = 0.f;
            if (o < a.o && i < a.ic) {
                if (a.phases == 1) {
                    val = wget(a, o, i, tap / a.kw, tap % a.kw);
                } else {
                    // Wp[py,px][o,i,ta,tb] = 4 * sum_{fy,ky: py + fy - 1 - ky = 2 (ta - 1)} sum_{fx,kx: px + fx - 1 - kx = 2 (tb - 1)} k[fy,fx] w'[o,i,ky,kx]
                    // (conv_transpose2d(stride 2) then the 4x4 FIR, conv2d_resample.py:125-139, as one 3x3 stencil per output phase)
                    const int py = phase >> 1, px = phase & 1, ta = tap / 3, tb = tap % 3;
                    for (int fy = 0; fy < 4; fy++) {
                        const int ky = py + fy - 1 - 2 * (ta - 1);
                        if (ky < 0 || ky > 2) continue;
                        for (int fx = 0; fx < 4; fx++) {
                            const int kx = px + fx - 1 - 2 * (tb - 1);
                            if (kx < 0 || kx > 2) continue;
                            val = fmaf(s_fir[fy * 4 + fx], wget(a, o, i, ky, kx), val);
                        }
                    }
                }
                val *= a.scale;
            }
            v[j] = val;
        }
        const long long dst = ((long long)tap * a.o_rows + a.o_off + row) * a.c_pad + cg * 8;
        if (a.master) {
            float4* m = reinterpret_cast<float4*>(a.master + dst);
            m[0] = make_float4(v[0], v[1], v[2], v[3]);
            m[1] = make_float4(v[4], v[5], v[6], v[7]);
        }
        for (int part = 0; part < (a.out ? a.parts : 0); part++) {
            __align__(16) uint16_t q[8];
            #pragma unroll
            for (int j = 0; j < 8; j++) {
                if (a.f16) {
                    const __half h = __float2half_rn(v[j]);
                    q[j] = __half_as_ushort(h);
                    v[j] -= __half2float(h);
                } else {
                    const __nv_bfloat16 h = __float2bfloat16_rn(v[j]);
                    q[j] = __bfloat16_as_ushort(h);
                    v[j] -= __bfloat162float(h);
                }
            }
            *reinterpret_cast<uint4*>(a.out + part * a.part_stride + dst) = *reinterpret_cast<const uint4*>(q);
        }
    }
}

// e4m3 weights with one scale per GEMM column (pgpp_quantize_weights_e4m3): one CTA per (column g, sample n).  Pass 1: absmax over
// every tap and channel of the column; pass 2: bytes = e4m3(v / scale), four channels per 32-bit store.
__global__ void __launch_bounds__(256) quantize_weights_e4m3_kernel(const float* __restrict__ master, const float* __restrict__ s, int taps,
                                                                    int o_rows, int c_pad, int c_in, uint8_t* __restrict__ out,
                                                                    float* __restrict__ scale) {
    __shared__ float s_red[8];
    const int g = blockIdx.x, n = blockIdx.y;
    const int q4 = c_pad >> 2, total = taps * q4;
    auto value = [&](int t, int c) -> float {
        if (c >= c_in) return 0.f;
        const float m = master[((long long)t * o_rows + g) * c_pad + c];
        return s ? m * s[(long long)n * c_in + c] : m;
    };
    float amax = 0.f;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
        const int t = e / q4, c = (e - t * q4) * 4;
        #pragma unroll
        for (int j = 0; j < 4; j++) amax = fmaxf(amax, fabsf(value(t, c + j)));
    }
    #pragma unroll
    for (int m = 16; m > 0; m >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, m));
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = amax;
    __syncthreads();
    amax = s_red[0];
    for (int w = 1; w < 8; w++) amax = fmaxf(amax, s_red[w]);
    const float sc = __fdiv_rn(amax, 448.f);
    if (threadIdx.x == 0) scale[(long long)n * o_rows + g] = sc;
    uint8_t* dst = out + (long long)n * taps * o_rows * c_pad;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
        const int t = e / q4, c = (e - t * q4) * 4;
        float v[4];
        #pragma unroll
        for (int j = 0; j < 4; j++) v[j] = sc > 0.f ? __fdiv_rn(value(t, c + j), sc) : 0.f;
        *reinterpret_cast<uint32_t*>(dst + ((long long)t * o_rows + g) * c_pad + c) = e4m3x4(v[0], v[1], v[2], v[3]);
    }
}

// gradient of the polyphase weights back to the 3x3 kernel: the adjoint of the construction above
//   dW[o,i,ky,kx] = sum_{py,px,ta,tb,fy,fx matching} 4 k[fy,fx] dWp[py,px][o,i,ta,tb]
struct WUnpackArgs { const float* g; float* out; const float* fir; int flip_filter, flip, o, ic; long long total; };

__global__ void __launch_bounds__(256) up2_weight_adjoint_kernel(WUnpackArgs a) {
    __shared__ float s_fir[16];
    if (threadIdx.x < 16) {
        const int fy = threadIdx.x >> 2, fx = threadIdx.x & 3;
        s_fir[threadIdx.x] = 4.f * (a.flip_filter ? a.fir[fy * 4 + fx] : a.fir[(3 - fy) * 4 + (3 - fx)]);
    }
    __syncthreads();
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < a.total; e += (long long)gridDim.x * blockDim.x) {
        // e indexes the logical (unflipped-storage) weight [o][i][ky_s][kx_s]
        const int kxs = (int)(e % 3), kys = (int)((e / 3) % 3);
        const int i = (int)((e / 9) % a.ic), o = (int)(e / (9ll * a.ic));
        const int ky = a.flip ? 2 - kys : kys, kx = a.flip ? 2 - kxs : kxs;
        float acc = 0.f;
        for (int py = 0; py < 2; py++)
            for (int fy = 0; fy < 4; fy++) {
                const int num = py + fy - 1 - ky;
                if (num & 1) continue;
                const int ta = num / 2 + 1;     // num in {-3..4}; even values -2, 0, 2, 4 -> ta 0..3
                if (num < -2 || ta > 2) continue;
                for (int px = 0; px < 2; px++)
                    for (int fx = 0; fx < 4; fx++) {
                        const int nx = px + fx - 1 - kx;
                        if (nx & 1) continue;
                        const int tb = nx / 2 + 1;
                        if (nx < -2 || tb > 2) continue;
                        // g layout: [4 phases][O][I][3][3]
                        acc = fmaf(s_fir[fy * 4 + fx], a.g[((((long long)(py * 2 + px) * a.o + o) * a.ic + i) * 3 + ta) * 3 + tb], acc);
                    }
            }
        a.out[e] = acc;
    }
}

} // namespace pgpp

extern "C" int pgpp_pack_weights(const void* w, int w_dtype, const int64_t w_size[4], const int64_t w_stride[4], int transpose_io, int flip,
                                 float scale, int phases, int phase_stride, const float* fir, int flip_filter,
                                 void* out, float* master, int parts, int operand_f16, int o_rows, int o_off, int c_pad, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(w && (out || master), "w and out (or master) must be device pointers");
    PGPP_REQUIRE(w_dtype >= 0 && w_dtype <= 3, "unsupported weight dtype");
    PGPP_REQUIRE(parts >= 1 && parts <= 3 && (!operand_f16 || parts == 1), "parts must be 1..3 (1 for fp16 operands)");
    PGPP_REQUIRE(c_pad >= 8 && c_pad % 8 == 0, "c_pad must be a positive multiple of 8");
    PGPP_REQUIRE(phases == 1 || phases == 4, "phases must be 1 or 4");
    WPackArgs a;
    a.w = w; a.w_dtype = w_dtype;
    const int d_o = transpose_io ? 1 : 0, d_i = transpose_io ? 0 : 1;
    a.o = (int)w_size[d_o]; a.ic = (int)w_size[d_i]; a.kh = (int)w_size[2]; a.kw = (int)w_size[3];
    a.s_o = w_stride[d_o]; a.s_i = w_stride[d_i]; a.s_y = w_stride[2]; a.s_x = w_stride[3];
    a.flip = flip ? 1 : 0; a.scale = scale;
    a.phases = phases; a.phase_stride = phases == 4 ? phase_stride : a.o;
    a.fir = fir; a.flip_filter = flip_filter ? 1 : 0;
    PGPP_REQUIRE(a.o >= 1 && a.ic >= 1 && a.kh >= 1 && a.kw >= 1, "empty weight tensor");
    PGPP_REQUIRE(a.ic <= c_pad, "c_pad is smaller than the input channel count");
    if (phases == 4) {
        PGPP_REQUIRE(a.kh == 3 && a.kw == 3 && fir != nullptr, "the polyphase up=2 form needs a 3x3 kernel and the 4x4 FIR");
        PGPP_REQUIRE(phase_stride >= a.o, "phase_stride must be >= out channels");
        a.taps = 9;
    } else {
        a.taps = a.kh * a.kw;
    }
    const int rows = phases == 4 ? 4 * a.phase_stride : a.o;
    PGPP_REQUIRE(o_off >= 0 && o_off + rows <= o_rows, "rows do not fit the destination (o_off + rows > o_rows)");
    a.o_rows = o_rows; a.o_off = o_off; a.c_pad = c_pad; a.parts = parts; a.f16 = operand_f16 ? 1 : 0;
    a.out = (uint16_t*)out; a.master = master;
    a.part_stride = (long long)a.taps * o_rows * c_pad;
    PGPP_REQUIRE(((uintptr_t)out & 15) == 0 && ((uintptr_t)master & 15) == 0, "destinations must be 16-byte aligned");
    const long long total8 = (long long)a.taps * rows * (c_pad / 8);
    long long blocks = (total8 + 255) / 256;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    pack_weights_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, total8);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

extern "C" int pgpp_up2_weight_adjoint(const float* grad_polyphase, const float* fir, int flip_filter, int flip, int o, int ic,
                                       float* grad_weight, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(grad_polyphase && fir && grad_weight && o >= 1 && ic >= 1, "bad arguments");
    WUnpackArgs a{grad_polyphase, grad_weight, fir, flip_filter ? 1 : 0, flip ? 1 : 0, o, ic, 9ll * o * ic};
    long long blocks = (a.total + 255) / 256;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    up2_weight_adjoint_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}

extern "C" int pgpp_quantize_weights_e4m3(const float* master, const float* s, int n, int taps, int o_rows, int c_pad, int c_in,
                                          void* out, float* scale, void* stream) {
    using namespace pgpp;
    PGPP_REQUIRE(master && out && scale, "master, out and scale must be device pointers");
    PGPP_REQUIRE(n >= 1 && n <= 65535 && taps >= 1 && o_rows >= 1 && c_pad >= 16 && c_pad % 16 == 0 && c_in >= 1 && c_in <= c_pad,
                 "bad quantize_weights_e4m3 arguments");
    PGPP_REQUIRE(s != nullptr || n == 1, "shared weights (s == NULL) need n == 1");
    PGPP_REQUIRE(((uintptr_t)out & 3) == 0, "out must be 4-byte aligned");
    quantize_weights_e4m3_kernel<<<dim3((unsigned)o_rows, (unsigned)n), 256, 0, (cudaStream_t)stream>>>(master, s, taps, o_rows, c_pad, c_in,
                                                                                                         (uint8_t*)out, scale);
    count_launch();
    PGPP_CUDA_OK(cudaGetLastError());
    return PGPP_OK;
}
