// Memory-bound ops of the quantized forward: quantize / dequantize / relu / 2x2 max-pool / min-max.
// All are HBM-bound byte streams: 16-byte vector accesses, grids sized in multiples of the SM count,
// warp-shuffle reductions.  Arithmetic follows SURVEY.md Appendix A bit for bit.
#include "common.cuh"

namespace b200q {

static inline int grid_for(int64_t work_items, int threads, int max_waves = 8) {
  int64_t blocks = (work_items + threads - 1) / threads;
  int64_t cap = (int64_t)num_sms() * max_waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

__device__ __forceinline__ uint32_t pack4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  return a | (b << 8) | (c << 16) | (d << 24);
}

// ---------------------------------------------------------------------------------------------------------
// aten::quantize_per_tensor, fp32 NCHW (c <= 4) -> uint8 NHWC with 4 channels per pixel.
// Each thread converts 4 consecutive pixels: c float4 loads (one per plane), one 16-byte store.
__global__ void __launch_bounds__(256) quantize_nchw_to_nhwc4_kernel(const float* __restrict__ x,
                                                                     uint32_t* __restrict__ y, int64_t n_img, int c,
                                                                     int hw, float inv_scale, int zp) {
  const int64_t quads_per_img = hw / 4;
  const int64_t total = n_img * quads_per_img;
  const uint32_t zpb = (uint32_t)zp;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t img = i / quads_per_img;
    const int64_t q = i - img * quads_per_img;
    const float* base = x + img * c * hw + q * 4;
    uint32_t px[4] = {0, 0, 0, 0};
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
      if (ch < c) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(base + (int64_t)ch * hw));
        px[0] |= quantize_u8(v.x, inv_scale, zp) << (8 * ch);
        px[1] |= quantize_u8(v.y, inv_scale, zp) << (8 * ch);
        px[2] |= quantize_u8(v.z, inv_scale, zp) << (8 * ch);
        px[3] |= quantize_u8(v.w, inv_scale, zp) << (8 * ch);
      } else {
#pragma unroll
        for (int p = 0; p < 4; ++p) px[p] |= zpb << (8 * ch);
      }
    }
    reinterpret_cast<uint4*>(y)[i] = make_uint4(px[0], px[1], px[2], px[3]);
  }
}

// Generic (any c, c_pad) fallback: one thread per output byte.
__global__ void quantize_nchw_to_nhwc_generic_kernel(const float* __restrict__ x, uint8_t* __restrict__ y,
                                                     int64_t n_img, int c, int hw, int c_pad, float inv_scale,
                                                     int zp) {
  const int64_t total = n_img * hw * c_pad;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ch = (int)(i % c_pad);
    const int64_t pix = i / c_pad;
    const int64_t img = pix / hw;
    const int64_t p = pix - img * hw;
    y[i] = ch < c ? (uint8_t)quantize_u8(__ldg(x + (img * c + ch) * hw + p), inv_scale, zp) : (uint8_t)zp;
  }
}

// Flat quantize: 16 floats in (4 x float4), 16 bytes out per thread-iteration.
// qp (optional, device): {min, max, scale, inv_scale, zp-as-float} produced by minmax_kernel.
__global__ void __launch_bounds__(256) quantize_flat_kernel(const float* __restrict__ x, uint8_t* __restrict__ y,
                                                            int64_t n, float inv_scale, int zp,
                                                            const float* __restrict__ qp) {
  if (qp != nullptr) {
    inv_scale = qp[3];
    zp = (int)qp[4];
  }
  const int64_t nvec = n / 16;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const float4* src = reinterpret_cast<const float4*>(x) + i * 4;
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 v = __ldg(src + j);
      w[j] = pack4(quantize_u8(v.x, inv_scale, zp), quantize_u8(v.y, inv_scale, zp), quantize_u8(v.z, inv_scale, zp),
                   quantize_u8(v.w, inv_scale, zp));
    }
    reinterpret_cast<uint4*>(y)[i] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  if (blockIdx.x == 0) {
    for (int64_t i = nvec * 16 + threadIdx.x; i < n; i += blockDim.x) y[i] = (uint8_t)quantize_u8(x[i], inv_scale, zp);
  }
}

// aten::dequantize.  The output is four times the input, so the kernel is bound by its WRITES: every store instruction
// of a warp covers 512 contiguous bytes (lane l converts word l of a 128-byte group into one float4); four independent
// groups per thread and iteration keep enough loads in flight.  (The first version gave each thread 16 input bytes and
// four float4 stores 64 bytes apart: 3.9 TB/s; r02 ncu.)
__global__ void __launch_bounds__(256) dequantize_kernel(const uint8_t* __restrict__ q, float* __restrict__ y,
                                                         int64_t n, float scale, int zp) {
  const int64_t nword = n / 4;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(q);
  float4* dst = reinterpret_cast<float4*>(y);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nword; i += 4 * stride) {
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = (i + j * stride < nword) ? __ldg(src + i + j * stride) : 0u;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (i + j * stride >= nword) break;
      float4 o;
      o.x = __fmul_rn(__int2float_rn((int)(w[j] & 0xff) - zp), scale);
      o.y = __fmul_rn(__int2float_rn((int)((w[j] >> 8) & 0xff) - zp), scale);
      o.z = __fmul_rn(__int2float_rn((int)((w[j] >> 16) & 0xff) - zp), scale);
      o.w = __fmul_rn(__int2float_rn((int)(w[j] >> 24) - zp), scale);
      dst[i + j * stride] = o;
    }
  }
  if (blockIdx.x == 0) {
    for (int64_t i = nword * 4 + threadIdx.x; i < n; i += blockDim.x)
      y[i] = __fmul_rn(__int2float_rn((int)q[i] - zp), scale);
  }
}

// aten::relu on quint8 = max(q, zp), 16 bytes per thread-iteration via per-byte SIMD max.
__global__ void __launch_bounds__(256) relu_q_kernel(const uint8_t* __restrict__ q, uint8_t* __restrict__ y, int64_t n,
                                                     int zp) {
  const uint32_t z4 = (uint32_t)zp * 0x01010101u;
  const int64_t nvec = n / 16;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(q) + i);
    v.x = __vmaxu4(v.x, z4);
    v.y = __vmaxu4(v.y, z4);
    v.z = __vmaxu4(v.z, z4);
    v.w = __vmaxu4(v.w, z4);
    reinterpret_cast<uint4*>(y)[i] = v;
  }
  if (blockIdx.x == 0) {
    for (int64_t i = nvec * 16 + threadIdx.x; i < n; i += blockDim.x) y[i] = q[i] > zp ? q[i] : (uint8_t)zp;
  }
}

// aten::quantized_max_pool2d 2x2/2 on uint8 NHWC: one thread = 16 channels of one output pixel.
__global__ void __launch_bounds__(256) max_pool2x2_nhwc_kernel(const uint4* __restrict__ x, uint4* __restrict__ y,
                                                               int64_t n_img, int h, int w, int c16) {
  const int ho = h / 2, wo = w / 2;
  const int64_t total = n_img * ho * wo * c16;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % c16);
    int64_t p = i / c16;
    const int xo = (int)(p % wo);
    p /= wo;
    const int yo = (int)(p % ho);
    const int64_t img = p / ho;
    const int64_t r0 = ((img * h + 2 * yo) * w + 2 * xo) * c16 + cv;
    const int64_t r1 = r0 + (int64_t)w * c16;
    const uint4 a = __ldg(x + r0), b = __ldg(x + r0 + c16), c = __ldg(x + r1), d = __ldg(x + r1 + c16);
    uint4 o;
    o.x = max4_u8x4(a.x, b.x, c.x, d.x);
    o.y = max4_u8x4(a.y, b.y, c.y, d.y);
    o.z = max4_u8x4(a.z, b.z, c.z, d.z);
    o.w = max4_u8x4(a.w, b.w, c.w, d.w);
    y[i] = o;
  }
}

// ---------------------------------------------------------------------------------------------------------
// Per-tensor dynamic range: grid-stride float4 loads -> warp shuffle -> block partials -> last block finalises.
// scratch layout: float partial_min[1024], float partial_max[1024], uint32 counter (self-resetting).
// Finaliser also derives the fbgemm reduce_range (qmax=127) activation qparams: out[2]=scale, out[3]=1/scale,
// out[4]=zero-point (as float), mirroring ChooseQuantizationParams as reached by quantized::linear_dynamic.
constexpr int MINMAX_MAX_BLOCKS = 1024;

// Port of ChooseQuantizationParams (ATen/native/quantized/cpu/QuantUtils.h) as quantized::linear_dynamic reaches it:
// qmin = 0, qmax = 255, reduce_range = true (-> 0..127), preserve_sparsity = false.  Double intermediates, the tests on
// float(scale), the SMALL_SCALE_THRESHOLD cut-off with its min/max rescaling and the "smaller error terms" choice
// between the two zero-point candidates follow the original step by step.
__device__ __forceinline__ void choose_qparams_reduce_range(float mn, float mx, float* out) {
  const int qmin = 0, qmax = 127;
  constexpr float SMALL_SCALE_THRESHOLD = 6.1e-5f;
  mn = fminf(mn, 0.f);
  mx = fmaxf(mx, 0.f);
  double scale = ((double)mx - (double)mn) / (double)(qmax - qmin);
  if ((float)scale == 0.0f || isinf(__fdiv_rn(1.0f, (float)scale))) scale = 0.1;
  if (scale < (double)SMALL_SCALE_THRESHOLD) {
    const float org_scale = (float)scale;
    scale = (double)SMALL_SCALE_THRESHOLD;
    if (mn == 0.0f) {
      mx = __fmul_rn(SMALL_SCALE_THRESHOLD, (float)(qmax - qmin));
    } else if (mx == 0.0f) {
      mn = -__fmul_rn(SMALL_SCALE_THRESHOLD, (float)(qmax - qmin));
    } else {
      const float amplifier = __fdiv_rn(SMALL_SCALE_THRESHOLD, org_scale);
      mn = __fmul_rn(mn, amplifier);
      mx = __fmul_rn(mx, amplifier);
    }
  }
  const double zp_from_min = (double)qmin - (double)mn / scale;
  const double zp_from_max = (double)qmax - (double)mx / scale;
  const double err_min = fabs((double)qmin) - fabs((double)mn / scale);
  const double err_max = fabs((double)qmax) - fabs((double)mx / scale);
  const double izp = err_min < err_max ? zp_from_min : zp_from_max;
  int zp;
  if (izp < (double)qmin) zp = qmin;
  else if (izp > (double)qmax) zp = qmax;
  else zp = (int)nearbyint(izp);
  const float s = (float)scale;
  out[2] = s;
  out[3] = __fdiv_rn(1.0f, s);
  out[4] = (float)zp;
}

// DYNAMIC = true: quantized::linear_dynamic's range (always contains 0) + its qparams; false: plain torch.aminmax.
template <bool DYNAMIC>
__global__ void __launch_bounds__(256) minmax_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ out,
                                                     float* __restrict__ partial, unsigned int* __restrict__ counter) {
  const float MN0 = DYNAMIC ? 0.0f : __int_as_float(0x7f800000), MX0 = DYNAMIC ? 0.0f : __int_as_float(0xff800000);
  float mn = MN0, mx = MX0;  // DYNAMIC: range always includes 0 (fbgemm: min(x,0), max(x,0))
  const int64_t nvec = n / 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
    mn = fminf(fminf(mn, v.x), fminf(fminf(v.y, v.z), v.w));
    mx = fmaxf(fmaxf(mx, v.x), fmaxf(fmaxf(v.y, v.z), v.w));
  }
  if (blockIdx.x == 0) {
    for (int64_t i = nvec * 4 + threadIdx.x; i < n; i += blockDim.x) {
      mn = fminf(mn, x[i]);
      mx = fmaxf(mx, x[i]);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  __shared__ float smn[8], smx[8];
  __shared__ bool is_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    smn[warp] = mn;
    smx[warp] = mx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) {
      mn = fminf(mn, smn[i]);
      mx = fmaxf(mx, smx[i]);
    }
    partial[blockIdx.x] = mn;
    partial[MINMAX_MAX_BLOCKS + blockIdx.x] = mx;
    __threadfence();
    const unsigned int done = atomicAdd(counter, 1u);
    is_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    mn = MN0;
    mx = MX0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
      mn = fminf(mn, __ldcg(partial + i));
      mx = fmaxf(mx, __ldcg(partial + MINMAX_MAX_BLOCKS + i));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __syncthreads();
    if (lane == 0) {
      smn[warp] = mn;
      smx[warp] = mx;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int i = 1; i < (int)(blockDim.x >> 5); ++i) {
        mn = fminf(mn, smn[i]);
        mx = fmaxf(mx, smx[i]);
      }
      out[0] = mn;
      out[1] = mx;
      if constexpr (DYNAMIC) choose_qparams_reduce_range(mn, mx, out);
      *counter = 0;  // ready for the next call on this stream
    }
  }
}

int launch_minmax(const float* x, int64_t n, float* out5, void* scratch, cudaStream_t s, bool dynamic) {
  float* partial = reinterpret_cast<float*>(scratch);
  unsigned int* counter = reinterpret_cast<unsigned int*>(partial + 2 * MINMAX_MAX_BLOCKS);
  int blocks = grid_for(n / 4 + 1, 256, 4);
  if (blocks > MINMAX_MAX_BLOCKS) blocks = MINMAX_MAX_BLOCKS;
  if (dynamic)
    minmax_kernel<true><<<blocks, 256, 0, s>>>(x, n, out5, partial, counter);
  else
    minmax_kernel<false><<<blocks, 256, 0, s>>>(x, n, out5, partial, counter);
  return launched("minmax_kernel");
}

// ---------------------------------------------------------------------------------------------------------
// torch.histc for the calibration observers: per-block shared-memory histogram (32-bit counts, shared atomics), flushed
// with one 64-bit global atomic per non-empty bin.  The bin of an element is ATen's CPU rule evaluated in fp32 with the
// same operation order: int(((x - lo) * bins) / (hi - lo)).
constexpr int HISTC_MAX_BINS = 4096;
__global__ void __launch_bounds__(256) histc_kernel(const float* __restrict__ x, int64_t n, float lo, float hi, int bins,
                                                    unsigned long long* __restrict__ hist) {
  __shared__ unsigned int s_hist[HISTC_MAX_BINS];
  for (int i = threadIdx.x; i < bins; i += blockDim.x) s_hist[i] = 0u;
  __syncthreads();
  const float fb = (float)bins, width = __fsub_rn(hi, lo);
  auto count = [&](float v) {
    if (v >= lo && v <= hi) {
      int pos = (int)__fdiv_rn(__fmul_rn(__fsub_rn(v, lo), fb), width);
      if (pos >= bins) pos = bins - 1;
      atomicAdd(&s_hist[pos], 1u);
    }
  };
  const int64_t nvec = n / 4;
  // chunked so that a block's 32-bit counters cannot overflow: <= 2^31 elements per block between flushes is
  // guaranteed by the grid (>= 1 block per 2^24 elements would be enough; the grid is far larger)
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
    count(v.x);
    count(v.y);
    count(v.z);
    count(v.w);
  }
  if (blockIdx.x == 0)
    for (int64_t i = nvec * 4 + threadIdx.x; i < n; i += blockDim.x) count(x[i]);
  __syncthreads();
  for (int i = threadIdx.x; i < bins; i += blockDim.x) {
    const unsigned int c = s_hist[i];
    if (c) atomicAdd(hist + i, (unsigned long long)c);
  }
}

// Byte-wise table look-up y[i] = lut[x[i]]: the table lives in shared memory replicated 32 times with a 4-byte
// interleave (entry v of copy l at word v*32 + l), so the 32 lanes of a warp always hit 32 different banks whatever
// bytes they look up.  16 bytes per thread and iteration.
// In the sandwich forward's PDL chain (b200q_sandwich_forward) the table is filled while the previous conv still runs;
// every access to x and y waits: x is that conv's output and y the buffer it reads.
struct LutTable {
  uint8_t v[256];
};
__global__ void __launch_bounds__(256) lut_u8_kernel(const uint8_t* __restrict__ x, uint8_t* __restrict__ y, int64_t n,
                                                     const __grid_constant__ LutTable lut) {
  __shared__ uint32_t s_lut[256 * 32];
  pdl_launch_dependents();
  for (int i = threadIdx.x; i < 256 * 32; i += blockDim.x) s_lut[i] = lut.v[i >> 5];
  __syncthreads();
  pdl_wait();
  const uint32_t* tab = s_lut + (threadIdx.x & 31);
  auto map4 = [&](uint32_t w) {
    return tab[(w & 0xffu) << 5] | (tab[((w >> 8) & 0xffu) << 5] << 8) | (tab[((w >> 16) & 0xffu) << 5] << 16) |
           (tab[(w >> 24) << 5] << 24);
  };
  const int64_t nvec = n / 16;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(x) + i);
    v.x = map4(v.x);
    v.y = map4(v.y);
    v.z = map4(v.z);
    v.w = map4(v.w);
    reinterpret_cast<uint4*>(y)[i] = v;
  }
  if (blockIdx.x == 0)
    for (int64_t i = nvec * 16 + threadIdx.x; i < n; i += blockDim.x) y[i] = lut.v[x[i]];
}

int launch_quantize_flat(const float* x, uint8_t* y, int64_t n, float inv_scale, int zp, const float* qp_dev,
                         cudaStream_t s) {
  quantize_flat_kernel<<<grid_for(n / 16 + 1, 256), 256, 0, s>>>(x, y, n, inv_scale, zp, qp_dev);
  return launched("quantize_flat_kernel");
}

}  // namespace b200q

using namespace b200q;

extern "C" int b200q_quantize_nchw_to_nhwc(const float* x, uint8_t* y, int64_t b, int c, int h, int w, int c_pad,
                                           float inv_scale, int zp, void* stream) {
  B200Q_REQUIRE(x && y && b >= 0 && c > 0 && h > 0 && w > 0 && c_pad >= c, "quantize_nchw_to_nhwc: bad arguments");
  if (b == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const int hw = h * w;
  if (c_pad == 4 && c <= 4 && hw % 4 == 0 && ((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0)) {
    quantize_nchw_to_nhwc4_kernel<<<grid_for(b * (hw / 4), 256), 256, 0, s>>>(x, reinterpret_cast<uint32_t*>(y), b, c,
                                                                             hw, inv_scale, zp);
  } else {
    quantize_nchw_to_nhwc_generic_kernel<<<grid_for(b * hw * c_pad, 256), 256, 0, s>>>(x, y, b, c, hw, c_pad,
                                                                                      inv_scale, zp);
  }
  return launched("quantize_nchw_to_nhwc");
}

extern "C" int b200q_quantize_flat(const float* x, uint8_t* y, int64_t n, float inv_scale, int zp, void* stream) {
  B200Q_REQUIRE((x && y) || n == 0, "quantize_flat: null pointer");
  B200Q_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0), "quantize_flat: pointers must be 16-byte aligned");
  if (n == 0) return 0;
  return launch_quantize_flat(x, y, n, inv_scale, zp, nullptr, (cudaStream_t)stream);
}

extern "C" int b200q_dequantize(const uint8_t* q, float* y, int64_t n, float scale, int zp, void* stream) {
  B200Q_REQUIRE((q && y) || n == 0, "dequantize: null pointer");
  B200Q_REQUIRE(((uintptr_t)q % 16 == 0) && ((uintptr_t)y % 16 == 0), "dequantize: pointers must be 16-byte aligned");
  if (n == 0) return 0;
  dequantize_kernel<<<grid_for(n / 16 + 1, 256), 256, 0, (cudaStream_t)stream>>>(q, y, n, scale, zp);  // 4 words / thread / iteration
  return launched("dequantize_kernel");
}

extern "C" int b200q_relu_q(const uint8_t* q, uint8_t* y, int64_t n, int zp, void* stream) {
  B200Q_REQUIRE((q && y) || n == 0, "relu_q: null pointer");
  B200Q_REQUIRE(((uintptr_t)q % 16 == 0) && ((uintptr_t)y % 16 == 0), "relu_q: pointers must be 16-byte aligned");
  B200Q_REQUIRE(zp >= 0 && zp <= 255, "relu_q: zero-point out of range");
  if (n == 0) return 0;
  relu_q_kernel<<<grid_for(n / 16 + 1, 256), 256, 0, (cudaStream_t)stream>>>(q, y, n, zp);
  return launched("relu_q_kernel");
}

extern "C" int b200q_max_pool2x2_nhwc(const uint8_t* x, uint8_t* y, int64_t b, int h, int w, int c, void* stream) {
  B200Q_REQUIRE((x && y) || b == 0, "max_pool2x2: null pointer");
  B200Q_REQUIRE(h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0 && c > 0 && c % 16 == 0,
                "max_pool2x2: need even h,w and c %% 16 == 0 (got h=%d w=%d c=%d)", h, w, c);
  B200Q_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0), "max_pool2x2: pointers must be 16-byte aligned");
  if (b == 0) return 0;
  const int64_t total = b * (h / 2) * (w / 2) * (c / 16);
  max_pool2x2_nhwc_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), b, h, w, c / 16);
  return launched("max_pool2x2_nhwc_kernel");
}

extern "C" int b200q_minmax(const float* x, int64_t n, float* out5, void* scratch, void* stream) {
  B200Q_REQUIRE(x && out5 && scratch && n > 0, "minmax: bad arguments");
  B200Q_REQUIRE((uintptr_t)x % 16 == 0, "minmax: x must be 16-byte aligned");
  return launch_minmax(x, n, out5, scratch, (cudaStream_t)stream, true);
}

extern "C" int b200q_aminmax(const float* x, int64_t n, float* out2, void* scratch, void* stream) {
  B200Q_REQUIRE(x && out2 && scratch && n > 0, "aminmax: bad arguments");
  B200Q_REQUIRE((uintptr_t)x % 16 == 0, "aminmax: x must be 16-byte aligned");
  return launch_minmax(x, n, out2, scratch, (cudaStream_t)stream, false);
}

extern "C" int b200q_histc(const float* x, int64_t n, float lo, float hi, int bins, int64_t* hist, void* stream) {
  B200Q_REQUIRE((x && hist) || n == 0, "histc: null pointer");
  B200Q_REQUIRE(bins > 0 && bins <= HISTC_MAX_BINS, "histc: bins must be in [1, %d] (got %d)", HISTC_MAX_BINS, bins);
  B200Q_REQUIRE(lo < hi, "histc: need lo < hi (got %g, %g)", (double)lo, (double)hi);
  B200Q_REQUIRE((uintptr_t)x % 16 == 0 && (uintptr_t)hist % 8 == 0, "histc: misaligned buffers");
  if (n == 0) return 0;
  histc_kernel<<<grid_for(n / 4 + 1, 256, 4), 256, 0, (cudaStream_t)stream>>>(
      x, n, lo, hi, bins, reinterpret_cast<unsigned long long*>(hist));
  return launched("histc_kernel");
}

extern "C" int b200q_lut_u8(const uint8_t* x, uint8_t* y, int64_t n, const uint8_t* lut_host, void* stream) {
  B200Q_REQUIRE(((x && y) || n == 0) && lut_host, "lut_u8: null pointer");
  B200Q_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0), "lut_u8: pointers must be 16-byte aligned");
  if (n == 0) return 0;
  LutTable t;
  for (int i = 0; i < 256; ++i) t.v[i] = lut_host[i];
  return launch_kernel("lut_u8_kernel", lut_u8_kernel, grid_for(n / 16 + 1, 256, 4), 256, 0, (cudaStream_t)stream, x, y,
                       n, t);
}
