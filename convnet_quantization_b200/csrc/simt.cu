// CUDA-core (dp4a) kernels: the first convolution (cin=3, K=27: memory-bound, not tensor-core shaped),
// small linears, and (development builds only, -DB200Q_DEV) a plain direct convolution used as a cross-check for the
// tcgen05 path.
#include "common.cuh"

namespace b200q {

// =========================================================================================================
// First conv (cin = 3 stored as 4, cout = 64, 32x32 images).  Input kinds (C1In):
//   C1_IN_NHWC4  uint8 NHWC4, already quantised (b200q_conv3x3_first);
//   C1_IN_F32    fp32 NCHW, fused with aten::quantize_per_tensor (b200q_quantize_conv3x3_first);
//   C1_IN_U8     raw uint8 NHWC pixels [b,32,32,3] through the host table C1Lut (b200q_u8_conv3x3_first): the halo word
//                lut[0][p0] | lut[1][p1]<<8 | lut[2][p2]<<16 | zp_x<<24 is the word C1_IN_F32 builds from the
//                normalised pixels, and everything after the halo load is shared, so the two agree bit for bit.
// Block = 8 output rows x 32 columns of one image (256 threads, one pixel each, all 64 output channels).
// The quantized halo (10 x 34 pixels, one 32-bit word per pixel) lives in shared memory; out-of-image taps hold
// zp_x (real-domain zero), so acc_true = sum_all x*w - zp_x*sum_all w = raw - corr[interior][c] for every pixel.
// Weights [9 taps][64 cout] words are read as broadcast uint4 (4 output channels per LDS.128).
// CGROUPS: 16-channel groups per CTA.  4 = all 64 channels (grid.y = 1); 1 = one group per CTA (grid.y = 4), the shape
// the whole-network executor uses up to CONV1_TINY_MAX_B images (16 CTAs per image, ~350 instructions per thread: the
// tensor-core kernel of conv1_tc.cu spends ~6 us on a few images in barrier / TMEM / MMA round trips).
constexpr int C1_ROWS = 8;
constexpr int C1_COUT = 64;
constexpr int CONV1_TINY_MAX_B = 32;  // measured: ahead of conv1_tc.cu up to 32 images, level at 64 (r02 sweep)

enum C1In { C1_IN_NHWC4 = 0, C1_IN_F32 = 1, C1_IN_U8 = 2 };

template <int IN, int CGROUPS>
__global__ void __launch_bounds__(256) conv1_kernel(const void* __restrict__ xin, uint8_t* __restrict__ y,
                                                    const uint32_t* __restrict__ w_words,  // [64][9] words
                                                    const int32_t* __restrict__ corr,      // [9][64], row 4 = interior
                                                    const float* __restrict__ mult, const float* __restrict__ bdiv,
                                                    int zp_x, int zp_out, int relu, float inv_scale, int img,
                                                    const __grid_constant__ C1Lut lut) {  // read by C1_IN_U8 only
  __shared__ uint32_t s_in[(C1_ROWS + 2) * 34];
  __shared__ uint4 s_w[9 * (C1_COUT / 4)];
  __shared__ float s_mult[C1_COUT], s_bdiv[C1_COUT];
  __shared__ int s_corr[C1_COUT];
  __shared__ uint32_t s_lut[IN == C1_IN_U8 ? 3 * 256 / 4 : 1];  // [3][256] bytes

  const int tiles_per_img = img / C1_ROWS;
  const int64_t image = blockIdx.x / tiles_per_img;
  const int row0 = (blockIdx.x % tiles_per_img) * C1_ROWS;
  const int tid = threadIdx.x;
  const uint32_t zp_word = (uint32_t)zp_x * 0x01010101u;
  pdl_launch_dependents();

  for (int i = tid; i < 9 * C1_COUT; i += 256) {
    // s_w[tap][c/4].{x,y,z,w} = word(tap, c)
    const int tap = i / C1_COUT, c = i % C1_COUT;
    reinterpret_cast<uint32_t*>(s_w)[tap * C1_COUT + c] = __ldg(w_words + c * 9 + tap);
  }
  if (tid < C1_COUT) {
    s_mult[tid] = __ldg(mult + tid);
    s_bdiv[tid] = __ldg(bdiv + tid);
    s_corr[tid] = __ldg(corr + 4 * C1_COUT + tid);
  }
  if constexpr (IN == C1_IN_U8) {  // the table is a kernel parameter, not the previous kernel's output
    if (tid < 3 * 256 / 4) s_lut[tid] = reinterpret_cast<const uint32_t*>(&lut.q[0][0])[tid];
    __syncthreads();
  }
  pdl_wait();  // y may still be read by the previous kernel of the stream (weights and constants above are not its output)
  for (int i = tid; i < (C1_ROWS + 2) * 34; i += 256) {
    const int r = i / 34 + row0 - 1, c = i % 34 - 1;
    uint32_t word = zp_word;
    if (r >= 0 && r < img && c >= 0 && c < img) {
      if constexpr (IN == C1_IN_F32) {
        const float* x = reinterpret_cast<const float*>(xin) + image * 3 * img * img + r * img + c;
        const uint32_t q0 = quantize_u8(__ldg(x), inv_scale, zp_x);
        const uint32_t q1 = quantize_u8(__ldg(x + img * img), inv_scale, zp_x);
        const uint32_t q2 = quantize_u8(__ldg(x + 2 * img * img), inv_scale, zp_x);
        word = q0 | (q1 << 8) | (q2 << 16) | ((uint32_t)zp_x << 24);
      } else if constexpr (IN == C1_IN_U8) {
        const uint8_t* p = reinterpret_cast<const uint8_t*>(xin) + ((image * img + r) * img + c) * 3;
        const uint8_t* t = reinterpret_cast<const uint8_t*>(s_lut);
        word = (uint32_t)t[__ldg(p)] | ((uint32_t)t[256 + __ldg(p + 1)] << 8) | ((uint32_t)t[512 + __ldg(p + 2)] << 16) |
               ((uint32_t)zp_x << 24);
      } else {
        word = __ldg(reinterpret_cast<const uint32_t*>(xin) + (image * img + r) * img + c);
      }
    }
    s_in[i] = word;
  }
  __syncthreads();

  const int lr = tid / 32, lc = tid % 32;
  if (lc >= img) return;  // (img is 32 for this network; kept for smaller test geometries)
  uint32_t xin9[9];
#pragma unroll
  for (int kh = 0; kh < 3; ++kh)
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) xin9[kh * 3 + kw] = s_in[(lr + kh) * 34 + lc + kw];

  const int lo = relu ? zp_out : 0;
  uint8_t* out = y + ((image * img + row0 + lr) * img + lc) * (int64_t)C1_COUT;
#pragma unroll
  for (int cgi = 0; cgi < CGROUPS; ++cgi) {
    const int cg = blockIdx.y * CGROUPS + cgi;
    uint32_t packed[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const uint4 wv = s_w[tap * (C1_COUT / 4) + cg * 4 + q];
        a0 = dp4a_us(xin9[tap], wv.x, a0);
        a1 = dp4a_us(xin9[tap], wv.y, a1);
        a2 = dp4a_us(xin9[tap], wv.z, a2);
        a3 = dp4a_us(xin9[tap], wv.w, a3);
      }
      const int c = cg * 16 + q * 4;
      packed[q] = requant_u8(a0 - s_corr[c], s_bdiv[c], s_mult[c], zp_out, lo) |
                  (requant_u8(a1 - s_corr[c + 1], s_bdiv[c + 1], s_mult[c + 1], zp_out, lo) << 8) |
                  (requant_u8(a2 - s_corr[c + 2], s_bdiv[c + 2], s_mult[c + 2], zp_out, lo) << 16) |
                  (requant_u8(a3 - s_corr[c + 3], s_bdiv[c + 3], s_mult[c + 3], zp_out, lo) << 24);
    }
    reinterpret_cast<uint4*>(out)[cg] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
  }
}

#ifdef B200Q_DEV
// =========================================================================================================
// Plain direct 3x3 conv, any cin % 4 == 0: one thread per (pixel, output channel).  Bring-up cross-check only.
__global__ void conv3x3_direct_kernel(const uint8_t* __restrict__ x, uint8_t* __restrict__ y, int64_t n_img, int img,
                                      int cin, int cout, const int8_t* __restrict__ w,
                                      const float* __restrict__ mult, const float* __restrict__ bdiv, int zp_x,
                                      int zp_out, int relu) {
  const int64_t total = n_img * img * img * cout;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(i % cout);
    int64_t p = i / cout;
    const int xx = (int)(p % img);
    p /= img;
    const int yy = (int)(p % img);
    const int64_t b = p / img;
    int acc = 0;
    for (int kh = 0; kh < 3; ++kh) {
      const int r = yy + kh - 1;
      if (r < 0 || r >= img) continue;
      for (int kw = 0; kw < 3; ++kw) {
        const int c = xx + kw - 1;
        if (c < 0 || c >= img) continue;
        const uint32_t* xp = reinterpret_cast<const uint32_t*>(x + ((b * img + r) * img + c) * (int64_t)cin);
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(w + ((int64_t)co * 9 + kh * 3 + kw) * cin);
        int raw = 0, wsum = 0;
        for (int k = 0; k < cin / 4; ++k) {
          const uint32_t wv = __ldg(wp + k);
          raw = dp4a_us(__ldg(xp + k), wv, raw);
          wsum = dp4a_us(0x01010101u, wv, wsum);
        }
        acc += raw - zp_x * wsum;
      }
    }
    y[i] = (uint8_t)requant_u8(acc, __ldg(bdiv + co), __ldg(mult + co), zp_out, relu ? zp_out : 0);
  }
}

#endif  // B200Q_DEV

// =========================================================================================================
// Small linear on CUDA cores: y[b][n] = epilogue( sum_k x[b][k]*w[n][k] - zp_x*wsum[n] ).
// Tile 64 (batch) x 64 (n) per 256-thread block, K stepped 64 bytes through shared memory, 4x4 outputs per thread.
enum LinearEpilogue { EPI_REQUANT_U8 = 0, EPI_REQUANT_DEQUANT_F32 = 1 };

struct LinearArgs {
  const uint8_t* x;
  void* y;
  const int8_t* w;
  const int32_t* corr;   // [n] zp_x * wsum
  const float* mult;     // requant mult[n]
  const float* bdiv;     // bdiv[n]
  int64_t b;
  int k, n;
  int zp_out, relu;
  float out_scale;       // dequant scale (EPI_REQUANT_DEQUANT_F32)
};

template <int EPI>
__global__ void __launch_bounds__(256) linear_simt_kernel(const LinearArgs a) {
  constexpr int TB = 64, TN = 64, KW = 16;  // K step = 16 words = 64 bytes
  __shared__ uint32_t sx[TB][KW + 1];
  __shared__ uint32_t sw[TN][KW + 1];
  const int tid = threadIdx.x;
  const int64_t b0 = (int64_t)blockIdx.x * TB;
  const int n0 = blockIdx.y * TN;
  const int tb = (tid / 16) * 4, tn = (tid % 16) * 4;
  int acc[4][4] = {};
  const int kwords = a.k / 4;
  for (int k0 = 0; k0 < kwords; k0 += KW) {
    for (int i = tid; i < TB * KW; i += 256) {
      const int r = i / KW, c = i % KW;
      const int64_t bb = b0 + r;
      sx[r][c] = (bb < a.b && k0 + c < kwords)
                     ? __ldg(reinterpret_cast<const uint32_t*>(a.x + bb * a.k) + k0 + c) : 0u;
      const int nn = n0 + r;
      sw[r][c] = (nn < a.n && k0 + c < kwords)
                     ? __ldg(reinterpret_cast<const uint32_t*>(a.w + (int64_t)nn * a.k) + k0 + c) : 0u;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < KW; ++c) {
      uint32_t xv[4], wv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        xv[i] = sx[tb + i][c];
        wv[i] = sw[tn + i][c];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = dp4a_us(xv[i], wv[j], acc[i][j]);
    }
    __syncthreads();
  }
  const int lo = a.relu ? a.zp_out : 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t bb = b0 + tb + i;
    if (bb >= a.b) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int nn = n0 + tn + j;
      if (nn >= a.n) continue;
      const uint32_t q =
          requant_u8(acc[i][j] - __ldg(a.corr + nn), __ldg(a.bdiv + nn), __ldg(a.mult + nn), a.zp_out, lo);
      if constexpr (EPI == EPI_REQUANT_U8) {
        reinterpret_cast<uint8_t*>(a.y)[bb * a.n + nn] = (uint8_t)q;
      } else {
        reinterpret_cast<float*>(a.y)[bb * a.n + nn] = __fmul_rn(__int2float_rn((int)q - a.zp_out), a.out_scale);
      }
    }
  }
}

// ---- accuracy counting inside the head (EVAL instantiations; the rule is stated in b200q.h at B200Q_EVAL_COUNTERS).
// Called by the whole warp once per image, lane n < N holding the uint8 output q[n] (other lanes: anything).  The
// uint8 values are compared, not the logits: dequantisation is strictly monotone.  Every lane ends with the same
// counts; lane 0's are added up per CTA by eval_flush.
template <int N>
__device__ __forceinline__ void eval_image(uint32_t q, int lane, int64_t img, const EvalArgs& ev, uint32_t (&cnt)[5]) {
  static_assert(N >= 1 && N <= 32, "one class per lane");
  constexpr unsigned kClasses = N == 32 ? 0xffffffffu : (1u << N) - 1u;
  constexpr int K5 = N < 5 ? N : 5;
  const int64_t label = __ldg(ev.labels + img);
  const bool valid = label >= 0 && label < N;
  const int l = valid ? (int)label : 0;
  const uint32_t ql = __shfl_sync(0xffffffffu, q, l);
  const unsigned gt = __ballot_sync(0xffffffffu, q > ql) & kClasses;
  const unsigned eq = __ballot_sync(0xffffffffu, q == ql) & kClasses;
  const int g = __popc(gt), e = __popc(eq) - 1;  // e excludes the label itself
  const int rank = g + __popc(eq & ((1u << l) - 1u));
  if (valid) {
    cnt[B200Q_EVAL_TOP1] += rank < 1;
    cnt[B200Q_EVAL_TOP5] += rank < K5;
    cnt[B200Q_EVAL_TOP1_TIED] += g < 1 && 1 <= g + e;
    cnt[B200Q_EVAL_TOP5_TIED] += g < K5 && K5 <= g + e;
  }
  cnt[B200Q_EVAL_IMAGES] += 1;
  if (ev.pred != nullptr) {  // rank-0 class: the first index holding the maximum
    const uint32_t qmax = __reduce_max_sync(0xffffffffu, lane < N ? q : 0u);
    const unsigned at_max = __ballot_sync(0xffffffffu, q == qmax) & kClasses;
    if (lane == 0) ev.pred[img] = __ffs(at_max) - 1;
  }
}

// Block-wide sum of lane 0's counts, then one global atomicAdd per (non-zero) counter per CTA.  Integer adds: the
// totals do not depend on the order.  Every thread of the block must call it.
__device__ __forceinline__ void eval_flush(const uint32_t (&cnt)[5], const EvalArgs& ev) {
  __shared__ unsigned long long s_cnt[B200Q_EVAL_COUNTERS];
  if (threadIdx.x < B200Q_EVAL_COUNTERS) s_cnt[threadIdx.x] = 0ull;
  __syncthreads();
  if ((threadIdx.x & 31) == 0)
#pragma unroll
    for (int i = 0; i < B200Q_EVAL_COUNTERS; ++i)
      if (cnt[i]) atomicAdd(&s_cnt[i], (unsigned long long)cnt[i]);
  __syncthreads();
  if (threadIdx.x < B200Q_EVAL_COUNTERS && s_cnt[threadIdx.x]) atomicAdd(ev.counters + threadIdx.x, s_cnt[threadIdx.x]);
}

// Narrow head (fc2: k = 512, n = 10) fused with aten::dequantize.  The generic tile kernel above pads n to 64 and ran
// this 8 MB layer at 29 us; here a warp owns one image at a time: lane l reads bytes [16l, 16l+16) of the image's row
// (one coalesced 512-byte load per image), holds the matching 16 bytes of all N weight rows in registers, and the N
// dot products are completed with the warp-reduce instruction.  Lane n then requantises and dequantises output n.
// EVAL: also counts (eval_image); the logits store is skipped when a.y is nullptr.
template <int N, bool EVAL>
__global__ void __launch_bounds__(256) linear_head_dequant_kernel(const LinearArgs a, const EvalArgs ev) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  pdl_launch_dependents();
  uint4 w[N];
#pragma unroll
  for (int n = 0; n < N; ++n) w[n] = __ldg(reinterpret_cast<const uint4*>(a.w + (int64_t)n * 512) + lane);
  const int nn = lane < N ? lane : 0;
  const int corr = __ldg(a.corr + nn);
  const float bdiv = __ldg(a.bdiv + nn), mult = __ldg(a.mult + nn);
  const int lo = a.relu ? a.zp_out : 0;
  pdl_wait();  // x is the previous kernel's output (weights and constants above are not)
  uint4 xv = make_uint4(0, 0, 0, 0);
  if (warp < a.b) xv = __ldg(reinterpret_cast<const uint4*>(a.x + (int64_t)warp * 512) + lane);
  uint32_t cnt[5] = {0, 0, 0, 0, 0};
  for (int64_t img = warp; img < a.b; img += nwarps) {
    const uint4 x = xv;
    if (img + nwarps < a.b) xv = __ldg(reinterpret_cast<const uint4*>(a.x + (img + nwarps) * 512) + lane);  // prefetch
    int mine = 0;
#pragma unroll
    for (int n = 0; n < N; ++n) {
      int acc = dp4a_us(x.x, w[n].x, 0);
      acc = dp4a_us(x.y, w[n].y, acc);
      acc = dp4a_us(x.z, w[n].z, acc);
      acc = dp4a_us(x.w, w[n].w, acc);
      acc = __reduce_add_sync(0xffffffffu, acc);
      if (lane == n) mine = acc;
    }
    if (lane < N) {
      const uint32_t q = requant_u8(mine - corr, bdiv, mult, a.zp_out, lo);
      if (!EVAL || a.y != nullptr)
        reinterpret_cast<float*>(a.y)[img * N + lane] = __fmul_rn(__int2float_rn((int)q - a.zp_out), a.out_scale);
      if constexpr (EVAL) mine = (int)q;
    }
    if constexpr (EVAL) eval_image<N>((uint32_t)mine, lane, img, ev, cnt);
  }
  if constexpr (EVAL) eval_flush(cnt, ev);
}

// =========================================================================================================
// fp32 head of the sandwich net (b200q_sandwich_forward; b200q.h states the order): fc1's uint8 output through ReLU and
// DeQuantStub, then fp32 fc2 + bias.  Called by the whole warp for one image: lane l holds bytes [16l, 16l+16) of the
// 512-byte row, w4(n, j) returns this lane's float4 w[n][16l+4j .. 16l+4j+3], bias_n is fc2's bias of output `lane`
// (lanes >= 10: anything).  Returns y[lane] on lanes < 10.  Each multiply and add rounds on its own (no FMA) and the
// butterfly leaves the same sum in every lane, so the logits depend on neither the batch nor the kernel that calls it.
constexpr int SW_K = 512, SW_N = 10;

template <class W4>
__device__ __forceinline__ float sandwich_head_image(uint4 q, int lane, int zp, float scale, float bias_n, W4 w4) {
  const uint32_t words[4] = {q.x, q.y, q.z, q.w};
  float h[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int v = (int)((words[i / 4] >> (8 * (i % 4))) & 0xffu);
    h[i] = __fmul_rn(__int2float_rn(max(v, zp) - zp), scale);
  }
  float mine = 0.f;
#pragma unroll
  for (int n = 0; n < SW_N; ++n) {
    float p = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 w = w4(n, j);
      p = j == 0 ? __fmul_rn(h[0], w.x) : __fadd_rn(p, __fmul_rn(h[4 * j], w.x));
      p = __fadd_rn(p, __fmul_rn(h[4 * j + 1], w.y));
      p = __fadd_rn(p, __fmul_rn(h[4 * j + 2], w.z));
      p = __fadd_rn(p, __fmul_rn(h[4 * j + 3], w.w));
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) p = __fadd_rn(p, __shfl_xor_sync(0xffffffffu, p, d));
    if (lane == n) mine = p;
  }
  return __fadd_rn(mine, bias_n);
}

// Large batches: one warp per image as in linear_head_dequant_kernel.  The 20 KB of fp32 weights go to shared memory
// before the PDL wait, as [n][j][lane] float4s so that the 32 lanes of a warp read 32 consecutive float4s.
__global__ void __launch_bounds__(256) sandwich_head_kernel(const uint8_t* __restrict__ x, float* __restrict__ y,
                                                            int64_t b, const float* __restrict__ w,
                                                            const float* __restrict__ bias, int zp, float scale) {
  __shared__ float4 s_w[SW_N * 4 * 32];
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  pdl_launch_dependents();
  for (int i = threadIdx.x; i < SW_N * SW_K / 4; i += blockDim.x)  // source float4 i = (n * 32 + l) * 4 + j
    s_w[((i / 128) * 4 + i % 4) * 32 + (i / 4) % 32] = __ldg(reinterpret_cast<const float4*>(w) + i);
  const float bias_n = lane < SW_N ? __ldg(bias + lane) : 0.f;
  __syncthreads();
  pdl_wait();  // x is the previous kernel's output
  const auto w4 = [&](int n, int j) { return s_w[(n * 4 + j) * 32 + lane]; };
  uint4 xv = make_uint4(0, 0, 0, 0);
  if (warp < b) xv = __ldg(reinterpret_cast<const uint4*>(x + (int64_t)warp * SW_K) + lane);
  for (int64_t img = warp; img < b; img += nwarps) {
    const uint4 q = xv;
    if (img + nwarps < b) xv = __ldg(reinterpret_cast<const uint4*>(x + (img + nwarps) * SW_K) + lane);  // prefetch
    const float v = sandwich_head_image(q, lane, zp, scale, bias_n, w4);
    if (lane < SW_N) y[img * SW_N + lane] = v;
  }
}

// =========================================================================================================
// Small-batch classifier head (whole-network executor, b <= FC_SMALL_MAX_B): fc1 (+ReLU) and fc2 + dequantize in ONE
// launch.  At batch 1 the tensor-core fc1 kernel is a chain of 128 dependent-ish MMAs behind a 256 KB weight stream on
// eight SMs, followed by a second launch for ten dot products; here all 2 MB of fc1 weights are read once, 16 KB per
// CTA on 128 SMs, by dp4a:
//   * CTA c owns output channels 4c..4c+3 and keeps their four weight rows (16 KB) in shared memory - loaded BEFORE the
//     programmatic-dependent-launch wait, i.e. while the previous layer is still running;
//   * a warp takes one image at a time: its 4 KB row as eight 16-byte loads per lane (all in flight at once, the next
//     image's issued before this one is reduced), 4 x 32 dp4a per lane, REDUX across the warp, exact fbgemm
//     requantisation, one byte per (image, channel).  No block-wide synchronisation in the loop;
//   * the CTA that finishes LAST (a ticket in the caller's workspace, reset by that CTA) runs fc2 + dequantize on the
//     512-byte rows all CTAs wrote (read through L2), one warp per image as in linear_head_dequant_kernel.
// Integer accumulation is exact in any order, so the result is bit-identical to the two-kernel path.
constexpr int FC_SMALL_MAX_B = 32;  // measured: ahead of the two-kernel head up to 32 images, behind it at 64 (r02 sweep)

struct FcSmallArgs {
  const uint8_t* x;       // [b][4096] uint8 (NHWC-flattened pool3 output)
  uint8_t* h;             // [b][512] scratch: fc1 output
  float* logits;          // [b][10]
  unsigned int* ticket;   // zero on entry, zero on exit
  const int8_t* w1;       // [512][4096]
  const int32_t* corr1;
  const float* mult1;
  const float* bdiv1;
  const int8_t* w2;       // [10][512]
  const int32_t* corr2;
  const float* mult2;
  const float* bdiv2;
  int b;
  int zp1, lo1;           // fc1 output zero-point, lower clamp (ReLU: zp1)
  int zp2, lo2;
  float out_scale;
};
// fc_head_small_kernel<false, true> (sandwich net): fp32 fc2 [10][512] and bias [10], fc1's DeQuantStub scale (its
// zero-point is FcSmallArgs::zp1).
struct F32HeadArgs {
  const float* w;
  const float* bias;
  float scale;
};

// EVAL: the last CTA's fc2 stage also counts (eval_image), and skips the logits store when a.logits is nullptr.
// F32HEAD (sandwich net): the last CTA runs the fp32 head (sandwich_head_image) instead of the int8 fc2 + dequantize.
template <bool EVAL, bool F32HEAD = false>
__global__ void __launch_bounds__(256) fc_head_small_kernel(const FcSmallArgs a, const EvalArgs ev,
                                                            const F32HeadArgs f) {
  constexpr int K = 4096, N1 = 512, N2 = 10, CH = 4, KV = K / 16 / 32;  // KV: 16-byte vectors per lane and row
  __shared__ uint4 s_w[CH][K / 16];
  __shared__ bool s_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c0 = blockIdx.x * CH;
  pdl_launch_dependents();
#pragma unroll
  for (int c = 0; c < CH; ++c) s_w[c][tid] = __ldg(reinterpret_cast<const uint4*>(a.w1 + (int64_t)(c0 + c) * K) + tid);
  uint4 w2[N2];  // every CTA prefetches fc2's 5 KB (only the last one uses them): hides the load behind fc1
  if constexpr (!F32HEAD) {
#pragma unroll
    for (int n = 0; n < N2; ++n) w2[n] = __ldg(reinterpret_cast<const uint4*>(a.w2 + n * N1) + lane);
  }
  const int myc = c0 + (lane & 3);
  const int corr1 = __ldg(a.corr1 + myc);
  const float bdiv1 = __ldg(a.bdiv1 + myc), mult1 = __ldg(a.mult1 + myc);
  pdl_wait();  // x is the previous kernel's output
  __syncthreads();
  auto load_row = [&](uint4 (&v)[KV], int img) {
#pragma unroll
    for (int j = 0; j < KV; ++j) v[j] = __ldg(reinterpret_cast<const uint4*>(a.x + (int64_t)img * K) + j * 32 + lane);
  };
  uint4 cur[KV], nxt[KV];
  if (warp < a.b) load_row(cur, warp);
  for (int img = warp; img < a.b; img += 8) {
    if (img + 8 < a.b) load_row(nxt, img + 8);
    int acc[CH] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < KV; ++j)
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const uint4 wv = s_w[c][j * 32 + lane];
        acc[c] = dp4a_us(cur[j].x, wv.x, acc[c]);
        acc[c] = dp4a_us(cur[j].y, wv.y, acc[c]);
        acc[c] = dp4a_us(cur[j].z, wv.z, acc[c]);
        acc[c] = dp4a_us(cur[j].w, wv.w, acc[c]);
      }
#pragma unroll
    for (int c = 0; c < CH; ++c) acc[c] = __reduce_add_sync(0xffffffffu, acc[c]);
    if (lane < CH) {  // lane c requantises channel c0 + c
      const int mine = lane == 0 ? acc[0] : lane == 1 ? acc[1] : lane == 2 ? acc[2] : acc[3];
      a.h[(int64_t)img * N1 + myc] = (uint8_t)requant_u8(mine - corr1, bdiv1, mult1, a.zp1, a.lo1);
    }
#pragma unroll
    for (int j = 0; j < KV; ++j) cur[j] = nxt[j];
  }
  // ---- ticket: the last CTA to get here sees every other CTA's h rows (release: fence + atomic; acquire: fence)
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if constexpr (F32HEAD) {
    const float bias_n = lane < N2 ? __ldg(f.bias + lane) : 0.f;
    const auto w4 = [&](int n, int j) { return __ldg(reinterpret_cast<const float4*>(f.w) + (n * 32 + lane) * 4 + j); };
    for (int img = warp; img < a.b; img += 8) {
      const uint4 q = __ldcg(reinterpret_cast<const uint4*>(a.h + (int64_t)img * N1) + lane);  // written by other SMs: L2
      const float v = sandwich_head_image(q, lane, a.zp1, f.scale, bias_n, w4);
      if (lane < N2) a.logits[img * N2 + lane] = v;
    }
    if (tid == 0) *a.ticket = 0u;
    return;
  }
  const int nn = lane < N2 ? lane : 0;
  const int corr = __ldg(a.corr2 + nn);
  const float bdiv = __ldg(a.bdiv2 + nn), mult = __ldg(a.mult2 + nn);
  uint32_t cnt[5] = {0, 0, 0, 0, 0};
  for (int img = warp; img < a.b; img += 8) {
    const uint4 x = __ldcg(reinterpret_cast<const uint4*>(a.h + (int64_t)img * N1) + lane);  // written by other SMs: L2
    int mine = 0;
#pragma unroll
    for (int n = 0; n < N2; ++n) {
      int acc = dp4a_us(x.x, w2[n].x, 0);
      acc = dp4a_us(x.y, w2[n].y, acc);
      acc = dp4a_us(x.z, w2[n].z, acc);
      acc = dp4a_us(x.w, w2[n].w, acc);
      acc = __reduce_add_sync(0xffffffffu, acc);
      if (lane == n) mine = acc;
    }
    if (lane < N2) {
      const uint32_t q = requant_u8(mine - corr, bdiv, mult, a.zp2, a.lo2);
      if (!EVAL || a.logits != nullptr) a.logits[img * N2 + lane] = __fmul_rn(__int2float_rn((int)q - a.zp2), a.out_scale);
      if constexpr (EVAL) mine = (int)q;
    }
    if constexpr (EVAL) eval_image<N2>((uint32_t)mine, lane, img, ev, cnt);
  }
  if constexpr (EVAL) eval_flush(cnt, ev);
  if (tid == 0) *a.ticket = 0u;  // ready for the next forward on this workspace
}

// Returns 1 when the pair of layers / the batch is not the shape this kernel is written for.
int fc_head_small_dispatch(const uint8_t* x, uint8_t* h, float* logits, unsigned int* ticket, int64_t b,
                           const b200q_linear* fc1, const b200q_linear* fc2, float out_scale, const EvalArgs* eval,
                           cudaStream_t s, int* rc) {
  if (b < 1 || b > FC_SMALL_MAX_B || fc1->k != 4096 || fc1->n != 512 || fc2->k != 512 || fc2->n != 10) return 1;
  if ((uintptr_t)x % 16 || (uintptr_t)h % 16 || (uintptr_t)fc1->w % 16 || (uintptr_t)fc2->w % 16 || (uintptr_t)ticket % 4) return 1;
  FcSmallArgs a{x, h, logits, ticket, fc1->w, fc1->corr, fc1->rq.mult, fc1->rq.bdiv, fc2->w, fc2->corr, fc2->rq.mult,
                fc2->rq.bdiv, (int)b, fc1->rq.zp_out, fc1->rq.relu ? fc1->rq.zp_out : 0, fc2->rq.zp_out,
                fc2->rq.relu ? fc2->rq.zp_out : 0, out_scale};
  *rc = eval ? launch_kernel("fc_head_small_kernel", fc_head_small_kernel<true>, 512 / 4, 256, 0, s, a, *eval,
                            F32HeadArgs{})
             : launch_kernel("fc_head_small_kernel", fc_head_small_kernel<false>, 512 / 4, 256, 0, s, a, EvalArgs{},
                             F32HeadArgs{});
  return 0;
}

// Warps of the head kernel for b images: <= 8 blocks of 8 warps per SM.
static int head_blocks(int64_t b) {
  const int64_t warps = b < (int64_t)num_sms() * 64 ? b : (int64_t)num_sms() * 64;
  return (int)((warps + 7) / 8);
}

int sandwich_head_small_dispatch(const uint8_t* x, uint8_t* h, float* logits, unsigned int* ticket, int64_t b,
                                 const b200q_linear* fc1, const float* fc2_w, const float* fc2_b, float fc1_scale,
                                 cudaStream_t s, int* rc) {
  if (b < 1 || b > FC_SMALL_MAX_B || fc1->k != 4096 || fc1->n != 512) return 1;
  if ((uintptr_t)x % 16 || (uintptr_t)h % 16 || (uintptr_t)fc1->w % 16 || (uintptr_t)ticket % 4) return 1;
  FcSmallArgs a{x, h, logits, ticket, fc1->w, fc1->corr, fc1->rq.mult, fc1->rq.bdiv, nullptr, nullptr, nullptr, nullptr,
                (int)b, fc1->rq.zp_out, fc1->rq.relu ? fc1->rq.zp_out : 0, 0, 0, 0.f};
  *rc = launch_kernel("fc_head_small_kernel", fc_head_small_kernel<false, true>, 512 / 4, 256, 0, s, a, EvalArgs{},
                      F32HeadArgs{fc2_w, fc2_b, fc1_scale});
  return 0;
}

int sandwich_head(const uint8_t* x, float* logits, int64_t b, const float* fc2_w, const float* fc2_b, int zp,
                  float fc1_scale, cudaStream_t s) {
  if (b == 0) return 0;
  return launch_kernel("sandwich_head_kernel", sandwich_head_kernel, head_blocks(b), 256, 0, s, x, logits, b, fc2_w,
                       fc2_b, zp, fc1_scale);
}

int linear_head_eval(const uint8_t* x, float* logits, int64_t b, const b200q_linear* L, float out_scale,
                     const EvalArgs& eval, cudaStream_t s) {
  B200Q_REQUIRE(L->k == 512 && L->n == 10 && (uintptr_t)x % 16 == 0 && (uintptr_t)L->w % 16 == 0,
                "static_evaluate: the counting head needs fc2 k=512 n=10 and 16-byte aligned rows (k=%d n=%d)", L->k,
                L->n);
  if (b == 0) return 0;
  LinearArgs a{x, logits, L->w, L->corr, L->rq.mult, L->rq.bdiv, b, L->k, L->n, L->rq.zp_out, L->rq.relu, out_scale};
  return launch_kernel("linear_head_dequant_kernel", linear_head_dequant_kernel<10, true>, head_blocks(b), 256, 0, s, a,
                       eval);
}

template <int EPI>
static int launch_linear(const LinearArgs& a, cudaStream_t s) {
  dim3 grid((unsigned)((a.b + 63) / 64), (unsigned)((a.n + 63) / 64));
  linear_simt_kernel<EPI><<<grid, 256, 0, s>>>(a);
  return launched("linear_simt_kernel");
}

static int check_linear(const uint8_t* x, const void* y, int64_t b, const b200q_linear* L) {
  B200Q_REQUIRE(L && ((x && y) || b == 0), "linear: null pointer");
  B200Q_REQUIRE(L->k > 0 && L->k % 4 == 0 && L->n > 0, "linear: need k %% 4 == 0 (k=%d n=%d)", L->k, L->n);
  B200Q_REQUIRE(L->w && L->corr && L->rq.mult && L->rq.bdiv, "linear: unpacked layer");
  B200Q_REQUIRE((uintptr_t)x % 4 == 0 && (uintptr_t)L->w % 4 == 0, "linear: x and w must be 4-byte aligned");
  return 0;
}

}  // namespace b200q

using namespace b200q;

static int check_conv(const void* x, const void* y, int64_t b, const b200q_conv3x3* L) {
  B200Q_REQUIRE(L && ((x && y) || b == 0), "conv3x3: null pointer");
  B200Q_REQUIRE(L->w && L->corr && L->rq.mult && L->rq.bdiv, "conv3x3: unpacked layer");
  B200Q_REQUIRE(L->zp_x >= 0 && L->zp_x <= 255 && L->rq.zp_out >= 0 && L->rq.zp_out <= 255,
                "conv3x3: zero-point out of range");
  return 0;
}

// -DB200Q_DEV builds only: B200Q_CONV1_TINY_MAX_B overrides the cut-off (0 disables the shape; A-B timing only).
static int conv1_tiny_max_b() {
#ifndef B200Q_DEV
  return CONV1_TINY_MAX_B;
#endif
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200Q_CONV1_TINY_MAX_B");
    v = e ? atoi(e) : CONV1_TINY_MAX_B;
  }
  return v;
}

// kind: C1_IN_NHWC4 (x uint8 NHWC4), C1_IN_F32 (x fp32 NCHW, inv_scale) or C1_IN_U8 (x uint8 NHWC pixels, lut_host a HOST
// uint8[3][256] table).  The two raw-input kinds share the kernel selection: the CUDA-core shape for a few images, else
// the tensor-core kernel, else (layer without host mirrors / BOUNDED constants) the CUDA-core kernel for any batch.
static int conv_first_impl(const void* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, C1In kind, float inv_scale,
                           const uint8_t* lut_host, void* stream) {
  int rc = check_conv(x, y, b, L);
  if (rc) return rc;
  B200Q_REQUIRE(L->cin == 4 && L->cout == C1_COUT && L->img == 32,
                "conv3x3_first: geometry must be cin=3(padded 4), cout=64, img=32 (got %d,%d,%d)", L->cin, L->cout,
                L->img);
  B200Q_REQUIRE((uintptr_t)y % 16 == 0 && (uintptr_t)x % (kind == C1_IN_U8 ? 8 : 4) == 0,
                "conv3x3_first: misaligned buffers");
  if (b == 0) return 0;
  static const C1Lut kNoLut = {};
  C1Lut lut;
  if (kind == C1_IN_U8)
    for (int i = 0; i < 3 * 256; ++i) lut.q[i / 256][i % 256] = lut_host[i];
  const C1Lut& lut_arg = kind == C1_IN_U8 ? lut : kNoLut;
  const bool raw = kind != C1_IN_NHWC4;
  if (raw && b <= conv1_tiny_max_b()) {  // a few images: 16 CUDA-core CTAs per image, one round trip
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(b * (L->img / C1_ROWS)), 4);
    cfg.blockDim = dim3(256);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    if (pdl_enabled()) {
      attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
    }
    const cudaError_t e = cudaLaunchKernelEx(
        &cfg, kind == C1_IN_U8 ? conv1_kernel<C1_IN_U8, 1> : conv1_kernel<C1_IN_F32, 1>, x, y,
        reinterpret_cast<const uint32_t*>(L->w), L->corr, L->rq.mult, L->rq.bdiv, (int)L->zp_x, (int)L->rq.zp_out,
        (int)L->rq.relu, inv_scale, (int)L->img, lut_arg);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      return check_cuda(e, "conv1_kernel");
    }
    return launched("conv1_kernel");
  }
  if (raw) {  // tensor-core version unless the layer lacks host mirrors / the BOUNDED flag (dev builds: or B200Q_NO_CONV1_TC=1)
#ifdef B200Q_DEV
    static int no_tc = -1;
    if (no_tc < 0) {
      const char* e = getenv("B200Q_NO_CONV1_TC");
      no_tc = (e && e[0] == '1') ? 1 : 0;
    }
#else
    const int no_tc = 0;
#endif
    int trc = 0;
    const bool u8 = kind == C1_IN_U8;
    if (!no_tc && conv1_tc_dispatch(u8 ? nullptr : reinterpret_cast<const float*>(x),
                                    u8 ? reinterpret_cast<const uint8_t*>(x) : nullptr, u8 ? lut_host : nullptr, y, b,
                                    inv_scale, L, (cudaStream_t)stream, &trc) == 0)
      return trc;
  }
  const unsigned grid = (unsigned)(b * (L->img / C1_ROWS));
  const uint32_t* ww = reinterpret_cast<const uint32_t*>(L->w);
  void (*kernel)(const void*, uint8_t*, const uint32_t*, const int32_t*, const float*, const float*, int, int, int, float,
                 int, C1Lut) = kind == C1_IN_U8    ? conv1_kernel<C1_IN_U8, 4>
                               : kind == C1_IN_F32 ? conv1_kernel<C1_IN_F32, 4>
                                                   : conv1_kernel<C1_IN_NHWC4, 4>;
  kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, ww, L->corr, L->rq.mult, L->rq.bdiv, L->zp_x, L->rq.zp_out,
                                                 L->rq.relu, kind == C1_IN_F32 ? inv_scale : 0.f, L->img, lut_arg);
  return launched("conv1_kernel");
}

extern "C" int b200q_conv3x3_first(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, void* stream) {
  return conv_first_impl(x, y, b, L, C1_IN_NHWC4, 0.f, nullptr, stream);
}

extern "C" int b200q_quantize_conv3x3_first(const float* x, uint8_t* y, int64_t b, float inv_scale,
                                            const b200q_conv3x3* L, void* stream) {
  return conv_first_impl(x, y, b, L, C1_IN_F32, inv_scale, nullptr, stream);
}

extern "C" int b200q_u8_conv3x3_first(const uint8_t* x_nhwc, uint8_t* y, int64_t b, const uint8_t* lut_host,
                                      const b200q_conv3x3* L, void* stream) {
  B200Q_REQUIRE(lut_host != nullptr, "u8_conv3x3_first: null lut_host");
  return conv_first_impl(x_nhwc, y, b, L, C1_IN_U8, 0.f, lut_host, stream);
}

#ifdef B200Q_DEV
extern "C" int b200q_conv3x3_simt(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, void* stream) {
  int rc = check_conv(x, y, b, L);
  if (rc) return rc;
  B200Q_REQUIRE(L->cin % 4 == 0 && L->cout > 0 && L->img > 0, "conv3x3_simt: need cin %% 4 == 0");
  if (b == 0) return 0;
  const int64_t total = b * L->img * L->img * L->cout;
  int64_t blocks = (total + 255) / 256;
  if (blocks > (int64_t)num_sms() * 32) blocks = (int64_t)num_sms() * 32;
  conv3x3_direct_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      x, y, b, L->img, L->cin, L->cout, L->w, L->rq.mult, L->rq.bdiv, L->zp_x, L->rq.zp_out, L->rq.relu);
  return launched("conv3x3_direct_kernel");
}
#endif  // B200Q_DEV

extern "C" int b200q_linear_simt(const uint8_t* x, uint8_t* y, int64_t b, const b200q_linear* L, void* stream) {
  int rc = check_linear(x, y, b, L);
  if (rc) return rc;
  if (b == 0) return 0;
  LinearArgs a{x, y, L->w, L->corr, L->rq.mult, L->rq.bdiv, b, L->k, L->n, L->rq.zp_out, L->rq.relu, 0.f};
  return launch_linear<EPI_REQUANT_U8>(a, (cudaStream_t)stream);
}

extern "C" int b200q_linear_dequant(const uint8_t* x, float* y, int64_t b, const b200q_linear* L, float out_scale,
                                    void* stream) {
  int rc = check_linear(x, y, b, L);
  if (rc) return rc;
  if (b == 0) return 0;
  LinearArgs a{x, y, L->w, L->corr, L->rq.mult, L->rq.bdiv, b, L->k, L->n, L->rq.zp_out, L->rq.relu,
               out_scale};
  if (L->k == 512 && L->n == 10 && (uintptr_t)x % 16 == 0 && (uintptr_t)L->w % 16 == 0)
    return launch_kernel("linear_head_dequant_kernel", linear_head_dequant_kernel<10, false>, head_blocks(b), 256, 0,
                         (cudaStream_t)stream, a, EvalArgs{});
  return launch_linear<EPI_REQUANT_DEQUANT_F32>(a, (cudaStream_t)stream);
}
