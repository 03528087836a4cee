// First layer on the tensor cores: fused aten::quantize_per_tensor + quantized 3x3 conv (cin=3) + ReLU.
//
//   fp32 NCHW [b,3,32,32]  ->  uint8 NHWC [b,32,32,64]
//
// The MMAs run on fp16 operands (x - zp_x) and w with an fp32 accumulator (kind::f16).  Both operands are integers
// that fp16 holds exactly (|x - zp| <= 255, |w| <= 128), every product is an integer below 2^15 and every partial sum
// of the 27 taps an integer below 27 * 255 * 128 < 2^20, so the accumulator is exact in any summation order: it IS
// f32(acc - corr), the value fbgemm's requantisation starts from (tools/probe_f16_intacc.cu checks this on the
// hardware).  That removes, against an int8 MMA on x with a pre-biased accumulator: the re-arming tcgen05.st after every
// tile, the per-channel zero-point correction (one FADD per value) and, because the pads are now 0 instead of zp, any
// border handling.
//
// A operand: per image 34 rows x 32 pixels of 32-byte K-rows, fp16 [x(r, c-1) x4ch, x(r, c) x4ch, x(r, c+1) x4ch, 0 x4]
// (channel 3 and the last four lanes zero), SWIZZLE_32B K-major; rows 0 and 33 are the zero pad rows.  A tile is 16
// image rows x 8 columns (accumulator row = 8*image_row + column, descriptor SBO = one image row = 1 KB); tap row kh is
// the same buffer with the start address moved down kh rows, and kw x channel is the K = 16 of one MMA, so a tile is
// three MMAs (M=128, N=64, K=16) whose B operands are the weights of kernel rows 0, 1, 2.
//
// Roles (384 threads): warps 0..7 epilogue (epilogue16.cuh epi_pipeline<F32ACC>: 8x16-pixel block tiles, two sets of
// four warps taking alternate tiles, software-pipelined over the tiles), warps 8..11 producers.  There is no MMA warp:
// the first producer warp issues the image's 24 MMAs once the rows are complete, so the CTA has 12 warps = 3 per
// scheduler and 168 registers per thread.  The eight TMEM slots hold one whole image (slot = tile).
// Producers, per image: lane = image column, producer warp w owns image rows w, w+4, .., w+28; quantise (exact aten
// arithmetic, without the conversion pipe) to fp16 x - zp with the 0x6400 | q bit pattern (1024 + q) and one HADD2,
// take the left / right neighbours from lanes -1 / +1 by shuffle (0 beyond the image), and store each pixel's K-row.
#include <cuda_fp16.h>

#include "common.cuh"
#include "epilogue16.cuh"

namespace b200q {

constexpr int C1_EPI_WARPS = 8, C1_PROD_WARPS = 4;
constexpr int C1_SETS = C1_EPI_WARPS / 4;
constexpr int C1_PROD_WARP0 = C1_EPI_WARPS;
constexpr int C1_THREADS = 32 * (C1_EPI_WARPS + C1_PROD_WARPS);
constexpr int C1_SLOTS = 8;
constexpr int C1_IMG = 32, C1_COUT = 64, C1_KB = 32;         // K bytes per row (16 fp16)
constexpr int C1_TILES = 8;                                    // 2 x 4 blocks of 16 rows x 8 columns
constexpr int C1_ROWS_PER_PROD = C1_IMG / C1_PROD_WARPS;       // 8 image rows per producer thread
constexpr int C1_ROW_BYTES = C1_IMG * C1_KB;                   // 1 KB: one image row of K-rows = descriptor SBO
constexpr int C1_A_BYTES = (C1_IMG + 2) * C1_ROW_BYTES;        // 34 KB: pad row, 32 image rows, pad row
constexpr int C1_B_TAP = C1_COUT * C1_KB;                      // 2 KB per kernel row kh
constexpr int C1_B_BYTES = 3 * C1_B_TAP;
constexpr int C1_LUT_BYTES = 3 * 256 * 2;                      // fp16 (q - zp) per channel and pixel value (U8IN)
constexpr int C1_SMEM = 2 * C1_A_BYTES + C1_B_BYTES + 256 + C1_LUT_BYTES + 1024;
// Exactness of the fp32 accumulator: 27 products of |w| <= 128 and |x - zp| <= max(zp, 255 - zp) <= 255, every partial
// sum an integer below 2^24, whatever the weights and zero-point.
static_assert(27 * 128 * 255 < (1 << 24), "conv1 partial sums must be exact in fp32");

struct C1Args {
  const float* x;
  const uint8_t* xu8;  // uint8 NHWC [b,32,32,3] (U8IN kernels), else null
  uint8_t* y;
  const int8_t* w;     // [64][9][4] (cin padded to 4), device
  int64_t n_img;
  float inv_scale;
  int zp_x, zp_out, lo;
};

struct alignas(16) C1Consts {
  float bdiv[C1_COUT];
  float mult[C1_COUT];
};

__device__ __forceinline__ uint32_t hadd2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("add.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}

// aten::quantize_per_tensor without I2F/F2I: q = clamp(rne(x * inv_scale) + zp, 0, 255); identical to quantize_u8
// because the product is clamped to +-1024 before the round-to-nearest-even add.  Returns q | 0x6400, the fp16 bit
// pattern of 1024 + q.
__device__ __forceinline__ uint32_t quantize_h1024(float x, float inv_scale, int zp_sub) {
  float t = __fmul_rn(x, inv_scale);
  t = fminf(fmaxf(t, -1024.0f), 1024.0f);
  const int q = __float_as_int(__fadd_rn(t, MAGIC_F)) + zp_sub;  // zp_sub = zp - MAGIC_BITS
  return (uint32_t)max(0, min(q, 255)) | 0x6400u;
}

// CHECK is the accumulator range test of the int8 kernels and is always false here (the fp32 accumulator is exact); the
// parameter keeps the kernel's name, conv1_tc_kernel<false, U8IN>, what traces and tests match.
template <bool CHECK, bool U8IN>
__global__ void __launch_bounds__(C1_THREADS, 1)
conv1_tc_kernel(const __grid_constant__ C1Consts consts, const __grid_constant__ C1Lut lut, const C1Args args) {
  static_assert(!CHECK, "conv1's fp32 accumulator needs no range test");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* a_smem = smem;                                   // [2][34 rows][32 pixels][32 B]
  uint8_t* b_smem = a_smem + 2 * C1_A_BYTES;                // [3 kh][64][32 B]
  uint64_t* empty_bar = reinterpret_cast<uint64_t*>(b_smem + C1_B_BYTES);  // [2]
  uint64_t* tmem_full_bar = empty_bar + 2;                  // [C1_SLOTS]
  uint64_t* tmem_empty_bar = tmem_full_bar + C1_SLOTS;      // [C1_SLOTS]
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + C1_SLOTS);
  uint16_t* lut_smem = reinterpret_cast<uint16_t*>(reinterpret_cast<uint8_t*>(empty_bar) + 256);  // [3][256] (U8IN)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();

  if (warp == C1_PROD_WARP0 && lane == 0) {
    for (int i = 0; i < 2; ++i) mbar_init(empty_bar + i, 1);
    for (int i = 0; i < C1_SLOTS; ++i) {
      mbar_init(tmem_full_bar + i, 1);
      mbar_init(tmem_empty_bar + i, 4);  // the four warps of the set that drains this slot (slot = tile)
    }
    fence_barrier_init();
  }
  if (warp == C1_PROD_WARP0) {
    tmem_alloc(tmem_base_smem, C1_SLOTS * C1_COUT);
    tmem_relinquish();
  }
  if (warp < C1_EPI_WARPS) {
    const int t = threadIdx.x;
    if constexpr (U8IN) {
      for (int i = t; i < 3 * 256; i += 32 * C1_EPI_WARPS)
        lut_smem[i] = __half_as_ushort(__int2half_rn((int)lut.q[i / 256][i % 256] - args.zp_x));
    }
    // the pad rows (0 and 33) of both buffers: real-domain zero = 0, once
    for (int i = t; i < 2 * 2 * C1_ROW_BYTES / 16; i += 32 * C1_EPI_WARPS) {
      const int buf = i / (2 * C1_ROW_BYTES / 16), r = (i / (C1_ROW_BYTES / 16)) & 1, o = i % (C1_ROW_BYTES / 16);
      *reinterpret_cast<uint4*>(a_smem + buf * C1_A_BYTES + r * (C1_IMG + 1) * C1_ROW_BYTES + o * 16) =
          make_uint4(0u, 0u, 0u, 0u);
    }
    // weights [64][9][4] -> B operand of kernel row kh: [64][k = kw*4 + ch] fp16 (32-byte rows, SWIZZLE_32B), zero for
    // ch = 3 and kw = 3; row nr holds output channel epi_channel_of_column<16>(nr) (the epilogue's thread <-> channel
    // assignment)
    for (int i = t; i < 3 * C1_COUT * (C1_KB / 4); i += 32 * C1_EPI_WARPS) {
      const int kh = i / (C1_COUT * (C1_KB / 4)), nr = (i / (C1_KB / 4)) % C1_COUT, wd = i % (C1_KB / 4);
      const int n = epi_channel_of_column<16>(nr);
      uint32_t word = 0;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int k = wd * 2 + e, kw = k >> 2, ch = k & 3;
        if (kw < 3 && ch < 3)
          word |= (uint32_t)__half_as_ushort(__int2half_rn((int)__ldg(args.w + (n * 9 + kh * 3 + kw) * 4 + ch))) << (16 * e);
      }
      const uint32_t lin = nr * C1_KB + wd * 4;
      *reinterpret_cast<uint32_t*>(b_smem + kh * C1_B_TAP + (lin ^ (((lin >> 7) & 1) << 4))) = word;
    }
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;

  const int my_imgs = ((int64_t)blockIdx.x < args.n_img) ? (int)((args.n_img - 1 - blockIdx.x) / gridDim.x + 1) : 0;

  if (warp >= C1_PROD_WARP0) {
    // ================================================================== producers (128 threads)
    const int pw = warp - C1_PROD_WARP0;
    const int zp_sub = args.zp_x - (int)MAGIC_BITS;
    const uint32_t hneg = 0xE400u | (uint32_t)args.zp_x;  // fp16 -(1024 + zp): 1024 <= 1024 + zp < 2048, ulp 1
    const uint32_t hneg01 = hneg | (hneg << 16);
    const bool leader = elect_one() != 0;
    constexpr uint32_t idesc = make_idesc_f16(128, C1_COUT);
    const uint64_t b_desc0 = make_kmajor_desc<C1_KB>(smem_u32(b_smem), 8 * C1_KB);
    // The loads of image it+1 are issued right after image it has been quantised, so their HBM latency overlaps the
    // row stores and the barrier waits.  Row i of the thread is image row pw + 4i, column lane (coalesced 128-byte
    // rows of each fp32 plane; 96-byte rows of uint8 NHWC).
    float v[C1_ROWS_PER_PROD][3];
    uint32_t u[C1_ROWS_PER_PROD][3];
    auto load_image = [&](int it) {
      const int64_t img = (int64_t)blockIdx.x + (int64_t)it * gridDim.x;
#pragma unroll
      for (int i = 0; i < C1_ROWS_PER_PROD; ++i) {
        const int r = pw + C1_PROD_WARPS * i;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          if constexpr (U8IN)
            u[i][ch] = __ldg(args.xu8 + img * (3 * C1_IMG * C1_IMG) + (r * C1_IMG + lane) * 3 + ch);
          else
            v[i][ch] = __ldg(args.x + img * (3 * C1_IMG * C1_IMG) + ch * C1_IMG * C1_IMG + r * C1_IMG + lane);
        }
      }
    };
    pdl_wait();  // first access to memory another kernel of the stream may own
    if (my_imgs > 0) load_image(0);
    const int sw = (lane >> 2) & 1;  // SWIZZLE_32B: 16-byte chunk index ^= address bit 7 (pixel bit 2)
    for (int it = 0; it < my_imgs; ++it) {
      const int buf = it & 1;
      // ---- (1) quantise: own pixel = fp16 {c0, c1} {c2, 0}
      uint32_t px[C1_ROWS_PER_PROD][2];
#pragma unroll
      for (int i = 0; i < C1_ROWS_PER_PROD; ++i) {
        if constexpr (U8IN) {
          px[i][0] = (uint32_t)lut_smem[u[i][0]] | ((uint32_t)lut_smem[256 + u[i][1]] << 16);
          px[i][1] = lut_smem[512 + u[i][2]];
        } else {
          const uint32_t q0 = quantize_h1024(v[i][0], args.inv_scale, zp_sub);
          const uint32_t q1 = quantize_h1024(v[i][1], args.inv_scale, zp_sub);
          const uint32_t q2 = quantize_h1024(v[i][2], args.inv_scale, zp_sub);
          px[i][0] = hadd2(q0 | (q1 << 16), hneg01);
          px[i][1] = hadd2(q2, hneg);  // upper half: +0 + +0
        }
      }
      if (it + 1 < my_imgs) load_image(it + 1);
      // ---- (2) K-rows [left, own, right, 0] of the thread's eight pixels
      mbar_wait(empty_bar + buf, ((it >> 1) & 1) ^ 1);
      uint8_t* a_buf = a_smem + buf * C1_A_BYTES;
#pragma unroll
      for (int i = 0; i < C1_ROWS_PER_PROD; ++i) {
        uint32_t l0 = __shfl_up_sync(0xffffffffu, px[i][0], 1), l1 = __shfl_up_sync(0xffffffffu, px[i][1], 1);
        uint32_t r0 = __shfl_down_sync(0xffffffffu, px[i][0], 1), r1 = __shfl_down_sync(0xffffffffu, px[i][1], 1);
        if (lane == 0) l0 = l1 = 0u;
        if (lane == 31) r0 = r1 = 0u;
        uint8_t* rowp = a_buf + (pw + C1_PROD_WARPS * i + 1) * C1_ROW_BYTES + lane * C1_KB;
        *reinterpret_cast<uint4*>(rowp + (sw << 4)) = make_uint4(l0, l1, px[i][0], px[i][1]);
        *reinterpret_cast<uint4*>(rowp + ((sw ^ 1) << 4)) = make_uint4(r0, r1, 0u, 0u);
      }
      fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's async-proxy reads
      asm volatile("bar.sync 2, %0;" ::"n"(32 * C1_PROD_WARPS) : "memory");  // a_buf complete
      // ---- (3) the first producer warp issues the image's MMAs: three per tile (kernel rows), slot = tile
      if (warp == C1_PROD_WARP0) {
        tc_fence_after();
        const uint64_t a_desc0 = make_kmajor_desc<C1_KB>(smem_u32(a_buf), C1_ROW_BYTES);
        for (int t = 0; t < C1_TILES; ++t) {
          mbar_wait(tmem_empty_bar + t, (it & 1) ^ 1);  // drained by the epilogue of the previous image
          tc_fence_after();
          if (leader) {
            // tile t = image rows 16*(t/4) .., columns 8*(t%4) ..; tap row kh starts kh buffer rows further down
            const uint32_t a_off = (uint32_t)((t >> 2) * 16 * C1_ROW_BYTES + (t & 3) * 8 * C1_KB);
#pragma unroll
            for (int kh = 0; kh < 3; ++kh)
              tc_mma_f16(tmem_base + t * C1_COUT, a_desc0 + ((a_off + kh * C1_ROW_BYTES) >> 4),
                         b_desc0 + ((uint32_t)(kh * C1_B_TAP) >> 4), idesc, kh > 0 ? 1u : 0u);
            tc_commit(tmem_full_bar + t);
          }
          __syncwarp();
        }
        if (leader) tc_commit(empty_bar + buf);  // a_buf reusable once these MMAs have read it
        __syncwarp();
      }
    }
  } else {
    // ================================================================== epilogue warps (independent of each other)
    static_assert(C1_SLOTS == C1_TILES && C1_TILES % C1_SETS == 0, "slot = tile of the image");
    const int quarter = warp & 3;
    const int set = warp >> 2;                 // takes the tiles t with t % C1_SETS == set
    const int j = lane >> 2;                   // column of the 8-column block
    const int ch0 = 16 * (lane & 3);
    // bdiv / mult of the thread's 16 channels, pinned in registers through a self-shuffle (see epi_init)
    EpiRegs<16> K;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      K.bd[k] = __shfl_sync(0xffffffffu, consts.bdiv[ch0 + k], lane);
      K.mu[k] = __shfl_sync(0xffffffffu, consts.mult[ch0 + k], lane);
    }
    int it = 0, t = set;
    auto next = [&](EpiTile& e) -> bool {
      if (t >= C1_TILES) {
        t = set;
        ++it;
      }
      if (it >= my_imgs) return false;
      const int64_t img = (int64_t)blockIdx.x + (int64_t)it * gridDim.x;
      const int r0 = (t >> 2) * 16 + 4 * quarter, c = (t & 3) * 8 + j;
      e.t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + t * C1_COUT;
      e.full_bar = tmem_full_bar + t;
      e.empty_bar = tmem_empty_bar + t;
      e.parity = it & 1;
      e.out = args.y + ((img * C1_IMG + r0) * C1_IMG + c) * (int64_t)C1_COUT + ch0;
      e.valid0 = e.valid1 = true;
      t += C1_SETS;
      return true;
    };
    epi_pipeline<false, 16, true>(K, consts, ch0, true, args.zp_out, args.lo, (int64_t)C1_IMG * C1_COUT,
                                  2 * (int64_t)C1_IMG * C1_COUT, lane, next);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == C1_PROD_WARP0) {
    __syncwarp();
    tmem_dealloc(tmem_base, C1_SLOTS * C1_COUT);
  }
}

// x: fp32 NCHW input (lut_host == nullptr) or, with lut_host = uint8[3][256] on the HOST, xu8: uint8 NHWC input.
// Returns 1 when the layer cannot take this path (no host mirrors / constants not flagged as bounded).
int conv1_tc_dispatch(const float* x, const uint8_t* xu8, const uint8_t* lut_host, uint8_t* y, int64_t b,
                      float inv_scale, const b200q_conv3x3* L, cudaStream_t s, int* rc) {
  const b200q_requant& rq = L->rq;
  if (!L->corr_host || !rq.mult_host || !rq.bdiv_host || !(rq.flags & B200Q_RQ_BOUNDED)) return 1;
  if (L->cin != 4 || L->cout != C1_COUT || L->img != C1_IMG) return 1;
  C1Consts consts;
  for (int c = 0; c < C1_COUT; ++c) {  // no zero-point correction: the MMAs run on x - zp (pads 0)
    consts.bdiv[c] = rq.bdiv_host[c];
    consts.mult[c] = rq.mult_host[c];
  }
  C1Lut lut;
  const bool u8in = lut_host != nullptr;
  if (u8in)
    for (int i = 0; i < 3 * 256; ++i) lut.q[i / 256][i % 256] = lut_host[i];
  else
    for (int i = 0; i < 3 * 256; ++i) lut.q[i / 256][i % 256] = 0;
  void (*kernel)(C1Consts, C1Lut, C1Args) = u8in ? conv1_tc_kernel<false, true> : conv1_tc_kernel<false, false>;
  static uint64_t attr_mask[2] = {0, 0};
  *rc = ensure_dynamic_smem(reinterpret_cast<const void*>(kernel), C1_SMEM, &attr_mask[u8in ? 1 : 0]);
  if (*rc) return 0;
  C1Args args{x, xu8, y, L->w, b, inv_scale, L->zp_x, rq.zp_out, rq.relu ? rq.zp_out : 0};
  const int grid = b < num_sms() ? (int)b : num_sms();
  *rc = launch_kernel("conv1_tc_kernel", kernel, grid, C1_THREADS, C1_SMEM, s, consts, lut, args);
  return 0;
}

}  // namespace b200q

