// First layer on the tensor cores: fused aten::quantize_per_tensor + quantized 3x3 conv (cin=3) + ReLU.
//
//   fp32 NCHW [b,3,32,32]  ->  uint8 NHWC [b,32,32,64]
//
// K = 27 (9 taps x 3 channels) is padded to one 32-byte MMA K-step, so a tile of 128 output pixels needs ONE
// tcgen05.mma (M=128, N=64, K=32); the tensor-core time is negligible and the layer is bound by its epilogue (64
// requantised channels per pixel) and by the 77.8 KB/image it moves through HBM.  What the CUDA-core version
// (simt.cu) spent on 576 dp4a + 128 conversion-pipe instructions per pixel is gone.
//
// Roles (384 threads): warps 0..7 epilogue (epilogue16.cuh, same scheme as conv_halo.cu: 8x16-pixel block tiles,
// pre-biased accumulators, two sets of four warps taking alternate tiles, software-pipelined over the tiles), warps
// 8..11 producers.  There is no MMA warp: the first producer warp issues the image's eight MMAs right after the im2col
// rows are complete, so the CTA has 12 warps = 3 per scheduler and 168 registers per thread, which the pipelined
// epilogue (two accumulator halves + 48 constants in registers) needs.  The eight TMEM slots hold one whole image
// (slot = tile), so that warp only ever waits for the epilogue of the previous image.
// Producers, per image: (1) quantise the fp32 planes (exact aten arithmetic, without the conversion pipe) into a
// padded 34x34 image of {c0,c1,c2,zp} words whose border holds the zero-point; (2) gather the im2col rows
// [pixel][tap*3+ch] (27 bytes + 5 zero bytes) with byte permutes and store them tile-major in the 32-byte-swizzled
// K-major layout the MMA reads.  Because the pads hold the zero-point, the zero-point correction is one constant per
// output channel.
#include <type_traits>

#include "common.cuh"
#include "epilogue16.cuh"

namespace b200q {

constexpr int C1_EPI_WARPS = 8, C1_PROD_WARPS = 4;
constexpr int C1_SETS = C1_EPI_WARPS / 4;
constexpr int C1_PROD_WARP0 = C1_EPI_WARPS;
constexpr int C1_THREADS = 32 * (C1_EPI_WARPS + C1_PROD_WARPS);
constexpr int C1_SLOTS = 8;
constexpr int C1_IMG = 32, C1_COUT = 64, C1_KB = 32;       // K bytes per row
constexpr int C1_TILES = 8;                                  // 2 x 4 blocks of 16 rows x 8 columns
constexpr int C1_A_TILE = 128 * C1_KB, C1_A_BYTES = C1_TILES * C1_A_TILE;  // 4 KB, 32 KB
constexpr int C1_B_BYTES = C1_COUT * C1_KB;
constexpr int C1_QP = C1_IMG + 2;                            // padded quantised image pitch (words)
constexpr int C1_Q_BYTES = (C1_QP * C1_QP * 4 + 15) / 16 * 16;
constexpr int C1_LUT_BYTES = 3 * 256;
constexpr int C1_SMEM = 2 * C1_A_BYTES + C1_B_BYTES + C1_Q_BYTES + 256 + C1_LUT_BYTES + 1024;

struct C1Args {
  const float* x;
  const uint8_t* xu8;  // uint8 NHWC [b,32,32,3] (U8IN kernels), else null
  uint8_t* y;
  const int8_t* w;     // [64][9][4] (cin padded to 4), device
  int64_t n_img;
  float inv_scale;
  int zp_x, zp_out, lo, bounded;
};

struct alignas(16) C1Consts {
  int32_t cm[C1_COUT];
  float k1[C1_COUT];
  float bdiv[C1_COUT];
  float mult[C1_COUT];
};

// aten::quantize_per_tensor without I2F/F2I: clamp(rne(x * inv_scale) + zp, 0, 255); identical to quantize_u8 because the
// product is clamped to +-1024 before the round-to-nearest-even add.
__device__ __forceinline__ uint32_t quantize_magic(float x, float inv_scale, int zp_sub) {
  float t = __fmul_rn(x, inv_scale);
  t = fminf(fmaxf(t, -1024.0f), 1024.0f);
  const int q = __float_as_int(__fadd_rn(t, MAGIC_F)) + zp_sub;  // zp_sub = zp - MAGIC_BITS
  return (uint32_t)max(0, min(q, 255));
}

template <bool CHECK, bool U8IN>
__global__ void __launch_bounds__(C1_THREADS, 1)
conv1_tc_kernel(const __grid_constant__ C1Consts consts, const __grid_constant__ C1Lut lut, const C1Args args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* a_smem = smem;                                   // [2][8 tiles][128 rows][32 B]
  uint8_t* b_smem = a_smem + 2 * C1_A_BYTES;                // [64][32 B]
  uint32_t* q_img = reinterpret_cast<uint32_t*>(b_smem + C1_B_BYTES);  // [34][34] words {c0,c1,c2,zp}
  uint64_t* empty_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(q_img) + C1_Q_BYTES);  // [2]
  uint64_t* tmem_full_bar = empty_bar + 2;                  // [C1_SLOTS]
  uint64_t* tmem_empty_bar = tmem_full_bar + C1_SLOTS;      // [C1_SLOTS]
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + C1_SLOTS);
  uint32_t* magic_smem = tmem_base_smem + 1;  // holds MAGIC_BITS (epilogue16.cuh epi_init)
  uint8_t* lut_smem = reinterpret_cast<uint8_t*>(empty_bar) + 256;  // [3][256] (U8IN)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t zp4 = (uint32_t)args.zp_x * 0x01010101u;
  pdl_launch_dependents();

  if (warp == C1_PROD_WARP0 && lane == 0) {
    *magic_smem = MAGIC_BITS;
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
      for (int i = t; i < C1_LUT_BYTES / 4; i += 32 * C1_EPI_WARPS)
        reinterpret_cast<uint32_t*>(lut_smem)[i] = reinterpret_cast<const uint32_t*>(&lut.q[0][0])[i];
    }
    // border of the quantised image = zero-point, once
    for (int i = t; i < C1_QP * C1_QP; i += 32 * C1_EPI_WARPS) {
      const int r = i / C1_QP, c = i % C1_QP;
      if (r == 0 || r == C1_QP - 1 || c == 0 || c == C1_QP - 1) q_img[i] = zp4;
    }
    // weights [64][9][4] -> B operand [64][k = tap*3 + ch] (32-byte rows, SWIZZLE_32B), zero for k >= 27; row nr holds
    // output channel epi_channel_of_column<16>(nr) (the epilogue's thread <-> channel assignment)
    for (int i = t; i < C1_COUT * (C1_KB / 4); i += 32 * C1_EPI_WARPS) {
      const int nr = i / (C1_KB / 4), wd = i % (C1_KB / 4);
      const int n = epi_channel_of_column<16>(nr);
      uint32_t word = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int k = wd * 4 + b;
        if (k < 27) word |= (uint32_t)(uint8_t)__ldg(args.w + (n * 9 + k / 3) * 4 + k % 3) << (8 * b);
      }
      const int chunk = (wd >> 2) ^ ((nr >> 2) & 1);
      *reinterpret_cast<uint32_t*>(b_smem + nr * C1_KB + chunk * 16 + (wd & 3) * 4) = word;
    }
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;
  if (warp < 4) {  // pre-bias every accumulator slot (see requant4_prebiased)
    const uint32_t base = tmem_base + ((uint32_t)(warp * 32) << 16);
    for (int slot = 0; slot < C1_SLOTS; ++slot)
      for (int c = 0; c < C1_COUT; c += 8) tmem_st_fill8(base + slot * C1_COUT + c, MAGIC_BITS);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const int my_imgs = ((int64_t)blockIdx.x < args.n_img) ? (int)((args.n_img - 1 - blockIdx.x) / gridDim.x + 1) : 0;

  if (warp >= C1_PROD_WARP0) {
    // ================================================================== producers (128 threads)
    const int p = threadIdx.x - 32 * C1_PROD_WARP0;
    const int zp_sub = args.zp_x - (int)MAGIC_BITS;
    const uint32_t zp_hi = (uint32_t)args.zp_x << 24;
    const bool leader = elect_one() != 0;
    constexpr uint32_t idesc = make_idesc_i8(128, C1_COUT);
    const uint64_t b_desc = make_kmajor_desc<C1_KB>(smem_u32(b_smem), 8 * C1_KB);
    // thread p owns image row p/4, columns 8*(p%4) .. +7 of the fp32 planes.  The loads of image it+1 are issued right
    // after image it has been quantised, so their HBM latency overlaps the im2col pass and the barrier waits.
    const int row = p >> 2, col0 = (p & 3) * 8;
    float4 v[3][2];   // fp32 input: three planes x 8 pixels
    uint2 u[3];       // uint8 NHWC input: 8 pixels x 3 bytes = 24 contiguous bytes
    auto load_image = [&](int it) {
      const int64_t img = (int64_t)blockIdx.x + (int64_t)it * gridDim.x;
      if constexpr (U8IN) {
        const uint8_t* src = args.xu8 + img * (3 * C1_IMG * C1_IMG) + (row * C1_IMG + col0) * 3;
#pragma unroll
        for (int i = 0; i < 3; ++i) u[i] = __ldg(reinterpret_cast<const uint2*>(src) + i);
      } else {
        const float* src = args.x + img * (3 * C1_IMG * C1_IMG) + row * C1_IMG + col0;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          v[ch][0] = __ldg(reinterpret_cast<const float4*>(src + ch * C1_IMG * C1_IMG));
          v[ch][1] = __ldg(reinterpret_cast<const float4*>(src + ch * C1_IMG * C1_IMG) + 1);
        }
      }
    };
    pdl_wait();  // first access to memory another kernel of the stream may own
    if (my_imgs > 0) load_image(0);
    for (int it = 0; it < my_imgs; ++it) {
      const int buf = it & 1;
      // ---- (1) quantise
      if constexpr (U8IN) {
        uint32_t* dst = q_img + (row + 1) * C1_QP + col0 + 1;
        const uint32_t wds[6] = {u[0].x, u[0].y, u[1].x, u[1].y, u[2].x, u[2].y};
#pragma unroll
        for (int j = 0; j < 8; ++j) {  // pixel j = bytes 3j, 3j+1, 3j+2 of the 24
          uint32_t word = zp_hi;
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            const int byte = 3 * j + ch;
            const uint32_t pix = (wds[byte >> 2] >> (8 * (byte & 3))) & 0xffu;
            word |= (uint32_t)lut_smem[ch * 256 + pix] << (8 * ch);
          }
          dst[j] = word;
        }
      } else {
        uint32_t* dst = q_img + (row + 1) * C1_QP + col0 + 1;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float c0[4] = {v[0][h].x, v[0][h].y, v[0][h].z, v[0][h].w};
          const float c1[4] = {v[1][h].x, v[1][h].y, v[1][h].z, v[1][h].w};
          const float c2[4] = {v[2][h].x, v[2][h].y, v[2][h].z, v[2][h].w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
            dst[h * 4 + j] = quantize_magic(c0[j], args.inv_scale, zp_sub) |
                             (quantize_magic(c1[j], args.inv_scale, zp_sub) << 8) |
                             (quantize_magic(c2[j], args.inv_scale, zp_sub) << 16) | zp_hi;
        }
      }
      if (it + 1 < my_imgs) load_image(it + 1);
      asm volatile("bar.sync 2, %0;" ::"n"(32 * C1_PROD_WARPS) : "memory");
      // ---- (2) im2col rows: thread p builds row p of every tile; tile i = block (i/4, i%4), row p = pixel (p/8, p%8)
      mbar_wait(empty_bar + buf, ((it >> 1) & 1) ^ 1);
      uint8_t* a_buf = a_smem + buf * C1_A_BYTES;
#pragma unroll 2
      for (int i = 0; i < C1_TILES; ++i) {
        const int r = (i >> 2) * 16 + (p >> 3), c = (i & 3) * 8 + (p & 7);
        const uint32_t* q = q_img + r * C1_QP + c;  // tap (0,0) = pixel (r-1, c-1) = padded (r, c)
        const uint32_t s0 = q[0], s1 = q[1], s2 = q[2];
        const uint32_t s3 = q[C1_QP], s4 = q[C1_QP + 1], s5 = q[C1_QP + 2];
        const uint32_t s6 = q[2 * C1_QP], s7 = q[2 * C1_QP + 1], s8 = q[2 * C1_QP + 2];
        // 27 bytes: tap-major, 3 channels each; byte 3 of every source word (the zp filler) is dropped
        const uint4 lo4 = make_uint4(__byte_perm(s0, s1, 0x4210), __byte_perm(s1, s2, 0x5421),
                                     __byte_perm(s2, s3, 0x6542), __byte_perm(s4, s5, 0x4210));
        const uint4 hi4 = make_uint4(__byte_perm(s5, s6, 0x5421), __byte_perm(s6, s7, 0x6542), s8 & 0x00ffffffu, 0u);
        const int sw = (p >> 2) & 1;  // SWIZZLE_32B: 16-byte chunk index ^= address bit 7
        uint8_t* rowp = a_buf + i * C1_A_TILE + p * C1_KB;
        *reinterpret_cast<uint4*>(rowp + (sw << 4)) = lo4;
        *reinterpret_cast<uint4*>(rowp + ((sw ^ 1) << 4)) = hi4;
      }
      fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's async-proxy reads
      asm volatile("bar.sync 2, %0;" ::"n"(32 * C1_PROD_WARPS) : "memory");  // a_buf complete; q_img free again
      // ---- (3) the first producer warp issues the image's MMAs: one per tile, slot = tile
      if (warp == C1_PROD_WARP0) {
        tc_fence_after();
        const uint64_t a_desc0 = make_kmajor_desc<C1_KB>(smem_u32(a_buf), 8 * C1_KB);
        for (int t = 0; t < C1_TILES; ++t) {
          mbar_wait(tmem_empty_bar + t, (it & 1) ^ 1);  // drained by the epilogue of the previous image
          tc_fence_after();
          if (leader) {
            tc_mma_i8(tmem_base + t * C1_COUT, a_desc0 + (uint64_t)((t * C1_A_TILE) >> 4), b_desc, idesc, 1u);
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
    const bool fast = args.bounded != 0;
    EpiRegs<16> K;
    epi_init(consts, ch0, magic_smem, K);
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
    epi_pipeline<CHECK>(K, consts, ch0, fast, args.zp_out, args.lo, (int64_t)C1_IMG * C1_COUT, 2 * (int64_t)C1_IMG * C1_COUT,
                        lane, next);
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
  for (int c = 0; c < C1_COUT; ++c) {
    const int32_t corr = L->corr_host[4 * C1_COUT + c];  // class 4 = all nine taps (pads hold the zero-point)
    consts.cm[c] = (int32_t)(MAGIC_BITS - (uint32_t)corr);
    consts.k1[c] = -(MAGIC_F + (float)corr);
    consts.bdiv[c] = rq.bdiv_host[c];
    consts.mult[c] = rq.mult_host[c];
  }
  C1Lut lut;
  const bool u8in = lut_host != nullptr;
  if (u8in)
    for (int i = 0; i < 3 * 256; ++i) lut.q[i / 256][i % 256] = lut_host[i];
  else
    for (int i = 0; i < 3 * 256; ++i) lut.q[i / 256][i % 256] = 0;
  const bool check = !(rq.flags & B200Q_RQ_ACC22);
  void (*kernel)(C1Consts, C1Lut, C1Args) =
      u8in ? (check ? conv1_tc_kernel<true, true> : conv1_tc_kernel<false, true>)
           : (check ? conv1_tc_kernel<true, false> : conv1_tc_kernel<false, false>);
  static uint64_t attr_mask[4] = {0, 0, 0, 0};
  const int idx = (u8in ? 2 : 0) + (check ? 1 : 0);
  *rc = ensure_dynamic_smem(reinterpret_cast<const void*>(kernel), C1_SMEM, &attr_mask[idx]);
  if (*rc) return 0;
  C1Args args{x, xu8, y, L->w, b, inv_scale, L->zp_x, rq.zp_out, rq.relu ? rq.zp_out : 0, 1};
  const int grid = b < num_sms() ? (int)b : num_sms();
  *rc = launch_kernel("conv1_tc_kernel", kernel, grid, C1_THREADS, C1_SMEM, s, consts, lut, args);
  return 0;
}

}  // namespace b200q

