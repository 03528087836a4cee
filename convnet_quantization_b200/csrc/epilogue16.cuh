// Epilogue shared by the block-tile tensor-core kernels (conv1_tc.cu, conv_halo.cu): TMEM -> exact fbgemm
// requantisation (+ fused 2x2 max-pool) -> uint8 NHWC.
//
// The first version read the accumulators with tcgen05.ld.32x32b (thread = one pixel, 16 channels at a time, constants
// through the uniform datapath) and pooled AFTER requantising with warp shuffles on packed bytes.  ncu showed those
// layers issue-bound in the epilogue (conv2: 230 instructions per 32x16 accumulator block, conv1: 78 % issue-active), so
// this version is organised around the instruction count and around latency hiding:
//
// * Accumulators are read with tcgen05.ld.16x256b (mma fragment layout, tools/probe_ld16.cu): a thread holds rows
//   t/4 and t/4 + 8 of a 16-lane half and the column pairs 8i + 2(t&3) + {0,1}.  In the kernels' 8-column x 16-row
//   pixel blocks (accumulator row = 8*image_row + column) rows 8 apart are VERTICALLY ADJACENT pixels, so the
//   vertical half of the 2x2 max-pool is one VIMNMX per value inside a thread, on the raw accumulators, before any
//   requantisation arithmetic; the horizontal half is one SHFL.BFLY(4) per pooled value, arranged so that the two
//   threads of a pair end up with different pooled rows (no duplicated work).  Pooled layers requantise 1/4 of the
//   values.
// * A thread always works on the same NCH (8 or 16) output channels, so k1/bdiv/mult live in 3*NCH registers for the
//   lifetime of the CTA: no constant loads in the loop.  NCH = 8 keeps the kernel under 96 registers, which is what
//   16 epilogue warps + loader + issuers allow; with 8 warps the epilogue ran at ~0.2 instructions per cycle and warp
//   (TMEM-load and dependent-issue latency exposed: two warps per scheduler).
// * The weight rows (B operand) are stored in shared memory in a permuted order so that the channels of a thread are
//   CONSECUTIVE output channels (epi_channel_of_column): one 8/16-byte store per pixel and thread, 32/64 contiguous
//   bytes per pixel and 4-thread group.
// * A warp takes a whole 32-row x 4*NCH-column block (one TMEM lane quarter, one channel part) of a tile; warps are
//   grouped in sets that take alternate tiles (accumulator slots).
// * All tcgen05.ld of a block are issued up front (one exposed TMEM latency per block), the block is re-armed with the
//   pre-bias (common.cuh requant4_prebiased) by tcgen05.st from 8 registers the compiler cannot rematerialise, and the
//   slot is handed back to the MMA issuer before the arithmetic starts.
#pragma once
#include "common.cuh"

namespace b200q {

// TMEM column (= B operand row) -> output channel, within each part of PARTW = 4*NCH columns:
//   column = 16u + 8b + 2q + e   holds   channel = NCH*q + 4u + 2b + e        (u < NCH/4; q in 0..3; b,e in 0..1)
template <int NCH>
__host__ __device__ constexpr int epi_channel_of_column(int col) {
  constexpr int PARTW = 4 * NCH;
  const int c = col % PARTW;
  return (col - c) + NCH * ((c >> 1) & 3) + 4 * (c >> 4) + 2 * ((c >> 3) & 1) + (c & 1);
}

template <int NCH>
struct EpiRegs {
  float k1[NCH], bd[NCH], mu[NCH];  // per-thread constants of output channels ch0 .. ch0+NCH-1
  uint32_t fill[8];                 // MAGIC_BITS x 8 (operands of the re-arming tcgen05.st)
};

// ch0 = 4*NCH*part + NCH*(lane & 3).  magic_smem: a shared-memory word that holds MAGIC_BITS.  The fill registers are
// read from it with volatile loads: ptxas otherwise treats them as constants and rebuilds all eight with MOVs in front
// of every re-arming store (64 FMA-pipe instructions per block; declaring them read-write asm operands does not help,
// ptxas knows tcgen05.st only reads them).
template <int NCH, bool PIN = true, class Consts>
__device__ __forceinline__ void epi_init(const Consts& c, int ch0, const uint32_t* magic_smem, EpiRegs<NCH>& K) {
  // The constants pass through a self-shuffle for the same reason: under register pressure ptxas does not spill them
  // but RE-LOADS them with register-indexed LDC in the middle of the arithmetic, and those go through the
  // address-divergence pipe that tcgen05.ld/st and the mbarrier instructions need (measured: that pipe 89 % busy,
  // kernel 1.8x slower).  A shuffle result cannot be rematerialised.  PIN = false leaves the choice to ptxas (conv1,
  // whose 13 warps leave 128 registers: pinning all 48 constants there costs more than the occasional re-load).
  const int self = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    K.k1[k] = PIN ? __shfl_sync(0xffffffffu, c.k1[ch0 + k], self) : c.k1[ch0 + k];
    K.bd[k] = PIN ? __shfl_sync(0xffffffffu, c.bdiv[ch0 + k], self) : c.bdiv[ch0 + k];
    K.mu[k] = PIN ? __shfl_sync(0xffffffffu, c.mult[ch0 + k], self) : c.mult[ch0 + k];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(K.fill[i]) : "r"(smem_u32(magic_smem)) : "memory");
}

// 16 lanes x 8*REPS columns in the mma fragment layout: register r = 4i + 2s + e of thread t holds lane
// base + t/4 + 8s, column col + 8i + 2(t&3) + e   (i < REPS).
template <int REPS>
__device__ __forceinline__ void tmem_ld_frag(uint32_t taddr, uint32_t* v) {
  static_assert(REPS == 2 || REPS == 4 || REPS == 8, "REPS");
  if constexpr (REPS == 2) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
  } else if constexpr (REPS == 4) {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
  } else {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x256b.x8.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
  }
}
// Re-arm 16 lanes x 16 columns with the pre-bias.
__device__ __forceinline__ void tmem_st_fill_16x16(uint32_t taddr, const uint32_t (&f)[8]) {
  asm volatile("tcgen05.st.sync.aligned.16x256b.x2.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(f[0]),
               "r"(f[1]), "r"(f[2]), "r"(f[3]), "r"(f[4]), "r"(f[5]), "r"(f[6]), "r"(f[7])
               : "memory");
}

// Four consecutive channels K0..K0+3 (compile-time offset into the thread's NCH) of one pixel -> packed word.
template <bool CHECK, int K0, int NCH>
__device__ __forceinline__ uint32_t epi_requant4(uint32_t v0, uint32_t v1, uint32_t v2, uint32_t v3,
                                                 const EpiRegs<NCH>& K, int zp_sub, int lo, uint32_t& bad) {
  return requant4_prebiased<CHECK>(v0, v1, v2, v3, make_float4(K.k1[K0], K.k1[K0 + 1], K.k1[K0 + 2], K.k1[K0 + 3]),
                                   make_float4(K.bd[K0], K.bd[K0 + 1], K.bd[K0 + 2], K.bd[K0 + 3]),
                                   make_float4(K.mu[K0], K.mu[K0 + 1], K.mu[K0 + 2], K.mu[K0 + 3]), zp_sub, lo, bad);
}
// Exact conversion-pipe form of the same (rare: |acc| >= 2^22, or constants not flagged B200Q_RQ_BOUNDED).
template <class Consts>
__device__ __noinline__ uint32_t epi_requant4_exact(uint32_t v0, uint32_t v1, uint32_t v2, uint32_t v3, const Consts& c,
                                                    int ch, int zp_out, int lo) {
  // v = raw + MAGIC_BITS (wrapping), cm = MAGIC_BITS - corr  ->  raw - corr
  const uint32_t v[4] = {v0, v1, v2, v3};
  uint32_t out = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int acc = (int)(v[i] + (uint32_t)c.cm[ch + i] - 2u * MAGIC_BITS);
    out |= requant_u8(acc, c.bdiv[ch + i], c.mult[ch + i], zp_out, lo) << (8 * i);
  }
  return out;
}

template <int G>
__device__ __forceinline__ void epi_store(uint8_t* p, const uint32_t (&w)[G]) {
  if constexpr (G == 4) {
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  } else {
    static_assert(G == 2, "G");
    *reinterpret_cast<uint2*>(p) = make_uint2(w[0], w[1]);
  }
}

// Shared front half of both variants: read the whole block (both 16-lane halves), re-arm it, hand the slot back.
// v[half][r]: r = 8u + 4b + 2s + e  ->  block row 2*half + s, channel 4u + 2b + e of the thread.
template <int NCH, class Release>
__device__ __forceinline__ void epi_drain(uint32_t t_addr, EpiRegs<NCH>& K, uint32_t (&v)[2][2 * NCH], Release release) {
  constexpr int PARTW = 4 * NCH;
  tmem_ld_frag<PARTW / 8>(t_addr, v[0]);
  tmem_ld_frag<PARTW / 8>(t_addr + (16u << 16), v[1]);
  tmem_ld_wait();
#pragma unroll
  for (int c = 0; c < PARTW; c += 16) {
    tmem_st_fill_16x16(t_addr + c, K.fill);
    tmem_st_fill_16x16(t_addr + (16u << 16) + c, K.fill);
  }
  tmem_st_wait();
  tc_fence_before();
  __syncwarp();
  release();
}

// ------------------------------------------------------------------- low-register variants (conv12_fused.cu)
// Same arithmetic as epi_pipeline / epi_block_pool for 16 channels per thread, shaped for a 128-register budget: one
// 16-lane half at a time (read, re-arm, requantise), slot handed back after the second half has been read, and a
// caller-supplied store: `store(half, s, packed)` receives the 16 bytes of the thread's pixel at accumulator row
// 16*half + 8*s + lane/4 of the quarter.
template <bool CHECK, class Consts, class Store, class Release>
__device__ __forceinline__ void epi_block_store16(uint32_t t_addr, EpiRegs<16>& K, const Consts& consts, int ch0, bool fast,
                                                  int zp_out, int lo, Store store, Release release) {
  const int zp_sub = zp_out - (int)MAGIC_BITS;
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const uint32_t a = t_addr + ((uint32_t)(16 * half) << 16);
    uint32_t v[32];
    tmem_ld_frag<8>(a, v);
    tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < 64; c += 16) tmem_st_fill_16x16(a + c, K.fill);
    if (half == 1) {
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      release();
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      uint32_t packed[4];
      uint32_t bad = 0;
      const uint32_t* w = v + 2 * s;
      if (fast) {
        packed[0] = epi_requant4<CHECK, 0>(w[0], w[1], w[4], w[5], K, zp_sub, lo, bad);
        packed[1] = epi_requant4<CHECK, 4>(w[8], w[9], w[12], w[13], K, zp_sub, lo, bad);
        packed[2] = epi_requant4<CHECK, 8>(w[16], w[17], w[20], w[21], K, zp_sub, lo, bad);
        packed[3] = epi_requant4<CHECK, 12>(w[24], w[25], w[28], w[29], K, zp_sub, lo, bad);
      }
      if (!fast || (CHECK && __any_sync(0xffffffffu, requant_magic_out_of_range(bad)))) {
#pragma unroll
        for (int g = 0; g < 4; ++g)
          packed[g] = epi_requant4_exact(w[8 * g], w[8 * g + 1], w[8 * g + 4], w[8 * g + 5], consts, ch0 + 4 * g, zp_out, lo);
      }
      store(half, s, packed);
    }
  }
}

// 2x2 max-pool, one 16-column unit (4 channels of the thread) at a time, software-pipelined: the TMEM loads of unit
// u+1 are in flight while unit u is pooled and requantised (32 accumulator registers live instead of 64).  The block is
// re-armed and handed back once the last unit has been read.
template <bool CHECK, class Consts, class Release>
__device__ __forceinline__ void epi_block_pool16_units(uint32_t t_addr, EpiRegs<16>& K, const Consts& consts, int ch0,
                                                       bool fast, int zp_out, int lo, uint8_t* out, bool valid, int lane,
                                                       Release release) {
  const int zp_sub = zp_out - (int)MAGIC_BITS;
  const bool odd = (lane & 4) != 0;
  constexpr uint32_t HALF1 = 16u << 16;
  uint32_t packed[4];
  uint32_t top[2][8], bot[2][8];
  tmem_ld_frag<2>(t_addr, top[0]);          // block rows 0,1
  tmem_ld_frag<2>(t_addr + HALF1, bot[0]);  // block rows 2,3
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    tmem_ld_wait();  // unit u has landed
    if (u < 3) {
      tmem_ld_frag<2>(t_addr + 16 * (u + 1), top[(u + 1) & 1]);
      tmem_ld_frag<2>(t_addr + HALF1 + 16 * (u + 1), bot[(u + 1) & 1]);
    }
    const uint32_t(&tp)[8] = top[u & 1];
    const uint32_t(&bt)[8] = bot[u & 1];
    uint32_t r[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {  // k = 2b + e  <-  registers 4b + 2s + e
      const int i0 = 4 * (k >> 1) + (k & 1);
      const uint32_t m0 = max(tp[i0], tp[i0 + 2]);
      const uint32_t m1 = max(bt[i0], bt[i0 + 2]);
      const uint32_t send = odd ? m0 : m1;
      const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, 4);
      r[k] = max(odd ? m1 : m0, recv);
    }
    if (u == 3) {  // everything read (no load in flight): re-arm the block and hand the slot back
#pragma unroll
      for (int c = 0; c < 64; c += 16) {
        tmem_st_fill_16x16(t_addr + c, K.fill);
        tmem_st_fill_16x16(t_addr + HALF1 + c, K.fill);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      release();
    }
    uint32_t bad = 0;
    if (fast) {
      if (u == 0) packed[0] = epi_requant4<CHECK, 0>(r[0], r[1], r[2], r[3], K, zp_sub, lo, bad);
      if (u == 1) packed[1] = epi_requant4<CHECK, 4>(r[0], r[1], r[2], r[3], K, zp_sub, lo, bad);
      if (u == 2) packed[2] = epi_requant4<CHECK, 8>(r[0], r[1], r[2], r[3], K, zp_sub, lo, bad);
      if (u == 3) packed[3] = epi_requant4<CHECK, 12>(r[0], r[1], r[2], r[3], K, zp_sub, lo, bad);
    }
    if (!fast || (CHECK && __any_sync(0xffffffffu, requant_magic_out_of_range(bad))))
      packed[u] = epi_requant4_exact(r[0], r[1], r[2], r[3], consts, ch0 + 4 * u, zp_out, lo);
  }
  if (valid) *reinterpret_cast<uint4*>(out) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
}

// ------------------------------------------------------------------------------ no pooling, software-pipelined
// The un-pooled layers (conv3, conv5; conv1) requantise every accumulator and are bound by their epilogue warps, which
// with one block at a time idle through a TMEM round trip per block (both warps of a scheduler wait, read, compute and
// store in lock-step).  Here a warp keeps one 16-lane half in flight while it computes the other: the tcgen05.ld of
// half 1 is issued before the arithmetic of half 0, and the first half of the NEXT tile before the arithmetic of
// half 1.  `next(EpiTile&)` yields the warp's tiles in order (false when there are none left).
// A tile of the warp is one 32-lane quarter x 4*NCH columns of an accumulator slot.  Thread (j = lane/4, q = lane&3)
// produces channels ch0..ch0+NCH-1 of four pixels: accumulator rows 16*half + 8*s + j of the quarter (half, s in 0..1),
// stored at out + half*stride_half + s*stride_s.  In the halo kernels' single-image blocks these are image rows
// 2*half + s of the quarter (stride_s = one image row); in conv_pair.cu s selects the image of the pair and half the
// image row.  valid0/valid1: store the s = 0 / 1 pixels.
struct EpiTile {
  uint32_t t_addr;        // tmem base + (quarter*32 << 16) + first column of the warp's part
  uint64_t* full_bar;     // accumulator complete (MMA commit)
  uint64_t* empty_bar;    // slot drained (one arrive per epilogue warp)
  uint32_t parity;        // phase parity of full_bar for this tile
  uint8_t* out;           // address of the thread's pixel (half 0, s 0), channel ch0; see epi_pipeline
  bool valid0, valid1;
};

template <bool CHECK, bool F32ACC, int NCH, class Consts>
__device__ __forceinline__ void epi_half(const uint32_t (&v)[2 * NCH], const EpiRegs<NCH>& K, const Consts& consts, int ch0,
                                         bool fast, int zp_out, int lo, uint8_t* out, int64_t stride_s, bool valid0,
                                         bool valid1) {
  constexpr int G = NCH / 4;
  const int zp_sub = zp_out - (int)MAGIC_BITS;
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    uint32_t packed[G];
    if constexpr (F32ACC) {  // exact fp32 accumulators, B200Q_RQ_BOUNDED constants: no range test, no fall-back
      const uint32_t* w = v + 2 * s;
#pragma unroll
      for (int g = 0; g < G; ++g)
        packed[g] = requant4_f32acc(w[8 * g], w[8 * g + 1], w[8 * g + 4], w[8 * g + 5],
                                    make_float4(K.bd[4 * g], K.bd[4 * g + 1], K.bd[4 * g + 2], K.bd[4 * g + 3]),
                                    make_float4(K.mu[4 * g], K.mu[4 * g + 1], K.mu[4 * g + 2], K.mu[4 * g + 3]), zp_sub, lo);
    } else {
      uint32_t bad = 0;
      if (fast) {
        const uint32_t* w = v + 2 * s;
        packed[0] = epi_requant4<CHECK, 0>(w[0], w[1], w[4], w[5], K, zp_sub, lo, bad);
        packed[1] = epi_requant4<CHECK, 4>(w[8], w[9], w[12], w[13], K, zp_sub, lo, bad);
        if constexpr (G == 4) {
          packed[2] = epi_requant4<CHECK, 8>(w[16], w[17], w[20], w[21], K, zp_sub, lo, bad);
          packed[3] = epi_requant4<CHECK, 12>(w[24], w[25], w[28], w[29], K, zp_sub, lo, bad);
        }
      }
      if (!fast || (CHECK && __any_sync(0xffffffffu, requant_magic_out_of_range(bad)))) {
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const uint32_t* w = v + 8 * g + 2 * s;
          packed[g] = epi_requant4_exact(w[0], w[1], w[4], w[5], consts, ch0 + 4 * g, zp_out, lo);
        }
      }
    }
    if (s == 0 ? valid0 : valid1) epi_store<G>(out + s * stride_s, packed);
  }
}

// F32ACC: the accumulators are exact fp32 values of acc - corr (conv1_tc.cu) and every MMA of a tile starts from zero:
// nothing to re-arm, so the slot goes back to the issuer as soon as half 1 has landed.
template <bool CHECK, int NCH, bool F32ACC = false, class Consts, class Next>
__device__ __forceinline__ void epi_pipeline(EpiRegs<NCH>& K, const Consts& consts, int ch0, bool fast, int zp_out, int lo,
                                             int64_t stride_s, int64_t stride_half, int lane, Next next) {
  constexpr int PARTW = 4 * NCH;
  constexpr uint32_t HALF1 = 16u << 16;
  EpiTile cur;
  bool have = next(cur);
  if (!have) return;
  uint32_t v0[2 * NCH], v1[2 * NCH];
  mbar_wait(cur.full_bar, cur.parity);
  tc_fence_after();
  tmem_ld_frag<PARTW / 8>(cur.t_addr, v0);
  while (have) {
    // TMEM loads and stores of a warp are served in order: a store issued right behind a load stalls the warp until
    // the load has been served, and tcgen05.wait::st exposes the store latency.  So every re-arming store is issued
    // when no load is in flight, and the slot is handed back after the arithmetic of half 1 (four slots: the issuer
    // needs it three tiles later).
    tmem_ld_wait();                                     // half 0 has landed
    tmem_ld_frag<PARTW / 8>(cur.t_addr + HALF1, v1);    // half 1 in flight during the arithmetic of half 0
    epi_half<CHECK, F32ACC>(v0, K, consts, ch0, fast, zp_out, lo, cur.out, stride_s, cur.valid0, cur.valid1);
    tmem_ld_wait();                                     // half 1 has landed
    if constexpr (F32ACC) {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(cur.empty_bar);        // slot read: back to the MMA issuer
    } else {
#pragma unroll
      for (int c = 0; c < PARTW; c += 16) {
        tmem_st_fill_16x16(cur.t_addr + c, K.fill);
        tmem_st_fill_16x16(cur.t_addr + HALF1 + c, K.fill);
      }
    }
    EpiTile nxt;
    const bool have_next = next(nxt);
    if (have_next) {                                    // first half of the next tile in flight during half 1
      mbar_wait(nxt.full_bar, nxt.parity);
      tc_fence_after();
      tmem_ld_frag<PARTW / 8>(nxt.t_addr, v0);
    }
    epi_half<CHECK, F32ACC>(v1, K, consts, ch0, fast, zp_out, lo, cur.out + stride_half, stride_s, cur.valid0, cur.valid1);
    if constexpr (!F32ACC) {
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(cur.empty_bar);        // slot read and re-armed: back to the MMA issuer
    }
    cur = nxt;
    have = have_next;
  }
}

// ---------------------------------------------------------------------------------------------------- 2x2 max-pool
// Same block; the quarter's 4 image rows x 8 columns become 2 x 4 pooled pixels.  Thread (j, q) ends up with the pooled
// pixel (pooled row j&1, pooled column j>>1) of the block, channels ch0..ch0+NCH-1; out = its address.
// PAIRED (conv_pair.cu): the quarter holds image rows {2q, 2q+1} of TWO images (accumulator row 16*half + 8*image + j),
// so the vertical maximum runs over the halves and thread (j, q) ends up with pooled column j>>1 of image j&1.
// max() on the biased bit patterns is monotone in the raw accumulator (|acc| < 2^27), and the requantisation is
// monotone non-decreasing in the accumulator, so pooling first equals aten::quantized_max_pool2d on the stored tensor.
template <bool CHECK, int NCH, bool PAIRED = false, class Consts, class Release>
__device__ __forceinline__ void epi_block_pool(uint32_t t_addr, EpiRegs<NCH>& K, const Consts& consts, int ch0, bool fast,
                                               int zp_out, int lo, uint8_t* out, bool valid, int lane, Release release) {
  constexpr int G = NCH / 4;
  const int zp_sub = zp_out - (int)MAGIC_BITS;
  const bool odd = (lane & 4) != 0;
  uint32_t v[2][2 * NCH];
  epi_drain<NCH>(t_addr, K, v, release);
  uint32_t r[NCH];
#pragma unroll
  for (int k = 0; k < NCH; ++k) {  // k = 4u + 2b + e  <-  registers 8u + 4b + 2s + e
    const int i0 = 8 * (k >> 2) + 4 * ((k >> 1) & 1) + (k & 1);
    // pooled row 0 / 1 of the block (PAIRED: pooled row of image 0 / 1), column j
    const uint32_t m0 = PAIRED ? max(v[0][i0], v[1][i0]) : max(v[0][i0], v[0][i0 + 2]);
    const uint32_t m1 = PAIRED ? max(v[0][i0 + 2], v[1][i0 + 2]) : max(v[1][i0], v[1][i0 + 2]);
    const uint32_t send = odd ? m0 : m1;
    const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, 4);
    r[k] = max(odd ? m1 : m0, recv);
  }
  uint32_t packed[G];
  uint32_t bad = 0;
  if (fast) {
    packed[0] = epi_requant4<CHECK, 0>(r[0], r[1], r[2], r[3], K, zp_sub, lo, bad);
    packed[1] = epi_requant4<CHECK, 4>(r[4], r[5], r[6], r[7], K, zp_sub, lo, bad);
    if constexpr (G == 4) {
      packed[2] = epi_requant4<CHECK, 8>(r[8], r[9], r[10], r[11], K, zp_sub, lo, bad);
      packed[3] = epi_requant4<CHECK, 12>(r[12], r[13], r[14], r[15], K, zp_sub, lo, bad);
    }
  }
  if (!fast || (CHECK && __any_sync(0xffffffffu, requant_magic_out_of_range(bad)))) {
#pragma unroll
    for (int g = 0; g < G; ++g)
      packed[g] = epi_requant4_exact(r[4 * g], r[4 * g + 1], r[4 * g + 2], r[4 * g + 3], consts, ch0 + 4 * g, zp_out, lo);
  }
  if (valid) epi_store<G>(out, packed);
}

}  // namespace b200q
