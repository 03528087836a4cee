// Shared device/host helpers for the b200q kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/b200q.h"

#if defined(__CUDA_ARCH__) && !defined(__CUDA_ARCH_FEAT_SM100_ALL)
#error "b200q kernels must be compiled with -gencode arch=compute_100a,code=sm_100a"
#endif

namespace b200q {

// ---------------------------------------------------------------- host-side error plumbing
void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
int launched(const char* what);  // after every <<<>>>: bumps b200q_launch_count(), returns the launch status
// Programmatic dependent launch (net.cu b200q_graph_create): while set on the calling thread, launch_kernel() marks
// every kernel "programmatic stream serialization allowed", i.e. it may START while its predecessor in the stream still
// runs; the kernel orders its dependent memory accesses itself with pdl_wait() (below).
void note_graph_replay(int kernels);  // a CUDA-graph replay launched `kernels` kernels (b200q_launch_count)
bool pdl_enabled();
void pdl_set(bool on);
#define B200Q_CUDA(expr) do { int _rc = ::b200q::check_cuda((expr), #expr); if (_rc) return _rc; } while (0)
#define B200Q_REQUIRE(cond, ...) do { if (!(cond)) { ::b200q::set_error(__VA_ARGS__); return B200Q_ERR_INVALID_ARG; } } while (0)
int num_sms();
// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: `mask` (one static per kernel instantiation)
// remembers on which devices of this process it has been raised for `kernel`.
int ensure_dynamic_smem(const void* kernel, int bytes, uint64_t* mask);
// uint8 input path (SURVEY 8f rank 4): raw uint8 NHWC pixels [b,32,32,3] go through a per-channel 256-entry table
// lut[c][v] = quantize_per_tensor(Normalize(ToTensor(v))) that the host builds with the reference's own torch CPU ops,
// so the result is bit-identical to quantising the fp32 tensor the reference's DataLoader would have produced.  The
// first-layer kernels (conv1_tc.cu, simt.cu) take it by value as a kernel parameter.
struct C1Lut {
  uint8_t q[3][256];
};

// conv_halo.cu: halo-resident kernel for the cin=64 layers; returns 1 when the geometry is not covered
// conv1_tc.cu: tensor-core first layer, fp32 NCHW x with the fused quantiser or (lut_host != nullptr, a HOST
// uint8[3][256] table) uint8 NHWC xu8; returns 1 when the layer cannot take that path
int conv1_tc_dispatch(const float* x, const uint8_t* xu8, const uint8_t* lut_host, uint8_t* y, int64_t b,
                      float inv_scale, const b200q_conv3x3* L, cudaStream_t s, int* rc);
int conv3x3_halo_dispatch(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, bool pool, cudaStream_t s,
                          int* rc);
// conv_halo2.cu: conv2 + fused pool on CTA pairs (tcgen05.mma.cta_group::2); returns 1 when not covered
int conv3x3_halo2_dispatch(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, bool pool, cudaStream_t s,
                           int* rc);
// Accuracy counting in the classifier head (b200q_static_evaluate, rule in b200q.h): labels int64 [b]; counters uint64
// [B200Q_EVAL_COUNTERS], accumulated into; pred int32 [b] or nullptr.  The head kernels also skip the logits store when
// their logits pointer is nullptr.
struct EvalArgs {
  const int64_t* labels;
  unsigned long long* counters;
  int32_t* pred;
};
// simt.cu: fc1 + ReLU + fc2 + dequantize in one launch for small batches (ticket must be zero on entry; the kernel leaves
// it zero); returns 1 when the shapes / batch are not covered.  eval != nullptr: counts as well (EvalArgs).
int fc_head_small_dispatch(const uint8_t* x, uint8_t* h, float* logits, unsigned int* ticket, int64_t b,
                           const b200q_linear* fc1, const b200q_linear* fc2, float out_scale, const EvalArgs* eval,
                           cudaStream_t s, int* rc);
// simt.cu: fc2 + dequantize + accuracy counting (the head of b200q_linear_dequant); logits may be nullptr.  Refuses
// (B200Q_ERR_INVALID_ARG) an fc2 that is not k = 512, n = 10 or buffers that are not 16-byte aligned.
int linear_head_eval(const uint8_t* x, float* logits, int64_t b, const b200q_linear* L, float out_scale,
                     const EvalArgs& eval, cudaStream_t s);
// simt.cu: the sandwich net's fp32 head (b200q_sandwich_forward; arithmetic stated in b200q.h).  fc1's uint8 output x
// [b][512] (zero-point zp, DeQuantStub scale fc1_scale) -> logits [b][10]; fc2_w fp32 [10][512] 16-byte aligned, x too.
int sandwich_head(const uint8_t* x, float* logits, int64_t b, const float* fc2_w, const float* fc2_b, int zp,
                  float fc1_scale, cudaStream_t s);
// ... and the same head fused with fc1 for b <= 32 (fc_head_small_kernel; ticket as for fc_head_small_dispatch);
// returns 1 when the shapes / batch are not covered.
int sandwich_head_small_dispatch(const uint8_t* x, uint8_t* h, float* logits, unsigned int* ticket, int64_t b,
                                 const b200q_linear* fc1, const float* fc2_w, const float* fc2_b, float fc1_scale,
                                 cudaStream_t s, int* rc);
// conv_small.cu: CUDA-core kernel for a handful of images (one round trip per layer); returns 1 when not covered
int conv3x3_tiny_dispatch(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, bool pool, cudaStream_t s,
                          int* rc);
// conv_pair.cu: pair-interleaved halo kernel for the 8x8 layers (conv5, conv6); returns 1 when not covered
int conv3x3_pair_dispatch(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, bool pool, cudaStream_t s,
                          int* rc);

// One launch site for the forward's kernels: <<<>>> semantics plus the PDL attribute when pdl_enabled().
template <class... KArgs, class... Args>
int launch_kernel(const char* what, void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t s,
                  Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  if (pdl_enabled()) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return check_cuda(e, what);
  }
  return launched(what);
}

// ---------------------------------------------------------------- programmatic dependent launch (device side)
// pdl_launch_dependents(): this CTA no longer holds back the launch of the next kernel in the stream (which then runs
// its prologue - barrier init, TMEM allocation, weights into shared memory - on whatever SMs are free).
// pdl_wait(): returns once the preceding kernel has completed and its memory is visible; executed by the thread(s) that
// issue the first access to memory the predecessor writes (or reads, for buffers this kernel overwrites: every store of a
// layer kernel is data-dependent on its loader's reads).  Both are no-ops in a launch without the PDL attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// uint8x4 . int8x4 + c
__device__ __forceinline__ int dp4a_us(uint32_t a_u8x4, uint32_t b_s8x4, int c) {
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_u8x4), "r"(b_s8x4), "r"(c));
  return d;
}

// ---------------------------------------------------------------- exact fbgemm requantisation
// t = f32(acc) + bdiv; t = t * mult; q = clamp(rne(t) + zp, lo, 255).  Intrinsics forbid FMA contraction
// (SURVEY.md Appendix A: fp32, RNE, no FMA).
__device__ __forceinline__ uint32_t requant_u8(int acc, float bdiv, float mult, int zp, int lo) {
  float t = __fadd_rn(__int2float_rn(acc), bdiv);
  t = __fmul_rn(t, mult);
  // clamp in the float domain first (bounds are integers, rne is monotone) so the int add cannot overflow
  t = fminf(fmaxf(t, -1024.0f), 1024.0f);
  int q = __float2int_rn(t) + zp;
  return (uint32_t)max(lo, min(q, 255));
}

// ---- fast requantisation (no I2F/F2I: on sm_100 the conversion pipe issues 16 lanes/clk/SM, 8x slower than FADD) --------
// Bit-identical to requant_u8 whenever |acc| < 2^22 and |t| < 2^22, using round-to-nearest-even of the fp32 adder itself:
//   f32(acc)  = as_float(acc + 0x4B400000) - 12582912.0f            (exact: 1.5*2^23 + acc is representable)
//   rne(t)    = as_int(t + 12582912.0f) - 0x4B400000                (ulp of [2^23, 2^24) is 1)
// Callers fold "-corr" into the first integer add and "+zp" into the last one, test the range with one LOP3 per
// element (requant_magic_range_bits) and fall back to requant_u8 for the whole chunk when any lane is out of range.
constexpr uint32_t MAGIC_BITS = 0x4B400000u;  // as_uint(12582912.0f) = 1.5 * 2^23
constexpr float MAGIC_F = 12582912.0f;

__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint64_t u2_pack(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ void u2_unpack(uint64_t v, uint32_t& lo, uint32_t& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
}
// Packed fp32 pairs (sm_100 FADD2 / FMUL2): IEEE round-to-nearest-even per lane, no contraction possible.
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
// d = bytes {sat_u8(b), sat_u8(a), c[7:0], c[15:8]} (low to high): one I2IP.U8.S32.SAT
__device__ __forceinline__ uint32_t pack_sat_u8(int a, int b, uint32_t c) {
  uint32_t d;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// Four output channels of one pixel.  acc: raw s32 accumulators; cm = MAGIC_BITS - corr (per channel, per border class);
// zp_sub = zp_out - MAGIC_BITS; lo = lower clamp (zp_out with ReLU, else 0).  `bad` accumulates range-check bits (see above) when
// CHECK; callers that know |acc - corr| < 2^22 statically (B200Q_RQ_ACC22) skip the test.
// The last add is scalar on purpose: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (even with -fmad=false),
// which would round t*mult + magic once instead of twice.
template <bool CHECK>
__device__ __forceinline__ uint32_t requant4_magic(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, const int4 cm,
                                                   const float4 bd, const float4 mu, int zp_sub, int lo,
                                                   uint32_t& bad) {
  const uint32_t m0 = a0 + (uint32_t)cm.x, m1 = a1 + (uint32_t)cm.y;
  const uint32_t m2 = a2 + (uint32_t)cm.z, m3 = a3 + (uint32_t)cm.w;
  if constexpr (CHECK) {
    bad |= (m0 ^ 0x4B000000u);
    bad |= (m1 ^ 0x4B000000u);
    bad |= (m2 ^ 0x4B000000u);
    bad |= (m3 ^ 0x4B000000u);
  }
  const uint64_t neg_magic = f2_pack(-MAGIC_F, -MAGIC_F);
  uint64_t t01 = f2_add(u2_pack(m0, m1), neg_magic);
  uint64_t t23 = f2_add(u2_pack(m2, m3), neg_magic);
  t01 = f2_mul(f2_add(t01, f2_pack(bd.x, bd.y)), f2_pack(mu.x, mu.y));
  t23 = f2_mul(f2_add(t23, f2_pack(bd.z, bd.w)), f2_pack(mu.z, mu.w));
  uint32_t r0, r1, r2, r3;
  u2_unpack(t01, r0, r1);
  u2_unpack(t23, r2, r3);
  // max(x + zp_sub, lo) is one VIADDMNMX; the upper clamp (and the pack) is the saturating I2IP.  (__vmaxu4 on the
  // packed word is emulated with ~7 instructions on sm_100.)
  const int q0 = max(__float_as_int(__fadd_rn(__uint_as_float(r0), MAGIC_F)) + zp_sub, lo);
  const int q1 = max(__float_as_int(__fadd_rn(__uint_as_float(r1), MAGIC_F)) + zp_sub, lo);
  const int q2 = max(__float_as_int(__fadd_rn(__uint_as_float(r2), MAGIC_F)) + zp_sub, lo);
  const int q3 = max(__float_as_int(__fadd_rn(__uint_as_float(r3), MAGIC_F)) + zp_sub, lo);
  const uint32_t hi = pack_sat_u8(q3, q2, 0u);
  return pack_sat_u8(q1, q0, hi);
}
// true when any accumulated range-check bit says |acc - corr| >= 2^22
__device__ __forceinline__ bool requant_magic_out_of_range(uint32_t bad) { return (bad >> 23) != 0u; }

// Variant for accumulators that were PRE-BIASED in TMEM with MAGIC_BITS (the epilogue re-arms each accumulator chunk with
// tcgen05.st after reading it, and every MMA accumulates): v = raw + MAGIC_BITS reinterpreted as float IS f32(raw)+MAGIC_F
// for |raw| < 2^22, so no integer instruction is needed at all.  k1 = -(MAGIC_F + corr) (exact for |corr| < 2^22) turns
// it into f32(raw - corr) with one exact subtraction.  The rounding add is fma(t, 1.0, MAGIC_F): still one rounding of
// t + MAGIC_F, but a packed instruction that ptxas cannot contract with the multiply before it.
template <bool CHECK>
__device__ __forceinline__ uint32_t requant4_prebiased(uint32_t v0, uint32_t v1, uint32_t v2, uint32_t v3, const float4 k1,
                                                       const float4 bd, const float4 mu, int zp_sub, int lo,
                                                       uint32_t& bad) {
  if constexpr (CHECK) {
    bad |= (v0 ^ 0x4B000000u);
    bad |= (v1 ^ 0x4B000000u);
    bad |= (v2 ^ 0x4B000000u);
    bad |= (v3 ^ 0x4B000000u);
  }
  const uint64_t ones = f2_pack(1.0f, 1.0f), magic = f2_pack(MAGIC_F, MAGIC_F);
  uint64_t t01 = f2_add(u2_pack(v0, v1), f2_pack(k1.x, k1.y));
  uint64_t t23 = f2_add(u2_pack(v2, v3), f2_pack(k1.z, k1.w));
  t01 = f2_mul(f2_add(t01, f2_pack(bd.x, bd.y)), f2_pack(mu.x, mu.y));
  t23 = f2_mul(f2_add(t23, f2_pack(bd.z, bd.w)), f2_pack(mu.z, mu.w));
  t01 = f2_fma(t01, ones, magic);
  t23 = f2_fma(t23, ones, magic);
  uint32_t r0, r1, r2, r3;
  u2_unpack(t01, r0, r1);
  u2_unpack(t23, r2, r3);
  const int q0 = max((int)r0 + zp_sub, lo), q1 = max((int)r1 + zp_sub, lo);
  const int q2 = max((int)r2 + zp_sub, lo), q3 = max((int)r3 + zp_sub, lo);
  return pack_sat_u8(q1, q0, pack_sat_u8(q3, q2, 0u));
}

// 32 consecutive output channels of one pixel (one tcgen05.ld 32x32b.x32 worth): v -> 8 packed words.
// cm: this pixel's border-class row of (MAGIC_BITS - corr), bd/mu: bdiv / mult, all at the chunk's first channel
// (shared memory, or register arrays after inlining).  `fast` = layer flagged B200Q_RQ_BOUNDED.
template <bool CHECK>
__device__ __forceinline__ void requant_chunk32(const uint32_t (&v)[32], const int4* cm, const float4* bd, const float4* mu,
                                                bool fast, int zp_out, int lo, uint32_t (&packed)[8]) {
  const int zp_sub = zp_out - (int)MAGIC_BITS;
  uint32_t bad = 0;
  if (fast) {
#pragma unroll
    for (int g = 0; g < 8; ++g)
      packed[g] = requant4_magic<CHECK>(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3], cm[g], bd[g], mu[g], zp_sub,
                                        lo, bad);
  }
  if (!fast || (CHECK && __any_sync(0xffffffffu, requant_magic_out_of_range(bad)))) {
    // exact conversion-pipe form (rare: |acc| >= 2^22, or constants not flagged as bounded)
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const int4 c = cm[g];
      const float4 b = bd[g], m = mu[g];
      packed[g] = requant_u8((int)(v[4 * g + 0] + (uint32_t)c.x - MAGIC_BITS), b.x, m.x, zp_out, lo) |
                  (requant_u8((int)(v[4 * g + 1] + (uint32_t)c.y - MAGIC_BITS), b.y, m.y, zp_out, lo) << 8) |
                  (requant_u8((int)(v[4 * g + 2] + (uint32_t)c.z - MAGIC_BITS), b.z, m.z, zp_out, lo) << 16) |
                  (requant_u8((int)(v[4 * g + 3] + (uint32_t)c.w - MAGIC_BITS), b.w, m.w, zp_out, lo) << 24);
    }
  }
}

// Per-byte max of four packed uint8x4 words.  sm_100 has no native byte SIMD max (__vmaxu4 is emulated with ~7
// instructions per pair); 16-bit lanes are native, so split even/odd bytes (PRMT), reduce with max.u16x2, re-interleave.
__device__ __forceinline__ uint32_t max_u16x2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("max.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t max4_u8x4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  const uint32_t e = max_u16x2(max_u16x2(__byte_perm(a, 0, 0x4240), __byte_perm(b, 0, 0x4240)),
                               max_u16x2(__byte_perm(c, 0, 0x4240), __byte_perm(d, 0, 0x4240)));
  const uint32_t o = max_u16x2(max_u16x2(__byte_perm(a, 0, 0x4341), __byte_perm(b, 0, 0x4341)),
                               max_u16x2(__byte_perm(c, 0, 0x4341), __byte_perm(d, 0, 0x4341)));
  return __byte_perm(e, o, 0x6240);
}

__device__ __forceinline__ uint32_t quantize_u8(float x, float inv_scale, int zp) {
  float t = __fmul_rn(x, inv_scale);
  t = fminf(fmaxf(t, -1024.0f), 1024.0f);
  int q = __float2int_rn(t) + zp;
  return (uint32_t)max(0, min(q, 255));
}

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// try_wait suspends the thread in hardware until the phase completes or the hint expires, whichever is first; a long
// hint keeps idle producer / MMA threads from burning issue slots the epilogue warps of the same sub-partition need.
// In practice a suspended try_wait also returns whenever ANY mbarrier of the CTA sees an arrival (measured: ~19 wake-ups
// per wait in conv3 with 16 epilogue warps), so the retry loop is kept to a handful of instructions.  Replacing the
// suspension by test_wait + timed __nanosleep polling (no spurious wake-ups) was measured 3-15 % SLOWER on every
// kernel: the wake-up latency matters more than the wasted issue slots.
constexpr uint32_t MBAR_SUSPEND_HINT_NS = 200000u;
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(MBAR_SUSPEND_HINT_NS)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug must abort the kernel (trap -> launch failure), never hang the GPU box.  (A leaner retry
// loop - spin counter instead of the timer read - was measured 1-5 % slower: the extra instructions act as back-off.)
#ifndef B200Q_WAIT_TIMEOUT_NS
#define B200Q_WAIT_TIMEOUT_NS 4000000000ull
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0 && globaltimer_ns() - t0 > B200Q_WAIT_TIMEOUT_NS) {
      printf("b200q: mbarrier wait timeout block %d thread %d bar@%u parity %u\n", blockIdx.x, threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// TMA (cp.async.bulk.tensor) tile loads, completion signalled on an mbarrier via complete_tx.
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// MMA completion -> mbarrier arrive (implicitly fences before_thread_sync)
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], 8-bit integer operands, s32 accumulate.  One thread issues.
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Fill 32 lanes x 8 consecutive 32-bit columns with one value (thread t writes lane base_lane + t).
__device__ __forceinline__ void tmem_st_fill8(uint32_t taddr, uint32_t value) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(value)
               : "memory");
}
// 16 lanes x 64 consecutive 32-bit columns in the mma-accumulator fragment layout (tools/probe_ld16.cu): register r
// of thread t holds lane base_lane + t/4 + 8*((r>>1)&1), column col + 8*(r>>2) + 2*(t&3) + (r&1).  A thread therefore
// holds PAIRS of rows 8 apart - in the halo kernels' 8-column block tiles those are vertically adjacent pixels.
__device__ __forceinline__ void tmem_ld_16x256b_x8(uint32_t taddr, uint32_t (&v)[32]) {
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
// 32 lanes x 32 consecutive 32-bit columns: thread t of the warp gets lane (base_lane + t), columns col..col+31.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

// ---------------------------------------------------------------- UMMA descriptors (cf. cute/arch/mma_sm100_desc.hpp)
// Shared-memory matrix descriptor, K-major operand, swizzled (SWIZZLE_64B or SWIZZLE_128B):
//   bits [0,14)  start address >> 4          bits [16,30) leading byte offset >> 4 (1 for swizzled K-major)
//   bits [32,46) stride byte offset >> 4     bits [46,48) version = 1 (Blackwell)
//   bits [49,52) base offset = 0             bits [61,64) layout type (2 = SW128, 4 = SW64, 6 = SW32)
// SBO = byte distance between consecutive 8-row groups.
template <int SWIZZLE_BYTES>
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr, uint32_t sbo_bytes) {
  constexpr uint64_t layout = SWIZZLE_BYTES == 128 ? 2 : SWIZZLE_BYTES == 64 ? 4 : 6;
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;
  d |= layout << 61;
  return d;
}
// Instruction descriptor for kind::i8: D=s32, A=u8 (activations), B=s8 (weights), both K-major, dense, no saturate.
__host__ __device__ constexpr uint32_t make_idesc_i8(int m, int n) {
  return (2u << 4)                      // c_format = S32
         | (0u << 7)                    // a_format = UINT8
         | (1u << 10)                   // b_format = INT8
         | (0u << 15) | (0u << 16)      // A, B K-major
         | ((uint32_t)(n >> 3) << 17)   // N
         | ((uint32_t)(m >> 4) << 24);  // M
}

// ---------------------------------------------------------------- host: TMA descriptor encoding (driver entry point
// resolved at run time so the library links without libcuda)
int encode_tensor_map(CUtensorMap* out, const void* gptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box, int swizzle_bytes);

}  // namespace b200q
