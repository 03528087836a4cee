/*
 * b200q.h — C ABI of the B200 (sm_100a) quantized-ConvNet hot path.
 *
 * Drop-in boundary for the arithmetic the reference (his0si/ConvNet-Quantization)
 * reaches through PyTorch's QuantizedCPU / FBGEMM ops.  The reference has no FFI
 * of its own (it is pure Python, SURVEY.md F1); every entry point below cites the
 * reference call site whose ATen op it replaces.  All pointers are DEVICE pointers
 * unless the name ends in _host; the caller owns every buffer; kernels never
 * allocate; `stream` is a cudaStream_t passed as void*.  Return value: 0 on
 * success, negative b200q_status otherwise (no exceptions cross this boundary).
 *
 * Layouts: activations uint8 NHWC; conv weights int8 [Cout][kh][kw][Cin]
 * ("K-major", K = 9*Cin); linear weights int8 [N][K].  All zero-points refer to
 * quint8 activations; weights are symmetric (zero-point 0), per-output-channel.
 */
#ifndef B200Q_H_
#define B200Q_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum b200q_status {
  B200Q_OK = 0,
  B200Q_ERR_INVALID_ARG = -1,   /* bad shape / null pointer / unsupported layer geometry */
  B200Q_ERR_CUDA = -2,          /* a CUDA runtime call failed; see b200q_last_error() */
  B200Q_ERR_NO_DEVICE = -3,     /* no sm_100 device is current */
  B200Q_ERR_DRIVER = -4         /* cuTensorMapEncodeTiled unavailable / failed */
} b200q_status;

/* Human-readable text of the last error raised on the calling thread. */
const char* b200q_last_error(void);
/* ABI version of this header (bumped on any signature change). */
int b200q_abi_version(void);
/* Number of CUDA kernels this library has launched in this process (all threads); bench.py reports the delta
 * over its timed region as "gpu_launches". */
uint64_t b200q_launch_count(void);

/* ---- per-output-channel requantisation constants (fbgemm semantics, SURVEY App. A) ----
 *   t = f32(acc) + bdiv[c];  t = t * mult[c];  q = clamp(rne(t) + zp_out, relu ? zp_out : 0, 255)
 * with mult[c] = (s_x*s_w[c])/s_out and bdiv[c] = bias[c]/(s_x*s_w[c]) precomputed in fp32 on the host. */
typedef struct b200q_requant {
  const float* mult;      /* [N]  */
  const float* bdiv;      /* [N]  */
  int32_t zp_out;
  int32_t relu;           /* 1: clamp low at zp_out (aten::relu on quint8 == max(q, zp)) */
  int32_t flags;          /* B200Q_RQ_* */
  int32_t reserved;
  /* Optional HOST copies of mult / bdiv (same contents).  When present (together with corr_host of the layer) the
   * kernels that take their per-channel constants as kernel parameters are eligible; NULL selects the kernels that
   * stage the device tables through shared memory. */
  const float* mult_host;
  const float* bdiv_host;
} b200q_requant;
/* Caller guarantees 0 <= mult[c] <= 0.5, |bdiv[c]| <= 2^21 and |corr| < 2^22 for every channel.  The tensor-core kernels then use a
 * conversion-free formulation of the same arithmetic (bit-identical; accumulators outside +-2^22 are detected at run
 * time and take the I2F/F2I form).  Without the flag the I2F/F2I form is always used. */
#define B200Q_RQ_BOUNDED 1
/* Caller guarantees |sum x*w| < 2^22 and |sum (x-zp_x)*w| < 2^22 for every possible uint8 input (a bound on the
 * layer's weights, see packing.acc_bound): lets the tensor-core kernels skip the per-element run-time range test. */
#define B200Q_RQ_ACC22 2

/* 3x3 / stride 1 / pad 1 quantized convolution layer, packed.
 * Replaces quantized::conv2d(+aten::relu) reached from the converted conv modules
 * (fusion list models/dynamic_ptq_model.py:289-299; layer shapes models/baseline_model.py:13-34). */
typedef struct b200q_conv3x3 {
  int32_t cin, cout;          /* cin in {3(padded to 4), 64, 128, 256}; cout in {64,128,256} */
  int32_t img;                /* H == W in {32, 16, 8} */
  int32_t zp_x;               /* input activation zero-point */
  const int8_t*  w;           /* [cout][3][3][cin_padded] */
  const int32_t* corr;        /* [9][cout]: zp_x * sum of w over the taps valid for border class (3*rowclass+colclass) */
  const int32_t* corr_host;   /* optional HOST copy of corr (see b200q_requant.mult_host) */
  b200q_requant rq;
} b200q_conv3x3;

/* Quantized linear layer, packed.  Replaces quantized::linear(+relu) (fc1/fc2, models/baseline_model.py:37-40). */
typedef struct b200q_linear {
  int32_t k, n;
  int32_t zp_x;
  const int8_t*  w;           /* [n][k] */
  const int32_t* corr;        /* [n]: zp_x * sum_k w[n][k] */
  const int32_t* corr_host;   /* optional HOST copy of corr */
  b200q_requant rq;
} b200q_linear;

/* ---- memory-bound element-wise ops -------------------------------------------------------- */

/* aten::quantize_per_tensor: fp32 NCHW [b,c,h,w] -> uint8 NHWC [b,h,w,c_pad] (channels >= c filled with zp).
 * q = clamp(rne(x * inv_scale) + zp, 0, 255), inv_scale = 1.0f/scale computed by the caller in fp32. */
int b200q_quantize_nchw_to_nhwc(const float* x, uint8_t* y, int64_t b, int c, int h, int w, int c_pad,
                                float inv_scale, int zp, void* stream);
/* Flat variant (layout preserved), n elements. */
int b200q_quantize_flat(const float* x, uint8_t* y, int64_t n, float inv_scale, int zp, void* stream);
/* aten::dequantize: y = f32(q - zp) * scale, n elements. */
int b200q_dequantize(const uint8_t* q, float* y, int64_t n, float scale, int zp, void* stream);
/* aten::relu on quint8: y = max(q, zp). */
int b200q_relu_q(const uint8_t* q, uint8_t* y, int64_t n, int zp, void* stream);
/* aten::quantized_max_pool2d k=2 s=2 on uint8 NHWC [b,h,w,c] -> [b,h/2,w/2,c]; c % 16 == 0. */
int b200q_max_pool2x2_nhwc(const uint8_t* x, uint8_t* y, int64_t b, int h, int w, int c, void* stream);
/* Bytes of device scratch (zero-initialised ONCE by the caller, self-resetting afterwards) that b200q_minmax,
 * b200q_aminmax and b200q_linear_dynamic need: block partials, the last-block counter and the 8-float qparams block. */
#define B200Q_REDUCE_SCRATCH_BYTES 8256
/* Dynamic range for quantized::linear_dynamic: out5 = {min(x,0), max(x,0), scale, 1/scale, zero_point} with the
 * (scale, zero_point) of ChooseQuantizationParams(min, max, 0, 255, reduce_range=true)
 * (ATen/native/quantized/cpu/QuantUtils.h), computed on device.  scratch: B200Q_REDUCE_SCRATCH_BYTES. */
int b200q_minmax(const float* x, int64_t n, float* out5, void* scratch, void* stream);
/* torch.aminmax as the calibration observers call it (torch/ao/quantization/observer.py: MinMaxObserver /
 * HistogramObserver.forward, reached from prepare() at models/custom_quantization_model.py:5): out2 = {min(x), max(x)}
 * (no zero extension).  scratch: B200Q_REDUCE_SCRATCH_BYTES. */
int b200q_aminmax(const float* x, int64_t n, float* out2, void* scratch, void* stream);
/* torch.histc(x, bins, min=lo, max=hi) for the HistogramObserver (SURVEY 8f rank 2: GPU-side calibration):
 * hist[i] += |{x : bin(x) == i}| with ATen's CPU rule bin(x) = int(((x - lo) * bins) / (hi - lo)) evaluated in fp32
 * (bin == bins -> bins - 1; values outside [lo, hi] are ignored; lo < hi required - the caller widens a degenerate
 * range to [lo-1, hi+1] like ATen does).  hist: int64[bins] on the device, ACCUMULATED into (zero it first).
 * bins <= 4096. */
int b200q_histc(const float* x, int64_t n, float lo, float hi, int bins, int64_t* hist, void* stream);
/* y[i] = lut[x[i]]: byte-wise table look-up (lut_host: HOST uint8[256]).  Used by the per-layer "sandwich" variant
 * (models/custom_quantization_model.py:34-58): DeQuantStub -> fp32 ReLU -> QuantStub of the next layer is a monotone
 * uint8 -> uint8 map, evaluated once per value of the table with the reference's own ops. */
int b200q_lut_u8(const uint8_t* x, uint8_t* y, int64_t n, const uint8_t* lut_host, void* stream);

/* ---- convolutions ---------------------------------------------------------------------------- */

/* Direct (CUDA-core, dp4a) 3x3 conv for the first layer (cin=3 padded to 4): uint8 NHWC4 -> uint8 NHWC. */
int b200q_conv3x3_first(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, void* stream);
/* Fused aten::quantize_per_tensor + first conv: fp32 NCHW [b,3,img,img] -> uint8 NHWC [b,img,img,cout]. */
int b200q_quantize_conv3x3_first(const float* x, uint8_t* y, int64_t b, float inv_scale,
                                 const b200q_conv3x3* L, void* stream);
/* uint8 data path (the step before the model in the reference: utils/dataset_manager.py:41-44 ToTensor + Normalize,
 * then QuantStub): raw uint8 NHWC pixels [b,32,32,3] -> conv1 output uint8 NHWC [b,32,32,64].  lut_host is a HOST
 * table uint8[3][256], lut[c][v] = quantize_per_tensor(Normalize(ToTensor(v)))[c], built by the caller with the
 * reference's own torch ops (convnet_quantization_b200.packing.input_lut), so results are bit-identical to the fp32
 * route.  L must be conv1 (cin 4, cout 64, img 32); x_nhwc 8-byte aligned, y 16-byte aligned.  Kernel selection is
 * that of b200q_quantize_conv3x3_first (CUDA cores for a few images or for layers without host mirrors /
 * B200Q_RQ_BOUNDED, tensor cores otherwise); results do not depend on it. */
int b200q_u8_conv3x3_first(const uint8_t* x_nhwc, uint8_t* y, int64_t b, const uint8_t* lut_host,
                           const b200q_conv3x3* L, void* stream);
#ifdef B200Q_DEV  /* development library (libb200q_dev.so) only: measured slower than the two kernels it replaces */
/* The first two layers and the first max-pool in one kernel (conv1's output never leaves shared memory):
 * aten::quantize_per_tensor + quantized::conv2d + relu (L1: cin 4, cout 64, img 32) + quantized::conv2d + relu
 * (L2: cin 64, cout 64) + aten::quantized_max_pool2d: fp32 NCHW [b,3,32,32] -> uint8 NHWC [b,16,16,64].
 * Reference call sites: models/baseline_model.py:60-66 on the converted net.  Both layers need host mirrors of
 * their constants and L1 must be B200Q_RQ_BOUNDED; otherwise B200Q_ERR_INVALID_ARG (use the separate entry points). */
int b200q_conv12_fused(const float* x, uint8_t* y, int64_t b, float inv_scale, const b200q_conv3x3* L1,
                       const b200q_conv3x3* L2, void* stream);
#endif
/* tcgen05 implicit-GEMM 3x3 conv (cin % 64 == 0): uint8 NHWC [b,img,img,cin] -> uint8 NHWC [b,img,img,cout]
 * or, with pool2x2 != 0, the 2x2/2 max-pooled [b,img/2,img/2,cout] (aten::quantized_max_pool2d fused). */
int b200q_conv3x3_tc(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, int pool2x2, void* stream);
#ifdef B200Q_DEV  /* development library only */
/* Reference-grade CUDA-core version of the same op (bring-up cross-check; not used by the net). */
int b200q_conv3x3_simt(const uint8_t* x, uint8_t* y, int64_t b, const b200q_conv3x3* L, void* stream);
#endif

/* ---- linear ----------------------------------------------------------------------------------- */

/* tcgen05 GEMM: uint8 [b,k] x int8 [n,k]^T -> uint8 [b,n]   (k % 128 == 0, n % 64 == 0). */
int b200q_linear_tc(const uint8_t* x, uint8_t* y, int64_t b, const b200q_linear* L, void* stream);
/* CUDA-core version (small n, e.g. fc2): uint8 [b,k] -> uint8 [b,n]. */
int b200q_linear_simt(const uint8_t* x, uint8_t* y, int64_t b, const b200q_linear* L, void* stream);
/* Small linear fused with aten::dequantize (fc2 + DeQuantStub): uint8 [b,k] -> fp32 [b,n]. */
int b200q_linear_dequant(const uint8_t* x, float* y, int64_t b, const b200q_linear* L, float out_scale, void* stream);

/* quantized::linear_dynamic(x, W, reduce_range=True) (models/dynamic_ptq_model.py:302-306 -> nnqd.Linear), two launches:
 * (1) per-tensor min/max of the WHOLE input -> (scale, zp) on device (b200q_minmax); (2) one tcgen05 GEMM kernel whose
 * producer warps quantise the fp32 rows straight into the swizzled K-major shared-memory tiles the tensor core reads
 * (the uint8 activations never exist in HBM), weights by TMA.  Arithmetic is fbgemm's, bit for bit:
 * x_q = clamp(rne(fma(x, 1/s_x, zp)), 0, 255) and y = fma(f32(acc - zp*wsum[n]), fl32(s_x*s_w), bias[n])
 * (+ ReLU when relu != 0, the F.relu that follows fc1 at models/baseline_model.py:80).
 * x fp32 [b,k] (k % 64 == 0); w int8 [n][k], per-tensor symmetric scale w_scale, n == 512 or n <= 16;
 * wsum[n] = sum_k w; bias fp32 [n]; y fp32 [b,n].  scratch: B200Q_REDUCE_SCRATCH_BYTES (its qparams block is left
 * holding {min, max, scale, 1/scale, zp} of this call at byte offset B200Q_REDUCE_QPARAMS_OFFSET). */
#define B200Q_REDUCE_QPARAMS_OFFSET 8224
int b200q_linear_dynamic(const float* x, float* y, int64_t b, int k, int n, const int8_t* w, const int32_t* wsum,
                         float w_scale, const float* bias, int relu, void* scratch, int64_t scratch_bytes,
                         void* stream);

/* ---- whole static-PTQ network ------------------------------------------------------------------ */

typedef struct b200q_static_net {
  float in_inv_scale;           /* 1.0f / QuantStub scale  */
  int32_t in_zp;
  b200q_conv3x3 conv[6];
  b200q_linear fc1, fc2;
  float out_scale;              /* fc2 output scale (DeQuantStub) ; zp is fc2.rq.zp_out */
} b200q_static_net;

/* Bytes of device workspace b200q_static_forward needs for batch b (two ping-pong activation buffers of b x 64 KiB plus
 * 2 KiB).  The contents need no initialisation; one workspace serves one forward at a time (forwards on different
 * streams need their own). */
int64_t b200q_static_workspace_bytes(int64_t b);
/* fp32 NCHW [b,3,32,32] -> fp32 logits [b,10]; restates models/baseline_model.py:58-83 on the converted model.
 * Enqueues eight kernels on `stream` (seven for b <= 32: fc1 + fc2 + dequantize fused), picking per layer the kernel
 * shape that fits the batch (small-batch tiles, one or three images per band, CTA pairs for conv2); results do not
 * depend on that choice.
 * taps (optional, may be NULL): 12 device pointers receiving the uint8 activations after
 * quant, conv1, conv2, pool1, conv3, conv4, pool2, conv5, conv6, pool3, fc1, fc2 (NHWC) for parity tests. */
int b200q_static_forward(const b200q_static_net* net, const float* x, float* logits, int64_t b,
                         void* workspace, int64_t workspace_bytes, uint8_t* const* taps, void* stream);
/* Same forward from raw uint8 NHWC pixels [b,32,32,3] (see b200q_u8_conv3x3_first for lut_host). */
int b200q_static_forward_u8(const b200q_static_net* net, const uint8_t* x_nhwc, const uint8_t* lut_host, float* logits,
                            int64_t b, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- accuracy counting (utils/model_evaluator.py:15-55: top-1 / top-5 hits over a labelled dataset) ----------------
 * The forward above with the counting done by the classifier-head kernel itself: no extra launch, and the logits need
 * not leave the device.  The rule, for one image with uint8 fc2 outputs q[0..n) and label L (uint8 values compared:
 * dequantisation is strictly monotone, so the logits give the same result):
 *   g = #{j : q[j] > q[L]},  e = #{j != L : q[j] == q[L]},  rank = g + #{j < L : q[j] == q[L]}
 *   top-k hit   <=> rank < k            (k = 1 and k = min(5, n); the order of torch.sort(descending, stable), for k = 1
 *                                        torch.argmax: ties go to the lower class index)
 *   top-k tied  <=> g < k <= g + e      (some order of the tied classes would flip this image's hit; so a topk-based
 *                                        count of the same logits differs from this one by at most the tied count)
 * A label outside [0, n) is a miss and not tied; it still counts in IMAGES.
 * counters: uint64 [B200Q_EVAL_COUNTERS] on the device (8-byte aligned), ACCUMULATED into (zero it first); integer
 * adds, so the totals are deterministic. */
#define B200Q_EVAL_COUNTERS 5
#define B200Q_EVAL_TOP1 0
#define B200Q_EVAL_TOP5 1
#define B200Q_EVAL_IMAGES 2
#define B200Q_EVAL_TOP1_TIED 3
#define B200Q_EVAL_TOP5_TIED 4
/* x fp32 NCHW [b,3,32,32]; labels int64 [b] (8-byte aligned); pred (optional, NULL skips it) int32 [b] receives the
 * rank-0 class; logits (optional, NULL skips the store) fp32 [b,10] receives what b200q_static_forward writes.  Same
 * kernels, launch count and workspace as b200q_static_forward (eager only: no graph).  Null labels or counters,
 * b < 0 and misaligned labels / counters / pred are refused before any CUDA call.  fc2 must be k = 512, n = 10. */
int b200q_static_evaluate(const b200q_static_net* net, const float* x, const int64_t* labels, int64_t b,
                          uint64_t* counters, int32_t* pred, float* logits, void* workspace, int64_t workspace_bytes,
                          void* stream);
/* The same from raw uint8 NHWC pixels [b,32,32,3] (lut_host: see b200q_u8_conv3x3_first). */
int b200q_static_evaluate_u8(const b200q_static_net* net, const uint8_t* x_nhwc, const uint8_t* lut_host,
                             const int64_t* labels, int64_t b, uint64_t* counters, int32_t* pred, float* logits,
                             void* workspace, int64_t workspace_bytes, void* stream);

/* ---- whole-network executor (SURVEY 8f rank 1) -----------------------------------------------------------------
 * The forward captured ONCE as a CUDA graph for a fixed batch and fixed buffers, with programmatic dependent launch
 * between the layer kernels (kernel N+1's prologue - weights into shared memory, TMEM allocation, pad initialisation -
 * overlaps kernel N), replayed with one call.  Serves the operating points of the reference's own driver
 * (utils/inference_benchmark.py:126-138: batch 1 and batch 32), where eight separate launches are latency-bound.
 * x_static / logits_static / workspace are caller-owned device buffers that must stay valid (and must not be
 * written by anyone else while a replay is in flight); the caller copies its input into x_static before each launch.
 * All three calls take the stream the graph is captured / replayed on.  The handle is not thread-safe. */
typedef struct b200q_graph b200q_graph;
#define B200Q_GRAPH_PDL 1   /* flags: programmatic dependent launch between the layer kernels */
/* Runs one eager forward on `stream` (first-use initialisation), then captures.  `stream` must not be the legacy
 * default stream (CUDA cannot capture it); replays may go to any stream. */
int b200q_graph_create(const b200q_static_net* net, const float* x_static, float* logits_static, int64_t b,
                       void* workspace, int64_t workspace_bytes, int flags, void* stream, b200q_graph** out);
/* Same executor for the uint8 data path (b200q_static_forward_u8): x_nhwc_static is the caller's uint8 NHWC [b,32,32,3]
 * pixel buffer.  lut_host (HOST uint8[3][256], see b200q_u8_conv3x3_first) is read during this call only: its contents
 * are captured by value into kernel parameters, so the caller may free or change it afterwards (replays keep using the
 * table as it was here).  Replay and destruction: b200q_graph_launch / b200q_graph_destroy. */
int b200q_graph_create_u8(const b200q_static_net* net, const uint8_t* x_nhwc_static, const uint8_t* lut_host,
                          float* logits_static, int64_t b, void* workspace, int64_t workspace_bytes, int flags,
                          void* stream, b200q_graph** out);
int b200q_graph_launch(b200q_graph* g, void* stream);
int b200q_graph_destroy(b200q_graph* g);

/* ---- per-layer "sandwich" network (models/custom_quantization_model.py:34-58, 202-261) ------------------------------
 * conv1..conv6 and fc1 each in QuantStub -> int8 layer -> DeQuantStub, fp32 ReLU / max-pool between them, fc2 in fp32.
 * Between two int8 layers, DeQuantStub -> ReLU -> next QuantStub is the monotone uint8 -> uint8 table lut_host[i]
 * (b200q_lut_u8); it commutes with the max-pool, so after conv2 / conv4 / conv6 it runs on the pooled tensor. */
typedef struct b200q_sandwich_net {
  float in_inv_scale;          /* 1.0f / conv1's QuantStub scale; its zero-point is conv[0].zp_x */
  b200q_conv3x3 conv[6];       /* rq.relu == 0 (the sandwich's output observer sees pre-ReLU values) */
  b200q_linear fc1;            /* rq.relu == 0; k 4096 in NHWC column order, n 512 */
  uint8_t lut_host[6][256];    /* boundary tables conv1->conv2 ... conv5->conv6, conv6->fc1 (ptq.sandwich_boundary_lut) */
  float fc1_scale;             /* fc1's DeQuantStub; zero-point fc1.rq.zp_out */
  const float* fc2_w;          /* fp32 [10][512], device, 16-byte aligned */
  const float* fc2_b;          /* fp32 [10], device, 4-byte aligned */
} b200q_sandwich_net;

/* fp32 NCHW [b,3,32,32] -> fp32 logits [b,10].  Workspace: b200q_static_workspace_bytes(b) (the same ping-pong buffers
 * and ticket word as b200q_static_forward).  Enqueues 14 kernels (13 for b <= 32, where fc1 and the head are one
 * kernel): quantize+conv1, then table + conv for conv2..conv6 (pools fused into conv2 / conv4 / conv6), the conv6->fc1
 * table, fc1, and the fp32 head.  The head is defined to the bit, independently of the batch and of the kernel:
 *   h[k] = f32(max(q[k], zp) - zp) * fc1_scale                       (ReLU + DeQuantStub of fc1's uint8 output q)
 *   p[l] = (((h[16l]*w[16l]) + h[16l+1]*w[16l+1]) + ...) + h[16l+15]*w[16l+15]   for l = 0..31, one rounding per op
 *   s    = butterfly: p[l] += p[l^16], then ^8, ^4, ^2, ^1 (every l ends with the same value)
 *   y[n] = s + fc2_b[n]                                              (w = fc2_w[n], all fp32, no FMA)
 * taps (optional, may be NULL): 7 device pointers receiving the uint8 NHWC output of conv1..conv6 (before ReLU and
 * pooling) and fc1; that route runs the pools as kernels of their own.  A null net, b < 0, a short workspace, layer
 * geometry other than the net's, fc1 other than 4096 -> 512, or null / misaligned fc2 pointers are refused with
 * B200Q_ERR_INVALID_ARG before any CUDA call. */
int b200q_sandwich_forward(const b200q_sandwich_net* net, const float* x, float* logits, int64_t b,
                           void* workspace, int64_t workspace_bytes, uint8_t* const* taps, void* stream);
/* Whole-network executor for b200q_sandwich_forward (as b200q_graph_create; replay and destruction:
 * b200q_graph_launch / b200q_graph_destroy).  The six tables are read during this call only. */
int b200q_sandwich_graph_create(const b200q_sandwich_net* net, const float* x_static, float* logits_static, int64_t b,
                                void* workspace, int64_t workspace_bytes, int flags, void* stream, b200q_graph** out);

/* Measurement hook (bench.py roofline): the same forward with a CUDA event recorded on `stream` before every layer
 * kernel and after the last one; synchronises on the last event and writes b200q_static_num_stages() per-kernel
 * durations in milliseconds to stage_ms_host (HOST memory).  Stage i is named b200q_static_stage_name(i). */
int b200q_static_num_stages(void);
const char* b200q_static_stage_name(int i);
int b200q_static_forward_profiled(const b200q_static_net* net, const float* x, float* logits, int64_t b,
                                  void* workspace, int64_t workspace_bytes, float* stage_ms_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200Q_H_ */
