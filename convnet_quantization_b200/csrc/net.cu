// Whole static-PTQ SimpleConvNet forward: the call order of models/baseline_model.py:58-83 on the converted
// (int8) model, as one C-ABI call that enqueues every kernel on the caller's stream.  No allocation, no sync.
#include <new>

#include "common.cuh"

using namespace b200q;

namespace {
constexpr int64_t BYTES_PER_IMG = 65536;  // largest activation: conv1/conv2 output, 32*32*64 uint8

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

int copy_tap(uint8_t* const* taps, int idx, const void* src, int64_t bytes, cudaStream_t s) {
  if (taps == nullptr || taps[idx] == nullptr) return 0;
  return check_cuda(cudaMemcpyAsync(taps[idx], src, (size_t)bytes, cudaMemcpyDeviceToDevice, s), "tap copy");
}
}  // namespace

extern "C" int64_t b200q_static_workspace_bytes(int64_t b) {
  if (b < 0) return B200Q_ERR_INVALID_ARG;
  return 2 * align_up(b * BYTES_PER_IMG, 1024) + 1024 /*alignment slack*/ + 1024 /*ticket word of the small-batch head*/;
}

namespace {
// One entry per kernel the fused forward enqueues; order == launch order.  In -DB200Q_DEV builds B200Q_FUSE12=1 runs conv1 and conv2 as ONE
// kernel (conv12_fused.cu: bit-exact, but measured slower than the two kernels - 1.05 ms against 0.39 + 0.48 ms at batch
// 16 384 - because all its requantisation work lands on eight 128-register epilogue warps; see DESIGN.md 5.7).
const char* const kStageNamesFused[] = {"conv1_conv2_pool", "conv3", "conv4_pool", "conv5",
                                        "conv6_pool",       "fc1",   "fc2_dequant"};
const char* const kStageNamesSplit[] = {"quant_conv1", "conv2_pool", "conv3", "conv4_pool",
                                        "conv5",       "conv6_pool", "fc1",   "fc2_dequant"};
constexpr int kMaxStages = 8;
constexpr bool kEagerPdlDefault = false;

bool fuse12_enabled() {
#ifndef B200Q_DEV
  return false;  // conv12_fused.cu is not part of the product library
#endif
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200Q_FUSE12");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}
bool fuse12_ok(const b200q_static_net* net) {
  const b200q_conv3x3 &a = net->conv[0], &b = net->conv[1];
  return fuse12_enabled() && a.corr_host && b.corr_host && a.rq.mult_host && a.rq.bdiv_host && b.rq.mult_host &&
         b.rq.bdiv_host && (a.rq.flags & B200Q_RQ_BOUNDED) && a.cin == 4 && a.cout == 64 && a.img == 32 && b.cin == 64 &&
         b.cout == 64 && b.img == 32 && b.zp_x == a.rq.zp_out;
}

// taps == nullptr: production path, 2x2 max-pools fused into the conv2/conv4/conv6 epilogues (8 kernels).
// taps != nullptr: parity path, every reference op materialised (unfused convs + stand-alone pools) and copied out.
// Programmatic dependent launch between the kernels of an EAGER forward (not only inside captured graphs): each layer
// kernel's prologue (up to 144 KB of weights into shared memory per CTA, TMEM allocation, pad initialisation) then
// overlaps the tail of the previous layer.  Development builds: B200Q_EAGER_PDL=0|1 overrides (A-B timing).
bool eager_pdl() {
#ifdef B200Q_DEV
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200Q_EAGER_PDL");
    v = e ? (e[0] == '1') : kEagerPdlDefault;
  }
  return v == 1;
#else
  return kEagerPdlDefault;
#endif
}
#ifdef B200Q_DEV
thread_local int g_stop_after = 0;
#endif
struct PdlScope {  // sets the thread's PDL launch flag for the lifetime of the scope
  bool prev, active;
  explicit PdlScope(bool on) : prev(pdl_enabled()), active(on) {
    if (active) pdl_set(true);
  }
  ~PdlScope() {
    if (active) pdl_set(prev);
  }
};

// ticket_is_zero: the caller is capturing a graph and guarantees the head kernel's ticket word (last 1 KiB of the
// workspace) already holds 0 (it was zeroed before the capture and every forward leaves it zero); otherwise it is
// cleared here.
// eval (production path only, no taps / events): the head kernel also counts (b200q_static_evaluate); logits may be
// nullptr then.
int forward_impl(const b200q_static_net* net, const float* x, float* logits, int64_t b, void* workspace,
                 int64_t workspace_bytes, uint8_t* const* taps, cudaEvent_t* ev, void* stream,
                 const uint8_t* x_u8 = nullptr, const uint8_t* lut_host = nullptr, bool ticket_is_zero = false,
                 const EvalArgs* eval = nullptr) {
  B200Q_REQUIRE(net && (((x || x_u8) && (logits || eval) && workspace) || b == 0), "static_forward: null pointer");
  B200Q_REQUIRE(b >= 0, "static_forward: negative batch");
  if (b == 0) return 0;
  B200Q_REQUIRE(workspace_bytes >= b200q_static_workspace_bytes(b), "static_forward: workspace too small (%lld < %lld)",
                (long long)workspace_bytes, (long long)b200q_static_workspace_bytes(b));
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* A = reinterpret_cast<uint8_t*>(align_up((int64_t)(uintptr_t)workspace, 1024));
  uint8_t* B = A + align_up(b * BYTES_PER_IMG, 1024);
  int rc;
  int stage = 0;
#ifdef B200Q_DEV  // timing experiments: stop the production forward after g_stop_after kernels (scripts/graph_breakdown.py)
#define STEP(call) do { rc = (call); if (rc) return rc; if (!taps && g_stop_after && ++steps_done >= g_stop_after) return 0; } while (0)
  int steps_done = 0;
#else
#define STEP(call) do { rc = (call); if (rc) return rc; } while (0)
#endif
#define MARK() do { if (ev) B200Q_CUDA(cudaEventRecord(ev[stage++], s)); } while (0)

  if (taps == nullptr) {
    PdlScope pdl(!ev && !ticket_is_zero && eager_pdl());  // (a capture sets the flag itself, from its B200Q_GRAPH_PDL flag)
    MARK();
    if (x_u8) {  // uint8 data path: table look-up instead of the fp32 quantiser, same kernel otherwise
      STEP(b200q_u8_conv3x3_first(x_u8, A, b, lut_host, &net->conv[0], stream));
      MARK();
      STEP(b200q_conv3x3_tc(A, B, b, &net->conv[1], 1, stream));
#ifdef B200Q_DEV
    } else if (fuse12_ok(net)) {
      STEP(b200q_conv12_fused(x, B, b, net->in_inv_scale, &net->conv[0], &net->conv[1], stream));  // -> [b,16,16,64]
#endif
    } else {
      STEP(b200q_quantize_conv3x3_first(x, A, b, net->in_inv_scale, &net->conv[0], stream));
      MARK();
      STEP(b200q_conv3x3_tc(A, B, b, &net->conv[1], 1, stream));  // -> [b,16,16,64]
    }
    MARK();
    STEP(b200q_conv3x3_tc(B, A, b, &net->conv[2], 0, stream));  // -> [b,16,16,128]
    MARK();
    STEP(b200q_conv3x3_tc(A, B, b, &net->conv[3], 1, stream));  // -> [b,8,8,128]
    MARK();
    STEP(b200q_conv3x3_tc(B, A, b, &net->conv[4], 0, stream));  // -> [b,8,8,256]
    MARK();
    STEP(b200q_conv3x3_tc(A, B, b, &net->conv[5], 1, stream));  // -> [b,4,4,256]
    MARK();
    if (!ev) {  // (the profiled forward keeps the two-kernel head: its stage list is fixed)
      // small batches: fc1 + ReLU + fc2 + dequantize as ONE launch (simt.cu fc_head_small_kernel)
      unsigned int* ticket = reinterpret_cast<unsigned int*>(B + align_up(b * BYTES_PER_IMG, 1024));
      int hrc = 0;
      if (b <= 32 && !ticket_is_zero) B200Q_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s));
#ifdef B200Q_DEV
      if (g_stop_after && steps_done >= g_stop_after) return 0;
#endif
      if (fc_head_small_dispatch(B, A, logits, ticket, b, &net->fc1, &net->fc2, net->out_scale, eval, s, &hrc) == 0)
        return hrc;
    }
    STEP(b200q_linear_tc(B, A, b, &net->fc1, stream));
    MARK();
    if (eval)
      STEP(linear_head_eval(A, logits, b, &net->fc2, net->out_scale, *eval, s));
    else
      STEP(b200q_linear_dequant(A, logits, b, &net->fc2, net->out_scale, stream));
    MARK();
    return 0;
  }

  if (taps[0]) STEP(b200q_quantize_nchw_to_nhwc(x, taps[0], b, 3, 32, 32, 4, net->in_inv_scale, net->in_zp, stream));
  STEP(b200q_quantize_conv3x3_first(x, A, b, net->in_inv_scale, &net->conv[0], stream));
  STEP(copy_tap(taps, 1, A, b * 65536, s));
  STEP(b200q_conv3x3_tc(A, B, b, &net->conv[1], 0, stream));
  STEP(copy_tap(taps, 2, B, b * 65536, s));
  STEP(b200q_max_pool2x2_nhwc(B, A, b, 32, 32, 64, stream));
  STEP(copy_tap(taps, 3, A, b * 16384, s));
  STEP(b200q_conv3x3_tc(A, B, b, &net->conv[2], 0, stream));
  STEP(copy_tap(taps, 4, B, b * 32768, s));
  STEP(b200q_conv3x3_tc(B, A, b, &net->conv[3], 0, stream));
  STEP(copy_tap(taps, 5, A, b * 32768, s));
  STEP(b200q_max_pool2x2_nhwc(A, B, b, 16, 16, 128, stream));
  STEP(copy_tap(taps, 6, B, b * 8192, s));
  STEP(b200q_conv3x3_tc(B, A, b, &net->conv[4], 0, stream));
  STEP(copy_tap(taps, 7, A, b * 16384, s));
  STEP(b200q_conv3x3_tc(A, B, b, &net->conv[5], 0, stream));
  STEP(copy_tap(taps, 8, B, b * 16384, s));
  STEP(b200q_max_pool2x2_nhwc(B, A, b, 8, 8, 256, stream));
  STEP(copy_tap(taps, 9, A, b * 4096, s));
  STEP(b200q_linear_tc(A, B, b, &net->fc1, stream));
  STEP(copy_tap(taps, 10, B, b * 512, s));
  if (taps[11]) STEP(b200q_linear_simt(B, taps[11], b, &net->fc2, stream));
  STEP(b200q_linear_dequant(B, logits, b, &net->fc2, net->out_scale, stream));
#undef STEP
#undef MARK
  return 0;
}
}  // namespace

extern "C" int b200q_static_forward(const b200q_static_net* net, const float* x, float* logits, int64_t b,
                                    void* workspace, int64_t workspace_bytes, uint8_t* const* taps, void* stream) {
  return forward_impl(net, x, logits, b, workspace, workspace_bytes, taps, nullptr, stream);
}

// Stage list of the production forward (seven stages with B200Q_FUSE12=1, else eight).
extern "C" int b200q_static_forward_u8(const b200q_static_net* net, const uint8_t* x_nhwc, const uint8_t* lut_host,
                                       float* logits, int64_t b, void* workspace, int64_t workspace_bytes,
                                       void* stream) {
  B200Q_REQUIRE(lut_host != nullptr && (x_nhwc != nullptr || b == 0), "static_forward_u8: null pointer");
  return forward_impl(net, nullptr, logits, b, workspace, workspace_bytes, nullptr, nullptr, stream, x_nhwc, lut_host);
}

namespace {
int check_evaluate(const b200q_static_net* net, const int64_t* labels, int64_t b, const uint64_t* counters,
                   const int32_t* pred) {
  B200Q_REQUIRE(labels != nullptr && counters != nullptr, "static_evaluate: null labels or counters");
  B200Q_REQUIRE(b >= 0, "static_evaluate: negative batch");
  B200Q_REQUIRE((uintptr_t)labels % 8 == 0 && (uintptr_t)counters % 8 == 0 && (uintptr_t)pred % 4 == 0,
                "static_evaluate: misaligned labels, counters or pred");
  B200Q_REQUIRE(net != nullptr, "static_evaluate: null net");
  B200Q_REQUIRE(net->fc2.k == 512 && net->fc2.n == 10, "static_evaluate: the counting head needs fc2 k=512 n=10 (k=%d n=%d)",
                net->fc2.k, net->fc2.n);
  return 0;
}
}  // namespace

extern "C" int b200q_static_evaluate(const b200q_static_net* net, const float* x, const int64_t* labels, int64_t b,
                                     uint64_t* counters, int32_t* pred, float* logits, void* workspace,
                                     int64_t workspace_bytes, void* stream) {
  if (int rc = check_evaluate(net, labels, b, counters, pred)) return rc;
  const EvalArgs eval{labels, reinterpret_cast<unsigned long long*>(counters), pred};
  return forward_impl(net, x, logits, b, workspace, workspace_bytes, nullptr, nullptr, stream, nullptr, nullptr, false,
                      &eval);
}

extern "C" int b200q_static_evaluate_u8(const b200q_static_net* net, const uint8_t* x_nhwc, const uint8_t* lut_host,
                                        const int64_t* labels, int64_t b, uint64_t* counters, int32_t* pred,
                                        float* logits, void* workspace, int64_t workspace_bytes, void* stream) {
  if (int rc = check_evaluate(net, labels, b, counters, pred)) return rc;
  B200Q_REQUIRE(lut_host != nullptr && (x_nhwc != nullptr || b == 0), "static_evaluate_u8: null pointer");
  const EvalArgs eval{labels, reinterpret_cast<unsigned long long*>(counters), pred};
  return forward_impl(net, nullptr, logits, b, workspace, workspace_bytes, nullptr, nullptr, stream, x_nhwc, lut_host,
                      false, &eval);
}

// ---------------------------------------------------------------------------------------------------- sandwich net
namespace {
int check_sandwich(const b200q_sandwich_net* net, const float* x, const float* logits, int64_t b, const void* workspace,
                   int64_t workspace_bytes) {
  B200Q_REQUIRE(net != nullptr, "sandwich_forward: null net");
  B200Q_REQUIRE(b >= 0, "sandwich_forward: negative batch");
  B200Q_REQUIRE((x && logits && workspace) || b == 0, "sandwich_forward: null pointer");
  B200Q_REQUIRE(workspace_bytes >= b200q_static_workspace_bytes(b),
                "sandwich_forward: workspace too small (%lld < %lld)", (long long)workspace_bytes,
                (long long)b200q_static_workspace_bytes(b));
  static const int kGeom[6][3] = {{4, 64, 32}, {64, 64, 32}, {64, 128, 16}, {128, 128, 16}, {128, 256, 8}, {256, 256, 8}};
  for (int i = 0; i < 6; ++i) {
    const b200q_conv3x3& c = net->conv[i];
    B200Q_REQUIRE(c.cin == kGeom[i][0] && c.cout == kGeom[i][1] && c.img == kGeom[i][2],
                  "sandwich_forward: conv%d geometry (cin %d, cout %d, img %d) is not the net's (%d, %d, %d)", i + 1,
                  c.cin, c.cout, c.img, kGeom[i][0], kGeom[i][1], kGeom[i][2]);
  }
  B200Q_REQUIRE(net->fc1.k == 4096 && net->fc1.n == 512, "sandwich_forward: fc1 must be 4096 -> 512 (got %d -> %d)",
                net->fc1.k, net->fc1.n);
  B200Q_REQUIRE(net->fc2_w && net->fc2_b && (uintptr_t)net->fc2_w % 16 == 0 && (uintptr_t)net->fc2_b % 4 == 0,
                "sandwich_forward: fc2 (fp32 [10][512] + [10]) needs non-null pointers, weights 16-byte aligned");
  return 0;
}

// Same buffers as forward_impl: A / B ping-pong of b x 64 KiB, the head's ticket word after B.  Every table reads the
// conv output and writes the buffer that conv read; taps != nullptr materialises the un-pooled conv outputs.
int sandwich_impl(const b200q_sandwich_net* net, const float* x, float* logits, int64_t b, void* workspace,
                  int64_t workspace_bytes, uint8_t* const* taps, void* stream, bool ticket_is_zero = false) {
  if (int rc = check_sandwich(net, x, logits, b, workspace, workspace_bytes)) return rc;
  if (b == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* A = reinterpret_cast<uint8_t*>(align_up((int64_t)(uintptr_t)workspace, 1024));
  uint8_t* B = A + align_up(b * BYTES_PER_IMG, 1024);
  const b200q_conv3x3* L = net->conv;
  const int zp_h = net->fc1.rq.zp_out;
  int rc;
#define STEP(call) do { rc = (call); if (rc) return rc; } while (0)
#define LUT(i, src, dst, bytes_per_img) STEP(b200q_lut_u8(src, dst, b * (bytes_per_img), net->lut_host[i], stream))

  if (taps == nullptr) {
    PdlScope pdl(!ticket_is_zero && eager_pdl());  // (a capture sets the flag itself, from its B200Q_GRAPH_PDL flag)
    STEP(b200q_quantize_conv3x3_first(x, A, b, net->in_inv_scale, &L[0], stream));  // -> [b,32,32,64]
    LUT(0, A, B, 65536);
    STEP(b200q_conv3x3_tc(B, A, b, &L[1], 1, stream));  // -> [b,16,16,64]
    LUT(1, A, B, 16384);
    STEP(b200q_conv3x3_tc(B, A, b, &L[2], 0, stream));  // -> [b,16,16,128]
    LUT(2, A, B, 32768);
    STEP(b200q_conv3x3_tc(B, A, b, &L[3], 1, stream));  // -> [b,8,8,128]
    LUT(3, A, B, 8192);
    STEP(b200q_conv3x3_tc(B, A, b, &L[4], 0, stream));  // -> [b,8,8,256]
    LUT(4, A, B, 16384);
    STEP(b200q_conv3x3_tc(B, A, b, &L[5], 1, stream));  // -> [b,4,4,256]
    LUT(5, A, B, 4096);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(B + align_up(b * BYTES_PER_IMG, 1024));
    if (b <= 32 && !ticket_is_zero) B200Q_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s));
    int hrc = 0;  // small batches: fc1 and the head in one kernel
    if (sandwich_head_small_dispatch(B, A, logits, ticket, b, &net->fc1, net->fc2_w, net->fc2_b, net->fc1_scale, s,
                                     &hrc) == 0)
      return hrc;
    STEP(b200q_linear_tc(B, A, b, &net->fc1, stream));
    STEP(sandwich_head(A, logits, b, net->fc2_w, net->fc2_b, zp_h, net->fc1_scale, s));
    return 0;
  }

  STEP(b200q_quantize_conv3x3_first(x, A, b, net->in_inv_scale, &L[0], stream));
  STEP(copy_tap(taps, 0, A, b * 65536, s));
  LUT(0, A, B, 65536);
  STEP(b200q_conv3x3_tc(B, A, b, &L[1], 0, stream));
  STEP(copy_tap(taps, 1, A, b * 65536, s));
  STEP(b200q_max_pool2x2_nhwc(A, B, b, 32, 32, 64, stream));
  LUT(1, B, A, 16384);
  STEP(b200q_conv3x3_tc(A, B, b, &L[2], 0, stream));
  STEP(copy_tap(taps, 2, B, b * 32768, s));
  LUT(2, B, A, 32768);
  STEP(b200q_conv3x3_tc(A, B, b, &L[3], 0, stream));
  STEP(copy_tap(taps, 3, B, b * 32768, s));
  STEP(b200q_max_pool2x2_nhwc(B, A, b, 16, 16, 128, stream));
  LUT(3, A, B, 8192);
  STEP(b200q_conv3x3_tc(B, A, b, &L[4], 0, stream));
  STEP(copy_tap(taps, 4, A, b * 16384, s));
  LUT(4, A, B, 16384);
  STEP(b200q_conv3x3_tc(B, A, b, &L[5], 0, stream));
  STEP(copy_tap(taps, 5, A, b * 16384, s));
  STEP(b200q_max_pool2x2_nhwc(A, B, b, 8, 8, 256, stream));
  LUT(5, B, A, 4096);
  STEP(b200q_linear_tc(A, B, b, &net->fc1, stream));
  STEP(copy_tap(taps, 6, B, b * 512, s));
  STEP(sandwich_head(B, logits, b, net->fc2_w, net->fc2_b, zp_h, net->fc1_scale, s));
#undef LUT
#undef STEP
  return 0;
}
}  // namespace

extern "C" int b200q_sandwich_forward(const b200q_sandwich_net* net, const float* x, float* logits, int64_t b,
                                      void* workspace, int64_t workspace_bytes, uint8_t* const* taps, void* stream) {
  return sandwich_impl(net, x, logits, b, workspace, workspace_bytes, taps, stream);
}

// ---------------------------------------------------------------------------------------------------- executor
struct b200q_graph {
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  int64_t batch = 0;
  int kernels = 0;  // kernels one replay launches (b200q_launch_count bookkeeping)
};

namespace {
// One capture body for every forward: fwd(ticket_is_zero) enqueues the whole forward on `stream`.  An eager forward
// first (per-device kernel attributes, lazy module loading and the tensor-map encoder are first-use work that does not
// belong inside a capture; it also leaves the small-batch head's ticket word zero), then the capture with the
// B200Q_GRAPH_PDL flag, counting the kernels one replay launches.
template <class Fwd>
int capture_graph(int flags, void* stream, int64_t b, b200q_graph** out, Fwd&& fwd) {
  cudaStream_t s = (cudaStream_t)stream;
  int rc = fwd(false);
  if (rc) return rc;
  B200Q_CUDA(cudaStreamSynchronize(s));
  B200Q_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  pdl_set((flags & B200Q_GRAPH_PDL) != 0);
#ifdef B200Q_DEV
  g_stop_after = (flags >> 8) & 15;  // development library: capture only the first k kernels (timing breakdown)
#endif
  const uint64_t launches0 = b200q_launch_count();
  rc = fwd(/*ticket_is_zero=*/true);
  const int captured_kernels = (int)(b200q_launch_count() - launches0);
  pdl_set(false);
#ifdef B200Q_DEV
  g_stop_after = 0;
#endif
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(s, &graph);  // always end the capture, also after a failed enqueue
  if (rc) {
    if (graph) cudaGraphDestroy(graph);
    (void)cudaGetLastError();
    return rc;
  }
  B200Q_CUDA(e);
  b200q_graph* g = new (std::nothrow) b200q_graph();
  if (!g) {
    cudaGraphDestroy(graph);
    set_error("graph_create: out of host memory");
    return B200Q_ERR_INVALID_ARG;
  }
  g->graph = graph;
  g->batch = b;
  g->kernels = captured_kernels;
  if (int irc = check_cuda(cudaGraphInstantiate(&g->exec, graph, 0), "cudaGraphInstantiate")) {
    cudaGraphDestroy(graph);
    delete g;
    return irc;
  }
  *out = g;
  return 0;
}

int check_graph_args(const void* net, bool inputs, const float* logits_static, const void* workspace, int64_t b,
                     void* stream, b200q_graph** out) {
  B200Q_REQUIRE(out != nullptr, "graph_create: null out");
  *out = nullptr;
  B200Q_REQUIRE(net && inputs && logits_static && workspace && b > 0, "graph_create: null pointer or empty batch");
  B200Q_REQUIRE(stream != nullptr, "graph_create: the legacy default stream cannot be captured; pass a created stream");
  return 0;
}

// Both input kinds of the static net: x (fp32 NCHW) or x_u8 + lut_host (uint8 NHWC pixels, HOST table).
int graph_create_impl(const b200q_static_net* net, const float* x, const uint8_t* x_u8, const uint8_t* lut_host,
                      float* logits_static, int64_t b, void* workspace, int64_t workspace_bytes, int flags, void* stream,
                      b200q_graph** out) {
  if (int rc = check_graph_args(net, x || (x_u8 && lut_host), logits_static, workspace, b, stream, out)) return rc;
  return capture_graph(flags, stream, b, out, [&](bool ticket_is_zero) {
    return forward_impl(net, x, logits_static, b, workspace, workspace_bytes, nullptr, nullptr, stream, x_u8, lut_host,
                        ticket_is_zero);
  });
}
}  // namespace

extern "C" int b200q_graph_create(const b200q_static_net* net, const float* x_static, float* logits_static, int64_t b,
                                  void* workspace, int64_t workspace_bytes, int flags, void* stream, b200q_graph** out) {
  return graph_create_impl(net, x_static, nullptr, nullptr, logits_static, b, workspace, workspace_bytes, flags, stream,
                           out);
}

extern "C" int b200q_graph_create_u8(const b200q_static_net* net, const uint8_t* x_nhwc_static, const uint8_t* lut_host,
                                     float* logits_static, int64_t b, void* workspace, int64_t workspace_bytes, int flags,
                                     void* stream, b200q_graph** out) {
  return graph_create_impl(net, nullptr, x_nhwc_static, lut_host, logits_static, b, workspace, workspace_bytes, flags,
                           stream, out);
}

extern "C" int b200q_sandwich_graph_create(const b200q_sandwich_net* net, const float* x_static, float* logits_static,
                                           int64_t b, void* workspace, int64_t workspace_bytes, int flags, void* stream,
                                           b200q_graph** out) {
  if (int rc = check_graph_args(net, x_static != nullptr, logits_static, workspace, b, stream, out)) return rc;
  if (int rc = check_sandwich(net, x_static, logits_static, b, workspace, workspace_bytes)) return rc;
  return capture_graph(flags, stream, b, out, [&](bool ticket_is_zero) {
    return sandwich_impl(net, x_static, logits_static, b, workspace, workspace_bytes, nullptr, stream, ticket_is_zero);
  });
}

extern "C" int b200q_graph_launch(b200q_graph* g, void* stream) {
  B200Q_REQUIRE(g && g->exec, "graph_launch: null graph");
  B200Q_CUDA(cudaGraphLaunch(g->exec, (cudaStream_t)stream));
  note_graph_replay(g->kernels);
  return 0;
}

extern "C" int b200q_graph_destroy(b200q_graph* g) {
  if (!g) return 0;
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->graph) cudaGraphDestroy(g->graph);
  delete g;
  return 0;
}

extern "C" int b200q_static_num_stages(void) { return fuse12_enabled() ? 7 : 8; }
extern "C" const char* b200q_static_stage_name(int i) {
  const int n = b200q_static_num_stages();
  if (i < 0 || i >= n) return "";
  return fuse12_enabled() ? kStageNamesFused[i] : kStageNamesSplit[i];
}

extern "C" int b200q_static_forward_profiled(const b200q_static_net* net, const float* x, float* logits, int64_t b,
                                             void* workspace, int64_t workspace_bytes, float* stage_ms_host,
                                             void* stream) {
  B200Q_REQUIRE(stage_ms_host != nullptr, "static_forward_profiled: null stage_ms_host");
  const int kNumStages = b200q_static_num_stages();
  B200Q_REQUIRE(!fuse12_enabled() || fuse12_ok(net),
                "static_forward_profiled: net does not qualify for the fused conv1+conv2 stage; unset B200Q_FUSE12");
  // one event set per (thread, device), created on first use and kept for the life of the thread: a device change
  // never re-creates (and so never leaks) events
  constexpr int kMaxDevices = 64;
  static thread_local cudaEvent_t ev_all[kMaxDevices][kMaxStages + 1];
  static thread_local bool ev_ready[kMaxDevices] = {};
  int dev = -1;
  B200Q_CUDA(cudaGetDevice(&dev));
  B200Q_REQUIRE(dev >= 0 && dev < kMaxDevices, "static_forward_profiled: device index %d not supported", dev);
  if (!ev_ready[dev]) {
    for (int i = 0; i <= kMaxStages; ++i) B200Q_CUDA(cudaEventCreate(&ev_all[dev][i]));
    ev_ready[dev] = true;
  }
  cudaEvent_t* ev = ev_all[dev];
  for (int i = 0; i < kNumStages; ++i) stage_ms_host[i] = 0.f;
  if (b == 0) return 0;
  int rc = forward_impl(net, x, logits, b, workspace, workspace_bytes, nullptr, ev, stream);
  if (rc) return rc;
  B200Q_CUDA(cudaEventSynchronize(ev[kNumStages]));
  for (int i = 0; i < kNumStages; ++i) B200Q_CUDA(cudaEventElapsedTime(&stage_ms_host[i], ev[i], ev[i + 1]));
  return 0;
}
