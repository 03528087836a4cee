"""GPU parity (bit-exact) of the convolution / linear kernels against the numpy integer restatement."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _packed(qparams, name):
    from convnet_quantization_b200.packing import PackedConv
    order = ["in", "conv1", "conv2", "conv3", "conv4", "conv5", "conv6"]
    prev = order[order.index(name) - 1]
    if prev == "in":
        s, zp = qparams["in_scale"], qparams["in_zp"]
    else:
        s, zp = qparams[prev]["out_scale"], qparams[prev]["out_zp"]
    return PackedConv(name, qparams[name], s, zp, "cuda"), s, zp


def _want_conv(x_u8, s, zp, L):
    from oracle import int_ops as IO
    return IO.conv2d_q(x_u8, s, zp, L["w_int8"], L["w_scales"], L["bias"], L["out_scale"], L["out_zp"], relu=True)


def _rand_u8(shape, seed):
    return torch.randint(0, 256, shape, dtype=torch.uint8, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("b", [1, 5, 40])  # <= 32 images: CUDA-core shape (16 CTAs per image); above: conv1_tc.cu
def test_conv1_first_and_fused(qparams, qparams_np, b):
    from convnet_quantization_b200 import ops, synth
    from oracle import int_ops as IO
    pc, s, zp = _packed(qparams, "conv1")
    x = synth.images_f32(b, seed=11) * 1.5
    xq = IO.quantize_per_tensor(x.numpy().transpose(0, 2, 3, 1), s, zp)
    want = _want_conv(xq, s, zp, qparams_np["conv1"])
    xq4 = ops.quantize_per_tensor(x.cuda(), s, zp, c_pad=4)
    got = ops.conv2d_q(xq4, pc, impl="first").cpu().numpy()
    assert np.array_equal(got, want)
    got_fused = ops.quantize_conv2d_first(x.cuda(), s, pc).cpu().numpy()
    assert np.array_equal(got_fused, want)
    got_simt = ops.conv2d_q(xq4, pc, impl="simt").cpu().numpy()
    assert np.array_equal(got_simt, want)


@pytest.mark.parametrize("name,b", [("conv2", 2), ("conv3", 3), ("conv4", 1), ("conv5", 3), ("conv6", 2)])
def test_conv_simt(qparams, qparams_np, name, b):
    from convnet_quantization_b200 import ops
    pc, s, zp = _packed(qparams, name)
    x = _rand_u8((b, pc.img, pc.img, pc.cin), 5)
    want = _want_conv(x.numpy(), s, zp, qparams_np[name])
    got = ops.conv2d_q(x.cuda(), pc, impl="simt").cpu().numpy()
    assert np.array_equal(got, want)


@pytest.mark.parametrize("name", ["conv2", "conv3", "conv4", "conv5", "conv6"])
@pytest.mark.parametrize("b", [1, 2, 3, 37, 300])
def test_conv_tc(qparams, qparams_np, name, b):
    """tcgen05 implicit-GEMM conv: odd batches, multi-tile-per-CTA batches, saturating inputs."""
    from convnet_quantization_b200 import ops
    pc, s, zp = _packed(qparams, name)
    x = _rand_u8((b, pc.img, pc.img, pc.cin), 7 * b)
    got = ops.conv2d_q(x.cuda(), pc, impl="tc")
    torch.cuda.synchronize()
    got = got.cpu().numpy()
    want = _want_conv(x.numpy(), s, zp, qparams_np[name])
    bad = got != want
    assert not bad.any(), f"{name} b={b}: {int(bad.sum())} / {bad.size} mismatches; first at {np.argwhere(bad)[:5].tolist()}"


@pytest.mark.parametrize("b", [1, 64, 129, 1000])
def test_linear_tc_fc1(qparams, qparams_np, b):
    from convnet_quantization_b200 import ops
    from convnet_quantization_b200.packing import PackedLinear
    from oracle import int_ops as IO
    s, zp = qparams["conv6"]["out_scale"], qparams["conv6"]["out_zp"]
    L = qparams_np["fc1"]
    pl = PackedLinear("fc1", qparams["fc1"], s, zp, "cuda", relu=True, nhwc_from=(256, 4, 4))
    x = _rand_u8((b, 4, 4, 256), b)  # NHWC activations as the engine holds them
    want = IO.linear_q(IO.flatten_nchw(x.numpy()), s, zp, L["w_int8"], L["w_scales"], L["bias"], L["out_scale"],
                       L["out_zp"], relu=True)
    xf = x.reshape(b, 4096).cuda()
    got_simt = ops.linear_q(xf, pl, impl="simt").cpu().numpy()
    assert np.array_equal(got_simt, want)
    got = ops.linear_q(xf, pl, impl="tc")
    torch.cuda.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("b", [1, 7, 200])
def test_fc2_and_dequant(qparams, qparams_np, b):
    from convnet_quantization_b200 import ops
    from convnet_quantization_b200.packing import PackedLinear
    from oracle import int_ops as IO
    s, zp = qparams["fc1"]["out_scale"], qparams["fc1"]["out_zp"]
    L = qparams_np["fc2"]
    pl = PackedLinear("fc2", qparams["fc2"], s, zp, "cuda", relu=False)
    x = _rand_u8((b, 512), b + 1)
    want_q = IO.linear_q(x.numpy(), s, zp, L["w_int8"], L["w_scales"], L["bias"], L["out_scale"], L["out_zp"])
    got_q = ops.linear_q(x.cuda(), pl, impl="simt").cpu().numpy()
    assert np.array_equal(got_q, want_q)
    got = ops.linear_dequant(x.cuda(), pl, L["out_scale"]).cpu().numpy()
    assert np.array_equal(got, IO.dequantize(want_q, L["out_scale"], L["out_zp"]))


@pytest.mark.parametrize("b,k,n", [(1, 4096, 512), (33, 4096, 512), (64, 512, 10)])
def test_linear_dynamic(b, k, n):
    """quantized::linear_dynamic vs the live torch op (tolerance: 1e-3 relative, BASELINE north_star)."""
    from convnet_quantization_b200 import ops
    torch.backends.quantized.engine = "fbgemm"
    g = torch.Generator().manual_seed(b + k)
    lin = torch.nn.Linear(k, n)
    with torch.no_grad():
        lin.weight.copy_(torch.randn(n, k, generator=g) * 0.05)
        lin.bias.copy_(torch.randn(n, generator=g) * 0.1)
    qlin = torch.ao.quantization.quantize_dynamic(torch.nn.Sequential(lin), {torch.nn.Linear}, dtype=torch.qint8)[0]
    x = torch.randn(b, k, generator=g).abs() * 0.7
    want = qlin(x)
    w = qlin.weight()
    dw = ops.DynamicLinearWeights(w.int_repr(), w.q_scale(), qlin.bias(), "cuda")
    for _ in range(2):  # twice: scratch counter must self-reset
        got = ops.linear_dynamic(x.cuda(), dw).cpu()
        assert torch.equal(got, want)  # bit-exact (fbgemm's fma forms), far inside the 1e-3 the north star asks for


@pytest.mark.parametrize("name", ["conv2", "conv3", "conv4", "conv5", "conv6"])
@pytest.mark.parametrize("pool", [False, True])
@pytest.mark.parametrize("b", [1, 2])
def test_conv_tiny_batches(qparams, qparams_np, name, pool, b):
    """One or two images take the CUDA-core kernel (csrc/conv_small.cu: K split across the lanes, zero-point halo in
    shared memory, exact requantisation, pooling on the requantised bytes): bit-exact against the integer oracle and
    identical to what the tensor-core kernels give for the same images inside a larger batch."""
    from convnet_quantization_b200 import ops
    from oracle import int_ops as IO
    pc, s, zp = _packed(qparams, name)
    x = _rand_u8((b, pc.img, pc.img, pc.cin), 31 * b + len(name))
    x[0, :2] = 255  # saturating rows at the top border
    x[-1, -1] = 0
    want = _want_conv(x.numpy(), s, zp, qparams_np[name])
    if pool:
        want = IO.max_pool2x2(want)
    got = ops.conv2d_q(x.cuda(), pc, pool2x2=pool, impl="tc")
    torch.cuda.synchronize()
    bad = got.cpu().numpy() != want
    assert not bad.any(), f"{name} b={b} pool={pool}: {int(bad.sum())} / {bad.size} mismatches; first at {np.argwhere(bad)[:5].tolist()}"
    big = torch.cat([x, _rand_u8((5, pc.img, pc.img, pc.cin), 3)]).cuda()  # 6-7 images: small-batch tensor-core shape
    assert torch.equal(ops.conv2d_q(big, pc, pool2x2=pool, impl="tc")[:b], got)


@pytest.mark.parametrize("name", ["conv2", "conv4", "conv6"])
@pytest.mark.parametrize("b", [1, 3, 150, 151])
def test_conv_tc_fused_pool(qparams, qparams_np, name, b):
    """conv + aten::quantized_max_pool2d fused in the epilogue == pooling the oracle's conv output."""
    from convnet_quantization_b200 import ops
    from oracle import int_ops as IO
    pc, s, zp = _packed(qparams, name)
    x = _rand_u8((b, pc.img, pc.img, pc.cin), 3 * b + 1)
    got = ops.conv2d_q(x.cuda(), pc, pool2x2=True, impl="tc")
    torch.cuda.synchronize()
    want = IO.max_pool2x2(_want_conv(x.numpy(), s, zp, qparams_np[name]))
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("b,gain", [(1, 1.0), (3, 1.0), (149, 1.0), (300, 1.0), (5, 4.0)])
def test_conv12_fused(qparams, qparams_np, b, gain):
    """quantize + conv1 + conv2 + 2x2 max-pool in one kernel (conv1's output never leaves shared memory) == the oracle's
    four ops, including CTAs that process several images and inputs far outside the calibrated range."""
    from convnet_quantization_b200 import ops, synth
    from oracle import int_ops as IO
    pc1, s, zp = _packed(qparams, "conv1")
    pc2, s1, zp1 = _packed(qparams, "conv2")
    x = synth.images_f32(b, seed=100 + b) * gain
    xq = IO.quantize_per_tensor(x.numpy().transpose(0, 2, 3, 1), s, zp)
    c1 = _want_conv(xq, s, zp, qparams_np["conv1"])
    want = IO.max_pool2x2(_want_conv(c1, s1, zp1, qparams_np["conv2"]))
    got = ops.quantize_conv2d_conv2d_pool(x.cuda(), s, pc1, pc2)
    torch.cuda.synchronize()
    got = got.cpu().numpy()
    bad = got != want
    assert not bad.any(), f"b={b}: {int(bad.sum())} / {bad.size} mismatches; first at {np.argwhere(bad)[:5].tolist()}"
    # and the two-kernel path it replaces
    two = ops.conv2d_q(ops.quantize_conv2d_first(x.cuda(), s, pc1), pc2, pool2x2=True).cpu().numpy()
    assert np.array_equal(two, want)


@pytest.mark.parametrize("name,b,pool", [("conv3", 900, False), ("conv5", 1300, False), ("conv6", 1300, True),
                                         ("conv4", 450, True), ("conv2", 701, True), ("conv2", 450, False)])
def test_conv_tc_many_bands_per_cta(qparams, qparams_np, name, b, pool):
    """Batches large enough that every persistent CTA (conv2 + pool: every CTA PAIR of conv_halo2.cu, with an odd image
    count so that the last pair is half empty) walks several bands: the weight ring wraps, the activation
    buffers and the TMEM slots change phase parity, the pipelined epilogue runs in steady state.  Oracle comparison on
    a random subset of images (the numpy restatement is the slow side), full-tensor comparison against the same
    kernel run on the subset alone."""
    from convnet_quantization_b200 import ops
    from oracle import int_ops as IO
    pc, s, zp = _packed(qparams, name)
    x = _rand_u8((b, pc.img, pc.img, pc.cin), 1000 + b)
    got = ops.conv2d_q(x.cuda(), pc, pool2x2=pool, impl="tc")
    torch.cuda.synchronize()
    got = got.cpu().numpy()
    idx = torch.randperm(b, generator=torch.Generator().manual_seed(b))[:48].sort().values
    want = _want_conv(x[idx].numpy(), s, zp, qparams_np[name])
    if pool:
        want = IO.max_pool2x2(want)
    assert np.array_equal(got[idx.numpy()], want)


def test_alternate_instantiations_stay_bit_exact():
    """The A-B switches of the DEVELOPMENT library select other template instantiations of the same kernels (16 epilogue
    warps x 8 channels in the halo kernels, the fused conv1+conv2 kernel, the generic shifted-TMA kernel for every
    conv); they are read once per process, so they are exercised in a child process: whole-net logits must equal the
    product configuration's bit for bit.  The product library must ignore every such variable."""
    import subprocess
    import sys
    code = (
        "import torch, warnings; warnings.filterwarnings('ignore')\n"
        "from convnet_quantization_b200 import synth\n"
        "from convnet_quantization_b200.models.static_ptq_model import StaticPTQModel\n"
        "m = StaticPTQModel(device='cuda'); m.fp32_model.load_state_dict(synth.make_state_dict(0)); q = m.quantize()\n"
        "y = q.engine.forward(synth.images_f32(333, seed=77).cuda()); torch.cuda.synchronize()\n"
        "import hashlib; print(hashlib.sha256(y.cpu().numpy().tobytes()).hexdigest())\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    digests = {}
    from convnet_quantization_b200 import _lib
    dev = str(_lib.build(dev=True))  # the switches exist in the development library only (-DB200Q_DEV)
    for name, env in (("default", {}), ("dev", {"B200Q_LIB": dev}), ("ew16", {"B200Q_LIB": dev, "B200Q_HALO_EW": "16"}),
                      ("fuse12", {"B200Q_LIB": dev, "B200Q_FUSE12": "1"}), ("no_halo", {"B200Q_LIB": dev, "B200Q_NO_HALO": "1"}),
                      ("no_cta2", {"B200Q_LIB": dev, "B200Q_NO_CTA2": "1"}), ("h2_slots4", {"B200Q_LIB": dev, "B200Q_H2_SLOTS": "4"}),
                      ("no_small", {"B200Q_LIB": dev, "B200Q_NO_SMALL": "1"}),
                      ("ignored", {"B200Q_HALO_DEBUG": "14", "B200Q_PAIR_DEBUG": "46", "B200Q_NO_HALO": "1"})):
        e = dict(os.environ)
        e.update(env)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=e, cwd=root, timeout=600)
        assert r.returncode == 0, f"{name}: {r.stderr[-1500:]}"
        digests[name] = r.stdout.strip().splitlines()[-1]
    assert len(set(digests.values())) == 1, digests  # "ignored": the product library has no such switches


@pytest.mark.parametrize("name,pool", [("conv2", False), ("conv2", True), ("conv3", False), ("conv4", False), ("conv4", True),
                                       ("conv5", False), ("conv6", False), ("conv6", True)])
@pytest.mark.parametrize("b", [3, 37])
def test_conv_tc_without_host_mirrors(qparams, qparams_np, name, pool, b):
    """Documented ABI branch (include/b200q.h, b200q_requant.mult_host): with corr_host / mult_host / bdiv_host NULL the
    kernels that take their constants as kernel parameters are not eligible and b200q_conv3x3_tc must run the
    shifted-TMA kernel that stages the DEVICE tables through shared memory (igemm_tc.cu, nine border classes) - all
    five geometries, pool on and off."""
    import ctypes as C
    from convnet_quantization_b200 import _lib
    from oracle import int_ops as IO
    pc, s, zp = _packed(qparams, name)
    bare = _lib.Conv3x3.from_buffer_copy(pc.c)
    bare.corr_host = None
    bare.rq.mult_host = None
    bare.rq.bdiv_host = None
    x = _rand_u8((b, pc.img, pc.img, pc.cin), 31 * b + len(name)).cuda()
    o = pc.img // 2 if pool else pc.img
    y = torch.empty((b, o, o, pc.cout), dtype=torch.uint8, device="cuda")
    lib = _lib.load()
    n0 = lib.b200q_launch_count()
    _lib.check(lib.b200q_conv3x3_tc(x.data_ptr(), y.data_ptr(), b, C.byref(bare), int(pool),
                                    torch.cuda.current_stream().cuda_stream), "conv3x3_tc")
    torch.cuda.synchronize()
    assert lib.b200q_launch_count() == n0 + 1
    want = _want_conv(x.cpu().numpy(), s, zp, qparams_np[name])
    if pool:
        want = IO.max_pool2x2(want)
    assert np.array_equal(y.cpu().numpy(), want)
    # same answer as the default (host-mirror) kernels
    from convnet_quantization_b200 import ops
    assert torch.equal(ops.conv2d_q(x, pc, pool2x2=pool), y)


@pytest.mark.parametrize("b,k,n,relu", [(1, 4096, 512, True), (127, 4096, 512, False), (128, 4096, 512, True),
                                         (300, 4096, 512, False), (1, 512, 10, False), (129, 512, 10, False),
                                         (1000, 512, 10, True), (40, 1024, 16, False)])
def test_linear_dynamic_tensor_core(b, k, n, relu):
    """quantized::linear_dynamic on the tensor cores (quantising producer, fp32 epilogue) vs the live torch op, BIT-exact:
    partial / several / many 128-row tiles, both N tiles (512 = two accumulators, <= 16 = TMA zero-filled rows)."""
    from convnet_quantization_b200 import ops
    from oracle import int_ops as IO
    torch.backends.quantized.engine = "fbgemm"
    g = torch.Generator().manual_seed(b + k + n)
    lin = torch.nn.Linear(k, n)
    with torch.no_grad():
        lin.weight.copy_(torch.randn(n, k, generator=g) * 0.05)
        lin.bias.copy_(torch.randn(n, generator=g) * 0.1)
    qlin = torch.ao.quantization.quantize_dynamic(torch.nn.Sequential(lin), {torch.nn.Linear}, dtype=torch.qint8)[0]
    x = torch.randn(b, k, generator=g) * 0.7 + 0.2
    want = qlin(x)
    if relu:
        want = torch.relu(want)
    w = qlin.weight()
    dw = ops.DynamicLinearWeights(w.int_repr(), w.q_scale(), qlin.bias(), "cuda")
    for _ in range(2):  # twice: the scratch counter must self-reset
        got = ops.linear_dynamic(x.cuda(), dw, relu=relu).cpu()
        assert torch.equal(got, want), f"{int((got != want).sum())} of {want.numel()} outputs differ from the live torch op"
    # the activation qparams the kernel used are the ATen ones, and against the integer restatement fed the SAME
    # quantised activations the result is exact up to the fp32 output rounding
    qp = dw.last_qparams().cpu()
    s, z = torch._choose_qparams_per_tensor(x, True)
    assert qp[2].item() == np.float32(s) and int(qp[4]) == z
    mine = IO.linear_dynamic(x.numpy(), w.int_repr().numpy(), w.q_scale(), qlin.bias().detach().numpy())
    if relu:
        mine = np.maximum(mine, 0)
    assert np.array_equal(got.numpy(), mine)
    assert tuple(ops.linear_dynamic(x[:0].cuda(), dw).shape) == (0, n)
