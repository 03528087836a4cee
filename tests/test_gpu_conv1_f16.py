"""conv1 on fp16 tensor-core MMAs (``conv1_tc_kernel``): bit-exact against the integer oracle on the weights, zero-points
and requantisation constants at the edges of what the kernel accepts.

The kernel multiplies ``x - zp_x`` by ``w`` in fp16 with an fp32 accumulator and takes that accumulator as fbgemm's
``f32(acc - corr)``.  That is exact only because every partial sum is an integer below 2^24; these cases push it: weights
all +127 / all -128 / alternating, input zero-points 0, 255 and odd values with saturated inputs (the largest
``|x - zp|``), ReLU on and off (the sandwich variant's ``lo = 0``), and ``mult`` / ``bdiv`` at the limits of
``B200Q_RQ_BOUNDED`` (``mult`` = 0.5 exactly, ``|bdiv|`` close to 2^21, rounding ties).  Both public entry points are
checked: fp32 NCHW input with the fused quantiser (``b200q_quantize_conv3x3_first``) and uint8 NHWC pixels through a
per-channel table (``b200q_u8_conv3x3_first``).  Batches from 33 images (the first that leaves the CUDA-core kernel)
through one and more rounds of the persistent grid to 16 384; every image is compared up to 160, a seeded sample
including the first, last and grid-boundary images above that."""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SIZES = [33, 147, 148, 149, 2048, 16384]
FULL = 160

# name -> (weights, zp_x, relu, constants, zp_out)
CASES = {
    "pos127-zp0-relu": ("pos", 0, True, "typical", 60),
    "neg128-zp255-relu": ("neg", 255, True, "typical", 17),
    "alt-zp131-norelu": ("alt", 131, False, "typical", 128),
    "rand-zp0-norelu": ("rand", 0, False, "typical", 100),  # the sandwich variant's conv1: zp_x 0, lower clamp 0
    "rand-zp77-edge-relu": ("rand", 77, True, "edge", 40),
    "alt-zp255-edge-norelu": ("alt", 255, False, "edge", 128),
    "pos127-zp1-edge-norelu": ("pos", 1, False, "edge", 0),
    "neg128-zp0-edge-relu": ("neg", 0, True, "edge", 3),
}


def _layer(weights: str, constants: str, zp_out: int):
    """A conv1 layer dict (``ptq.static_qparams`` form) and its input scale."""
    g = torch.Generator().manual_seed(zlib.crc32(f"{weights}/{constants}/{zp_out}".encode()))
    if weights == "pos":
        w = torch.full((64, 3, 3, 3), 127, dtype=torch.int8)
    elif weights == "neg":
        w = torch.full((64, 3, 3, 3), -128, dtype=torch.int8)
    elif weights == "alt":
        w = torch.where(torch.arange(64 * 27).view(64, 3, 3, 3) % 2 == 0, 127, -128).to(torch.int8)
    else:
        w = torch.randint(-128, 128, (64, 3, 3, 3), dtype=torch.int8, generator=g)
    c = torch.arange(64, dtype=torch.float64)
    if constants == "typical":
        s_x, out_scale = 0.02, 0.05
        ws = 0.002 + 0.008 * torch.rand(64, dtype=torch.float64, generator=g)
        bias = (0.1 * torch.randn(64, generator=g)).float()
    else:
        # mult = 0.5 exactly in channels 0, 16, 32, 48 (s_x * ws = 0.5, out_scale 1), halving down to 0.5 * 2^-15; bdiv
        # at +-0.99 * 2^21, 0 (ties of t = acc * 0.5 for odd acc) and half-integers
        s_x, out_scale = 0.25, 1.0
        ws = 2.0 * torch.pow(2.0, -(c % 16))
        atw = (torch.tensor(s_x, dtype=torch.float32) * ws.float()).double()
        bdiv_t = torch.tensor([0.99 * 2 ** 21, -0.99 * 2 ** 21, 0.0, 0.5, -0.5, 1234.25, -77.0, 0.0] * 8,
                              dtype=torch.float64)
        bias = (bdiv_t * atw).float()
    layer = {"w_int8": w, "w_scales": ws, "bias": bias, "out_scale": out_scale, "out_zp": zp_out}
    return layer, s_x


def _sample(b: int) -> np.ndarray:
    if b <= FULL:
        return np.arange(b)
    rng = np.random.default_rng(b)
    picks = {0, 1, 2, b - 2, b - 1, 147, 148, 149, 295, 296}
    picks |= set(int(i) for i in rng.choice(b, 38, replace=False))
    return np.array(sorted(i for i in picks if i < b))


def _fp32_input(b: int, s_x: float, seed: int) -> torch.Tensor:
    """fp32 NCHW: spread over the whole uint8 range, image 0 saturated high, image 1 low, beyond +-1024 / inv_scale."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((b, 3, 32, 32), generator=g) * (120.0 * s_x)
    x[0] = 1.0e6
    x[1] = -1.0e6
    x[-1, :, :16] = 3000.0 * s_x
    x[-1, 1, 16:] = -3000.0 * s_x
    return x


def _u8_input(b: int, seed: int):
    """uint8 NHWC pixels and a [3][256] table that reaches 0 and 255; image 0 all 255, image 1 all 0."""
    g = torch.Generator().manual_seed(seed)
    pix = torch.randint(0, 256, (b, 32, 32, 3), dtype=torch.uint8, generator=g)
    pix[0] = 255
    pix[1] = 0
    lut = torch.randint(0, 256, (3, 256), dtype=torch.uint8, generator=g)
    lut[:, 0] = 0
    lut[:, 255] = 255
    return pix, lut.contiguous()


def _run(case: str, b: int, u8: bool):
    """(device output [b,32,32,64], sampled image indices, oracle output of those images)."""
    from convnet_quantization_b200 import _lib, ops
    from convnet_quantization_b200.packing import PackedConv
    from oracle import int_ops as IO
    weights, zp_x, relu, constants, zp_out = CASES[case]
    layer, s_x = _layer(weights, constants, zp_out)
    pc = PackedConv("conv1", layer, s_x, zp_x, "cuda", relu=relu)
    assert pc.c.rq.flags & _lib.RQ_BOUNDED, "case must stay on the tensor-core kernel"
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    y = torch.empty((b, 32, 32, 64), dtype=torch.uint8, device="cuda")
    idx = _sample(b)
    if u8:
        pix, lut = _u8_input(b, 1000 + b)
        _lib.check(lib.b200q_u8_conv3x3_first(pix.cuda().data_ptr(), y.data_ptr(), b, lut.data_ptr(), pc.ptr(), stream),
                   "u8_conv3x3_first")
        p = pix[torch.from_numpy(idx)].numpy()
        q = np.stack([lut[ch].numpy()[p[..., ch]] for ch in range(3)], axis=-1)
    else:
        x = _fp32_input(b, s_x, 2000 + b)
        _lib.check(lib.b200q_quantize_conv3x3_first(x.cuda().data_ptr(), y.data_ptr(), b, ops._inv_scale(s_x), pc.ptr(),
                                                    stream), "quantize_conv3x3_first")
        xs = x[torch.from_numpy(idx)].permute(0, 2, 3, 1).contiguous().numpy()
        q = IO.quantize_per_tensor(xs, s_x, zp_x)
    want = IO.conv2d_q(q, s_x, zp_x, layer["w_int8"].numpy(), layer["w_scales"].numpy(), layer["bias"].numpy(),
                       layer["out_scale"], zp_out, relu=relu)
    return y, idx, want


@gpu
@pytest.mark.parametrize("u8", [False, True], ids=["fp32", "u8"])
@pytest.mark.parametrize("b", SIZES)
@pytest.mark.parametrize("case", list(CASES))
def test_conv1_tc_bit_exact_vs_oracle(case, b, u8):
    y, idx, want = _run(case, b, u8)
    got = y[torch.from_numpy(idx).cuda()].cpu().numpy()
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{len(bad)} bytes differ, first at (sample, h, w, c) {bad[0].tolist()}: " \
                          f"{got[tuple(bad[0])]} vs {want[tuple(bad[0])]}"


def _profile_cases() -> list:
    """Kernel names, in launch order, of one profiler session over every case at 33 and 2 048 images."""
    from torch.profiler import ProfilerActivity, profile
    runs = [(case, b, u8) for case in CASES for u8 in (False, True) for b in (SIZES[0], 2048)]
    for case, b, u8 in runs:  # first launches (module loading, smem attributes) outside the trace
        _run(case, b, u8)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for case, b, u8 in runs:
            _run(case, b, u8)
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                      and not e.name.startswith(("Memcpy", "Memset"))), key=lambda e: e.time_range.start)
    return [e.name for e in kernels]


@gpu
def test_conv1_cases_launch_the_tensor_core_kernel():
    """Every case of this file, fp32 and uint8 input, at the smallest batch and at one that takes several rounds of the
    persistent grid, launches exactly one kernel: conv1_tc_kernel.  The trace is taken in a child process so that this
    file's profiler session cannot touch the CUPTI state of traces other test files take later."""
    code = ("import json, tests.test_gpu_conv1_f16 as T; "
            "print('NAMES ' + json.dumps(T._profile_cases()))")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    names = json.loads(next(l for l in r.stdout.splitlines() if l.startswith("NAMES "))[6:])
    runs = len(CASES) * 2 * 2
    assert len(names) == runs, (runs, names)
    assert all("conv1_tc_kernel" in n for n in names), names
