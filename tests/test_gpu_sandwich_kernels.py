"""The per-layer sandwich variant (``CustomQuantizationModel(mode="sandwich")``, ``B200SandwichQuantizedNet``) against
the integer oracle (``oracle/int_ops.py``) in every kernel its forward reaches.

The sandwich runs the static net's conv and linear kernels with other settings: ReLU fusion off (``rq.relu = 0``, so
the epilogues clamp at ``lo = 0`` instead of ``zp_out``) and, for conv2-conv6 and fc1, input zero-point 0 (all
zero-point corrections are zero, pads hold 0).  About half of each int8 layer's output bytes lie below ``zp_out``,
which a ReLU-on test clamps away.  So every case here is fed what the layer sees in production (random bytes through
the previous boundary table ``net.luts[i - 1]``: many zeros), plus one saturated image and one half-zero image, and
asserts that its reference output reaches both clamps.

Batch sizes are derived from the SM count with the kernel-selection rules of ``b200q_conv3x3_tc`` /
``b200q_linear_tc`` (``csrc/igemm_tc.cu``), ``conv3x3_halo_dispatch`` (``csrc/conv_halo.cu``) and
``conv_first_impl`` (``csrc/simt.cu``); ``test_sandwich_cases_run_the_kernels_they_claim`` checks in a profiler trace
that each case really runs the kernel named here.  Both sides are fed the same ``ptq.calibrate_sandwich`` parameters,
so host-dependent calibration cannot make them differ; the layers under test are the ones ``B200SandwichQuantizedNet``
packs (``net.convs``, ``net.fc1``, ``net.luts``)."""
import re

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CONVS = ("conv2", "conv3", "conv4", "conv5", "conv6")
POOLS = {"conv2": (True, False), "conv3": (False,), "conv4": (True, False), "conv5": (False,), "conv6": (True, False)}
SIZES = ("1", "2", "3", "small_last", "band_first", "band_odd", "many")
CONV3_SIZES = ("nbi3_below", "nbi3_above")  # conv3: one image per band below 3 * SMs, three from there on
CONV1_SIZES = (1, 32, 33, 2048)  # conv1_kernel<C1_IN_F32, 1> up to CONV1_TINY_MAX_B = 32 images (simt.cu), conv1_tc_kernel above
FC1_SIZES = ("1", "7", "narrow_last", "wide_first")
NET_SIZES = ("1", "2", "pair_first", "nbi3_above", "fc1_wide")
WHOLE = 160   # up to this many images every output is compared with the oracle; above it, a sample
SAMPLE = 48


def _cases():
    out = []
    for layer in CONVS:
        for pool in POOLS[layer]:
            for size in SIZES + (CONV3_SIZES if layer == "conv3" else ()):
                out.append(pytest.param(layer, pool, size, id=f"{layer}-{'pool' if pool else 'nopool'}-{size}"))
    return out


CASES = _cases()


# ---------------------------------------------------------------------------------------------- kernel selection
def _geom(layer):
    from convnet_quantization_b200.packing import CONV_GEOMETRY
    return CONV_GEOMETRY[layer]  # (cin, cout, img)


def _small_last(layer, sms):
    """Largest batch for which ``b200q_conv3x3_tc`` runs the small-batch ``igemm_tc_kernel`` (N tile 64): the layer cut
    into 128-pixel x 64-channel tiles fits in two waves of CTAs (37 / 74 / 74 / 148 / 148 on 148 SMs)."""
    _, cout, img = _geom(layer)

    def m_tiles(b):
        return b * 8 if img == 32 else b * 2 if img == 16 else (b + 1) // 2

    b = 3
    while m_tiles(b + 1) * (cout // 64) <= 2 * sms:
        b += 1
    return b


def _conv_batch(layer, size, sms):
    last = _small_last(layer, sms)
    first = last + 1
    return {
        "1": 1, "2": 2,                      # conv3x3_tiny_kernel (CONV_TINY_MAX_B = 2)
        "3": 3, "small_last": last,          # igemm_tc_kernel<..., 64>
        "band_first": first,                 # first batch on the band-resident kernels
        # odd: the last CTA pair (conv2 + pool) or the last pair band (conv5 / conv6, 4 images) is partly empty
        "band_odd": first + 1 if first % 2 == 0 else first + 2,
        "nbi3_below": 3 * sms - 1, "nbi3_above": 3 * sms + 1,
        "many": 9 * sms + 5,                 # every persistent CTA (pair) walks three or more bands
    }[size]


def _conv_plan(layer, pool, b, sms):
    """(kernel-name pattern, images per band, bands in flight at once) that ``b200q_conv3x3_tc`` selects.  Patterns
    are matched against demangled names with the spaces and ``(int)`` / ``(bool)`` casts removed."""
    cin, cout, img = _geom(layer)
    p = "true" if pool else "false"
    if b <= 2:
        return rf"conv3x3_tiny_kernel<{img},{cin},{cout},{p}>", 1, b
    if b <= _small_last(layer, sms):
        return rf"igemm_tc_kernel<{img},{cin},{cout},false,{p},(true|false),64>", 1, b
    if layer == "conv2" and pool:
        return r"conv_halo2_kernel<(true|false),8>", 2, sms // 2
    if layer == "conv2":
        return r"conv_halo_kernel<32,64,64,1,false,(true|false),8>", 1, sms
    if layer == "conv3":
        nbi = 1 if b < 3 * sms else 3
        return rf"conv_halo_kernel<16,64,128,{nbi},false,(true|false),8>", nbi, sms
    if layer == "conv4":
        return rf"conv_halo_kernel<16,128,128,1,{p},(true|false),8>", 1, sms
    return rf"conv_pair_kernel<{cin},{p},(true|false)>", 4, sms // 2


def _conv1_kernel(b):
    return r"conv1_kernel<1,1>" if b <= 32 else r"conv1_tc_kernel<(true|false),false>"


def _fc1_batch(size, sms):
    narrow_last = 128 * (sms // 8)  # eight 64-column CTA tiles per 128 rows while they fit on the SMs
    return {"1": 1, "7": 7, "narrow_last": narrow_last, "wide_first": narrow_last + 1}[size]


def _fc1_kernel(b, sms):
    return rf"igemm_tc_kernel<0,4096,512,false,false,true,{64 if b <= 128 * (sms // 8) else 0}>"


def _net_batch(size, sms):
    return {"1": 1, "2": 2, "pair_first": sms + 1, "nbi3_above": 3 * sms + 1,
            "fc1_wide": _fc1_batch("wide_first", sms)}[size]


def _plain_kernel_name(name):
    return (name.replace(" ", "").replace("(int)", "").replace("(bool)0", "false").replace("(bool)1", "true"))


# ---------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def sp(fp32_net):
    from convnet_quantization_b200 import ptq, synth
    return ptq.calibrate_sandwich(fp32_net, synth.calibration_batches())


@pytest.fixture(scope="module")
def sp_np(sp):
    from tests.conftest import qparams_to_numpy
    return qparams_to_numpy(sp)


@pytest.fixture(scope="module")
def net(sp):
    from convnet_quantization_b200.models._gpu_modules import B200SandwichQuantizedNet
    return B200SandwichQuantizedNet(sp, "cuda")


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ---------------------------------------------------------------------------------------------- inputs and oracle
def _layer_input(lut, shape, seed):
    """What the layer sees in production: random bytes through the boundary table before it (ReLU: many zeros).  One
    saturated image and one image whose top half is zero; a single image gets two saturated rows and a zero half."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = lut.cuda()[torch.randint(0, 256, shape, generator=g, device="cuda")]
    img = shape[1]
    if shape[0] == 1:
        x[0, :2] = 255
        x[0, img // 2:] = 0
    else:
        x[0] = 255
        x[-1, : img // 2] = 0
    return x.contiguous()


def _conv1_input(b, seed, w_int8):
    """Synthetic images x 3 (the quantised input saturates at both ends).  Image 0's top twelve rows hold, for output
    channels 0-39, the 3x3 patch matched to that channel's weights (255 where w > 0, else 0), which drives those
    channels to 255."""
    from convnet_quantization_b200 import synth
    x = synth.images_f32(b, seed=seed) * 3
    for co in range(40):
        r, c = 1 + 3 * (co // 10), 1 + 3 * (co % 10)
        x[0, :, r - 1:r + 2, c - 1:c + 2] = torch.where(w_int8[co] > 0, 10.0, -10.0)
    return x


def _oracle_conv(x_u8, L, pool):
    from oracle import int_ops as IO
    y = IO.conv2d_q(x_u8, L["in_scale"], L["in_zp"], L["w_int8"], L["w_scales"], L["bias"], L["out_scale"],
                    L["out_zp"], relu=False)
    return IO.max_pool2x2(y) if pool else y


def _sample(b, band, walkers, seed):
    """Every image up to ``WHOLE``; above, a fixed sample of at least ``SAMPLE`` images: the first and last two, both
    sides of the first band boundary and of every boundary between rounds of the persistent CTAs, the last (maybe
    partial) band, and seeded random images."""
    if b <= WHOLE:
        return np.arange(b)
    idx = {0, 1, b - 2, b - 1, band - 1, band}
    step = band * walkers
    for lo in range(step, b, step):
        idx.update((lo - 1, lo))
    idx.update(range((b - 1) // band * band, b))
    rest = np.setdiff1d(np.arange(b), np.fromiter(idx, dtype=np.int64))
    fill = np.random.default_rng(seed).choice(rest, size=max(0, SAMPLE - len(idx)), replace=False)
    return np.sort(np.concatenate([np.fromiter(idx, dtype=np.int64), fill]))


def _assert_reaches_both_clamps(want, zp_out, what):
    below = float((want < zp_out).mean())
    assert (want == 0).any() and (want == 255).any() and below >= 0.10, (
        f"{what}: the reference must reach both clamps (has 0: {bool((want == 0).any())}, has 255: "
        f"{bool((want == 255).any())}, below zp_out={zp_out}: {below:.1%})")


def _assert_equal(got, want, what):
    bad = got != want
    assert not bad.any(), f"{what}: {int(bad.sum())} / {bad.size} mismatches; first at {np.argwhere(bad)[:5].tolist()}"


# ---------------------------------------------------------------------------------------------- per-layer sweep
@pytest.mark.parametrize("layer,pool,size", CASES)
def test_sandwich_conv_layer(net, sp_np, sms, layer, pool, size):
    """conv2-conv6 with ReLU off and input zero-point 0, in every kernel shape: bit-exact against the integer oracle
    (all images up to 64, a sample above), and the sampled images equal to the same op run on them alone."""
    from convnet_quantization_b200 import ops
    i = int(layer[-1]) - 1
    pc, L = net.convs[i], sp_np[layer]
    assert pc.c.rq.relu == 0 and pc.zp_x == 0
    b = _conv_batch(layer, size, sms)
    _, band, walkers = _conv_plan(layer, pool, b, sms)
    x = _layer_input(net.luts[i - 1], (b, pc.img, pc.img, pc.cin), seed=1000 * i + b)
    got = ops.conv2d_q(x, pc, pool2x2=pool)
    idx = _sample(b, band, walkers, seed=b)
    want = _oracle_conv(x[idx].cpu().numpy(), L, pool)
    what = f"{layer} pool={pool} b={b}"
    _assert_reaches_both_clamps(want, L["out_zp"], what)
    _assert_equal(got[idx].cpu().numpy(), want, what)
    if len(idx) < b:
        alone = ops.conv2d_q(x[idx].contiguous(), pc, pool2x2=pool)
        assert torch.equal(got[idx], alone), f"{what}: sampled images differ from the same op run on them alone"


@pytest.mark.parametrize("b", CONV1_SIZES)
def test_sandwich_conv1(net, sp, sp_np, sms, b):
    """Fused QuantStub + conv1 (input zero-point from calibration, ReLU off) on saturating synthetic images."""
    from convnet_quantization_b200 import ops
    from oracle import int_ops as IO
    pc, L = net.convs[0], sp_np["conv1"]
    assert pc.c.rq.relu == 0
    x = _conv1_input(b, seed=20 + b, w_int8=sp["conv1"]["w_int8"])
    got = ops.quantize_conv2d_first(x.cuda(), L["in_scale"], pc)
    idx = _sample(b, 1, sms, seed=b)  # conv1_tc_kernel: one image at a time per persistent CTA
    xq = IO.quantize_per_tensor(x[idx].numpy().transpose(0, 2, 3, 1), L["in_scale"], L["in_zp"])
    want = _oracle_conv(xq, L, pool=False)
    _assert_reaches_both_clamps(want, L["out_zp"], f"conv1 b={b}")
    _assert_equal(got[idx].cpu().numpy(), want, f"conv1 b={b}")
    if len(idx) < b:
        assert torch.equal(got[idx], ops.quantize_conv2d_first(x[idx].cuda(), L["in_scale"], pc))


@pytest.mark.parametrize("size", FC1_SIZES)
def test_sandwich_fc1(net, sp_np, sms, size):
    """fc1 (ReLU off, input zero-point 0) with 64- and 256-column CTA tiles; the input is conv6's pooled NHWC output,
    so the packed weight columns are permuted (``nhwc_from``) and the oracle flattens NCHW."""
    from convnet_quantization_b200 import ops
    from oracle import int_ops as IO
    L = sp_np["fc1"]
    assert net.fc1.c.rq.relu == 0 and net.fc1.zp_x == 0
    b = _fc1_batch(size, sms)
    x = _layer_input(net.luts[5], (b, 4, 4, 256), seed=77 + b)
    got = ops.linear_q(x.reshape(b, 4096), net.fc1).cpu().numpy()
    want = IO.linear_q(IO.flatten_nchw(x.cpu().numpy()), L["in_scale"], L["in_zp"], L["w_int8"], L["w_scales"], L["bias"],
                       L["out_scale"], L["out_zp"], relu=False)
    _assert_reaches_both_clamps(want, L["out_zp"], f"fc1 b={b}")
    _assert_equal(got, want, f"fc1 b={b}")


# ---------------------------------------------------------------------------------------------- kernel selection check
def test_sandwich_cases_run_the_kernels_they_claim(net, sms):
    """One profiler pass over every case of this file: each launches exactly one kernel, the one its batch size is
    meant to select (template arguments included), with ReLU off in every layer.  A threshold change that moves a case
    to another kernel fails here instead of silently leaving a kernel untested."""
    from torch.profiler import ProfilerActivity, profile
    from convnet_quantization_b200 import ops
    assert all(pc.c.rq.relu == 0 for pc in net.convs) and net.fc1.c.rq.relu == 0
    assert all(pc.zp_x == 0 for pc in net.convs[1:]) and net.fc1.zp_x == 0
    runs = []  # (label, expected pattern, callable)
    for p in CASES:
        layer, pool, size = p.values
        pc = net.convs[int(layer[-1]) - 1]
        b = _conv_batch(layer, size, sms)
        x = torch.zeros((b, pc.img, pc.img, pc.cin), dtype=torch.uint8, device="cuda")
        runs.append((f"{layer} pool={pool} b={b}", _conv_plan(layer, pool, b, sms)[0],
                     lambda x=x, pc=pc, pool=pool: ops.conv2d_q(x, pc, pool2x2=pool)))
    for b in CONV1_SIZES:
        x = torch.zeros((b, 3, 32, 32), dtype=torch.float32, device="cuda")
        runs.append((f"conv1 b={b}", _conv1_kernel(b), lambda x=x: ops.quantize_conv2d_first(x, 0.04, net.convs[0])))
    for size in FC1_SIZES:
        b = _fc1_batch(size, sms)
        x = torch.zeros((b, 4096), dtype=torch.uint8, device="cuda")
        runs.append((f"fc1 b={b}", _fc1_kernel(b, sms), lambda x=x: ops.linear_q(x, net.fc1)))
    for _, _, run in runs:  # first launches (module loading, smem attributes) outside the trace
        run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _, _, run in runs:
            run()
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                      and not e.name.startswith(("Memcpy", "Memset"))), key=lambda e: e.time_range.start)
    names = [_plain_kernel_name(e.name) for e in kernels]
    assert len(names) == len(runs), f"{len(runs)} cases, {len(names)} kernels: {names}"
    wrong = [(label, pattern, name) for (label, pattern, _), name in zip(runs, names) if not re.search(pattern, name)]
    assert not wrong, "cases that did not run the kernel they claim:\n" + "\n".join(map(str, wrong))


# ---------------------------------------------------------------------------------------------- whole net
def _net_sample(b, seed, boundaries=()):
    if b <= SAMPLE:
        return np.arange(b)
    idx = {0, 1, b - 1} | {i for lo in boundaries for i in (lo - 1, lo) if 0 < lo < b}
    rest = np.setdiff1d(np.arange(b), np.fromiter(idx, dtype=np.int64))
    fill = np.random.default_rng(seed).choice(rest, size=max(0, SAMPLE - len(idx)), replace=False)
    return np.sort(np.concatenate([np.fromiter(idx, dtype=np.int64), fill]))


def _assert_logits_close(got, want, what):
    """fc2 is an fp32 GEMM (cuBLAS here, float64 in the oracle): within 1e-3 of the largest absolute logit."""
    np.testing.assert_allclose(got, want, rtol=1e-3, atol=1e-3 * float(np.abs(want).max()), err_msg=what)


@pytest.mark.parametrize("size", NET_SIZES)
def test_sandwich_forward_with_taps(net, sp, sp_np, sms, size):
    """Un-pooled route: all seven int8 layer outputs bit-exact against ``IO.sandwich_forward`` on a sample, logits
    within tolerance; the production route (pools fused into conv2/4/6) returns the same logits bit for bit."""
    from oracle import int_ops as IO
    b = _net_batch(size, sms)
    x = _conv1_input(b, seed=300 + b, w_int8=sp["conv1"]["w_int8"])
    logits, taps = net.forward_with_taps(x)
    idx = _net_sample(b, seed=b)
    want_taps = {}
    want = IO.sandwich_forward(x[idx].numpy(), sp_np, want_taps)
    assert set(taps) == set(want_taps) == {"conv1", "conv2", "conv3", "conv4", "conv5", "conv6", "fc1"}
    for n, t in taps.items():
        _assert_equal(t[idx].cpu().numpy(), want_taps[n], f"{n} tap, b={b}")
    _assert_logits_close(logits[idx].cpu().numpy(), want, f"logits, b={b}")
    assert torch.equal(net(x.cuda()), logits)


def test_sandwich_forward_device_and_host_inputs(net, sp_np, sms):
    """``net(x)`` on a CUDA batch past the fc1 tile switch, and on a host batch that the two-stream pipeline cuts into
    two full chunks and a split tail: logits against the oracle on a sample that includes the chunk boundaries."""
    from convnet_quantization_b200 import synth
    from oracle import int_ops as IO
    b = _fc1_batch("wide_first", sms) + 2 * sms + 1
    x = synth.images_f32(b, seed=41) * 2.5
    got = net(x.cuda()).cpu().numpy()
    idx = _net_sample(b, seed=1)
    _assert_logits_close(got[idx], IO.sandwich_forward(x[idx].numpy(), sp_np), f"CUDA input, b={b}")

    b = 2 * net.HOST_CHUNK + 4 * net.TAIL_MIN + 7
    chunks = list(net._chunks(b))
    assert len(chunks) == 4 and chunks[1][1] == net.HOST_CHUNK and chunks[3][1] < chunks[2][1] < net.HOST_CHUNK, chunks
    x = synth.images_f32(b, seed=42) * 2.5
    got = net(x)
    assert not got.is_cuda
    idx = _net_sample(b, seed=2, boundaries=[lo for lo, _ in chunks])
    _assert_logits_close(got[idx].numpy(), IO.sandwich_forward(x[idx].numpy(), sp_np), f"host input, b={b}")
