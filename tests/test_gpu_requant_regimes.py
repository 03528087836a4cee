"""Every int8 conv and linear kernel instantiation of the product library in each requantisation form its pack-time
flags select (``tests/_requant_regimes.py``), bit-exact against the integer oracle.

The cases cover conv2-conv6 with and without the fused pool, at batch sizes derived from the SM count so that each
kernel shape runs: the CUDA-core kernel (1, 2 images), the small-batch N-tile-64 ``igemm_tc_kernel`` (3 and the
largest batch it takes), the band-resident kernels (first and odd batch past it, conv3's one and three images per band,
and a batch in which every persistent CTA walks several bands).  The layers without host copies of their constants run
the large-batch ``igemm_tc_kernel``; fc1 runs both CTA tilings and the 512 -> 64 linear that ``b200q_linear_tc`` also
accepts runs both ``CHECK`` instantiations.  ``test_regime_cases_run_the_kernels_they_claim`` checks in a profiler
trace that each case launches the instantiation named here, ``CHECK`` argument included;
``tests/test_requant_regimes.py`` checks that these names cover every instantiation compiled into the library."""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import _requant_regimes as R

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CONVS = ("conv2", "conv3", "conv4", "conv5", "conv6")
FULL = ("acc22", "range_mixed", "bdiv_edge")      # every kernel shape
EXACT = ("mult", "mult_many", "bdiv_over", "corr")  # exact form only: the CHECK = true kernels FULL runs already
SIZES = ("1", "2", "3", "small_last", "band_first", "band_odd", "many")
EXACT_SIZES = ("2", "3", "160", "many")
MIRRORLESS = ("acc22", "range_mixed", "mult")
MIRRORLESS_SIZES = ("band_first", "many")
FC1_SIZES = ("narrow_last", "wide_first")
LIN512_SIZES = (5, 300)
LIN512_REGIMES = ("acc22", "range_mixed", "mult")


def _conv_cases():
    out = []
    for regime in FULL + EXACT:
        for layer in CONVS:
            for pool in (False, True):
                if regime in FULL:
                    sizes = SIZES + (("160",) if regime == "range_mixed" else ())
                    sizes += ("nbi3_below", "nbi3_above") if layer == "conv3" else ()
                else:
                    sizes = EXACT_SIZES + (("nbi3_above",) if layer == "conv3" else ())
                for size in sizes:
                    out.append((layer, pool, size, regime))
    return out


CONV_CASES = _conv_cases()
MIRRORLESS_CASES = [(layer, pool, size, regime) for regime in MIRRORLESS for layer in CONVS for pool in (False, True)
                    for size in MIRRORLESS_SIZES]
LINEAR_CASES = ([("fc1", size, regime) for regime in R.REGIMES for size in FC1_SIZES]
                + [("lin512", b, regime) for regime in LIN512_REGIMES for b in LIN512_SIZES])


def _cid(case):
    return "-".join("pool" if v is True else "nopool" if v is False else str(v) for v in case)


@functools.lru_cache(maxsize=None)
def _layer(name, regime):
    return R.regime_layer(name, regime)


@functools.lru_cache(maxsize=None)
def _packed(name, regime, mirrors=True):
    from convnet_quantization_b200 import _lib
    from convnet_quantization_b200.packing import PackedConv, PackedLinear
    layer, s_x, zp_x = _layer(name, regime)
    relu = R.regime_relu(regime)
    if name in R.LINEARS:
        p = PackedLinear(name, layer, s_x, zp_x, "cuda", relu=relu, nhwc_from=(256, 4, 4) if name == "fc1" else None)
    else:
        p = PackedConv(name, layer, s_x, zp_x, "cuda", relu=relu)
    assert p.c.rq.flags == R.REGIMES[regime][0], (name, regime, p.c.rq.flags)
    if not mirrors:
        bare = _lib.Conv3x3.from_buffer_copy(p.c)
        bare.corr_host = None
        bare.rq.mult_host = None
        bare.rq.bdiv_host = None
        return p, bare
    return p, p.c


def _lin_batch(name, size, sms):
    return R._fc1_batch(size, sms) if name == "fc1" else size


def expected_kernels(sms):
    """(case label, demangled instantiation it must launch) for every case of this file, in the order
    ``_profile_cases`` runs them."""
    out = []
    for layer, pool, size, regime in CONV_CASES:
        b = R._conv_batch(layer, size, sms)
        out.append((f"{layer} pool={pool} b={b} {regime}", R._conv_plan(layer, pool, b, sms, R.REGIMES[regime][0])[0]))
    for layer, pool, size, regime in MIRRORLESS_CASES:
        b = R._conv_batch(layer, size, sms)
        out.append((f"{layer} pool={pool} b={b} {regime} no host mirrors",
                    R._conv_plan(layer, pool, b, sms, R.REGIMES[regime][0], mirrors=False)[0]))
    for name, size, regime in LINEAR_CASES:
        b = _lin_batch(name, size, sms)
        out.append((f"{name} b={b} {regime}", R._linear_kernel(name, b, sms, R.REGIMES[regime][0])))
    return out


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ---------------------------------------------------------------------------------------------- checks
def _run_conv(x, c, b, pool, img, cout):
    import ctypes as C
    from convnet_quantization_b200 import _lib
    o = img // 2 if pool else img
    y = torch.empty((b, o, o, cout), dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().b200q_conv3x3_tc(x.data_ptr(), y.data_ptr(), b, C.byref(c), int(pool),
                                            torch.cuda.current_stream().cuda_stream), "conv3x3_tc")
    return y


def _assert_not_vacuous(want, regime, what):
    values = np.unique(want)
    assert len(values) >= 16, f"{what}: the reference has only {len(values)} distinct values"
    if not R.regime_relu(regime):
        assert values[0] == 0 and values[-1] == 255, f"{what}: the reference must reach both clamps ({values[[0, -1]]})"


def _assert_range_test_mixed(x_u8, zp_x, w, band_kernel, what):
    """range_mixed: the quantity the kernel range-tests leaves +-2^22 for some compared elements and not for others."""
    frac = float(R.out_of_range(R.range_tested(x_u8, zp_x, w, band_kernel)).mean())
    assert 0.0 < frac < 1.0, f"{what}: fraction of accumulators outside +-2^22 is {frac}"


def _assert_equal(got, want, what):
    bad = got != want
    assert not bad.any(), f"{what}: {int(bad.sum())} / {bad.size} mismatches; first at {np.argwhere(bad)[:5].tolist()}"


def _check_conv(layer, pool, size, regime, sms, mirrors):
    from oracle import int_ops as IO
    cin, cout, img = R._geom(layer)
    b = R._conv_batch(layer, size, sms)
    flags = R.REGIMES[regime][0]
    kernel, band, walkers = R._conv_plan(layer, pool, b, sms, flags, mirrors)
    L, s_x, zp_x = _layer(layer, regime)
    _, c = _packed(layer, regime, mirrors)
    x = R.regime_input(regime, (b, img, img, cin), seed=31 * b + cin, device="cuda")
    got = _run_conv(x, c, b, pool, img, cout)
    idx = R._sample(b, band, walkers, seed=b)
    xs = x[torch.from_numpy(idx).cuda()].cpu().numpy()
    want = IO.conv2d_q(xs, s_x, zp_x, L["w_int8"].numpy(), L["w_scales"].numpy(), L["bias"].numpy(), L["out_scale"],
                       L["out_zp"], relu=R.regime_relu(regime))
    if pool:
        want = IO.max_pool2x2(want)
    what = f"{layer} pool={pool} b={b} {regime} ({kernel})"
    _assert_not_vacuous(want, regime, what)
    if regime == "range_mixed" and b > 2:
        _assert_range_test_mixed(xs, zp_x, L["w_int8"].numpy(), not kernel.startswith("igemm"), what)
    _assert_equal(got[torch.from_numpy(idx).cuda()].cpu().numpy(), want, what)
    if len(idx) < b:
        alone = _run_conv(x[torch.from_numpy(idx).cuda()].contiguous(), c, len(idx), pool, img, cout)
        assert torch.equal(got[torch.from_numpy(idx).cuda()], alone), f"{what}: sampled images differ run alone"


@gpu
@pytest.mark.parametrize("layer,pool,size,regime", CONV_CASES, ids=[_cid(c) for c in CONV_CASES])
def test_regime_conv_layer(sms, layer, pool, size, regime):
    """conv2-conv6, pool on and off, in every kernel shape and requantisation regime: bit-exact against the integer
    oracle (every image up to 160, a sample with band and round boundaries above), the sampled images equal to the
    same op run on them alone.  ``range_mixed`` saturates every 7th image, so in the many-band batches the exact-form
    fall-back fires in CTAs that walk several bands while their accumulator slots change parity."""
    _check_conv(layer, pool, size, regime, sms, mirrors=True)


@gpu
@pytest.mark.parametrize("layer,pool,size,regime", MIRRORLESS_CASES, ids=[_cid(c) for c in MIRRORLESS_CASES])
def test_regime_conv_without_host_mirrors(sms, layer, pool, size, regime):
    """Null host mirrors (``b200q_requant.mult_host``): past the small-batch sizes ``b200q_conv3x3_tc`` runs the
    large-batch ``igemm_tc_kernel`` (resident weights for conv2-conv4, streamed for conv5 / conv6), in the
    ``CHECK = false`` form for conv2 with ``acc22``."""
    _check_conv(layer, pool, size, regime, sms, mirrors=False)


@gpu
@pytest.mark.parametrize("name,size,regime", LINEAR_CASES, ids=[_cid(c) for c in LINEAR_CASES])
def test_regime_linear(sms, name, size, regime):
    """fc1 (NHWC column order, both CTA tilings) and the 512 -> 64 linear in each regime: bit-exact against the oracle
    and equal to the CUDA-core kernel (``impl="simt"``)."""
    from convnet_quantization_b200 import ops
    from oracle import int_ops as IO
    k, n = R.LINEARS[name]
    b = _lin_batch(name, size, sms)
    L, s_x, zp_x = _layer(name, regime)
    p, _ = _packed(name, regime)
    if name == "fc1":
        x = R.regime_input(regime, (b, 4, 4, 256), seed=b, device="cuda")
        xf = x.reshape(b, k)
        xo = IO.flatten_nchw(x.cpu().numpy())  # the oracle's NCHW flatten order
    else:
        xf = R.regime_input(regime, (b, k), seed=b, device="cuda")
        xo = xf.cpu().numpy()
    got = ops.linear_q(xf, p).cpu().numpy()
    want = IO.linear_q(xo, s_x, zp_x, L["w_int8"].numpy(), L["w_scales"].numpy(), L["bias"].numpy(), L["out_scale"],
                       L["out_zp"], relu=R.regime_relu(regime))
    what = f"{name} b={b} {regime}"
    _assert_not_vacuous(want, regime, what)
    if regime == "range_mixed":
        _assert_range_test_mixed(xo, zp_x, L["w_int8"].numpy(), False, what)
    _assert_equal(got, want, what)
    _assert_equal(ops.linear_q(xf, p, impl="simt").cpu().numpy(), want, what + " simt")


# ---------------------------------------------------------------------------------------------- kernel selection check
def _profile_cases():
    """Demangled kernel names, in launch order, of one profiler session over every case of this file (zero inputs:
    kernel selection does not depend on the data)."""
    from torch.profiler import ProfilerActivity, profile
    from convnet_quantization_b200 import _lib
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    lib = _lib.load()
    zeros = {}

    def zeros_like(shape):  # allocated outside the trace, shared by the cases of one shape
        if shape not in zeros:
            zeros[shape] = torch.zeros(shape, dtype=torch.uint8, device="cuda")
        return zeros[shape]

    runs = []
    for cases, mirrors in ((CONV_CASES, True), (MIRRORLESS_CASES, False)):
        for layer, pool, size, regime in cases:
            cin, cout, img = R._geom(layer)
            b = R._conv_batch(layer, size, sms)
            _, c = _packed(layer, regime, mirrors)
            x = zeros_like((b, img, img, cin))
            runs.append(lambda x=x, b=b, c=c, pool=pool, img=img, cout=cout: _run_conv(x, c, b, pool, img, cout))
    for name, size, regime in LINEAR_CASES:
        b = _lin_batch(name, size, sms)
        p, _ = _packed(name, regime)
        x = zeros_like((b, p.k))
        y = torch.empty((b, p.n), dtype=torch.uint8, device="cuda")
        runs.append(lambda x=x, b=b, p=p, y=y: _lib.check(lib.b200q_linear_tc(
            x.data_ptr(), y.data_ptr(), b, p.ptr(), torch.cuda.current_stream().cuda_stream), "linear_tc"))
    for run in runs:  # first launches (module loading, smem attributes) outside the trace
        run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for run in runs:
            run()
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                      and not e.name.startswith(("Memcpy", "Memset"))), key=lambda e: e.time_range.start)
    return sms, [R._plain_kernel_name(e.name) for e in kernels]


@gpu
def test_regime_cases_run_the_kernels_they_claim():
    """One profiler pass over every case of this file: each launches exactly one kernel, the instantiation its batch
    size and flags are meant to select, ``CHECK`` argument included (halo, halo2 and pair kernels: ``CHECK = false``
    exactly for ``BOUNDED | ACC22``; ``igemm_tc_kernel``: the same for ``COUT`` 64, true otherwise).  The trace is taken
    in a child process so that it cannot touch the CUPTI state of traces other test files take."""
    code = ("import json, tests.test_gpu_requant_regimes as T; "
            "print('NAMES ' + json.dumps(T._profile_cases()))")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-3000:]
    sms, names = json.loads(next(l for l in r.stdout.splitlines() if l.startswith("NAMES "))[6:])
    want = expected_kernels(sms)
    assert len(names) == len(want), f"{len(want)} cases, {len(names)} kernels"
    wrong = [(label, kernel, name) for (label, kernel), name in zip(want, names) if f"::{kernel}(" not in name]
    assert not wrong, "cases that did not run the kernel they claim:\n" + "\n".join(map(str, wrong))


# ---------------------------------------------------------------------------------------------- whole net
NET_SIZES = ("1", "2", "3", "32", "33", "sms_1", "3sms_1", "fc1_wide")
NET_FLAGS = {  # per net: layer -> (flag bits checked, their value)
    "acc22": {n: (R.FAST, R.FAST) for n in R.NET_LAYERS},
    "fires": {**{n: (R.FAST, R.FAST) for n in ("conv2", "conv3")},
              **{n: (R.FAST, R.RQ_BOUNDED) for n in ("conv4", "conv5", "conv6", "fc1")}},
    "unbounded": {n: (R.RQ_BOUNDED, 0) for n in R.NET_LAYERS},
}


def _net_batch(size, sms):
    return {"sms_1": sms + 1, "3sms_1": 3 * sms + 1, "fc1_wide": R._fc1_batch("wide_first", sms)}.get(size) or int(size)


@pytest.fixture(scope="module")
def regime_nets(qparams):
    from tests.conftest import qparams_to_numpy
    nets = {}
    for kind in R.NETS:
        qp = R.regime_net(qparams, kind)
        flags = R.net_flags(qp)
        assert all(flags[n] & m == v for n, (m, v) in NET_FLAGS[kind].items()), (kind, flags)
        nets[kind] = (qp, qparams_to_numpy(qp))
    return nets


def _oracle(qp_np, x):
    from oracle import int_ops as IO
    taps = {}
    logits = IO.static_forward(x.numpy(), qp_np, taps)
    return logits, taps


@gpu
@pytest.mark.parametrize("size", NET_SIZES)
@pytest.mark.parametrize("kind", R.NETS)
def test_regime_net(qparams, regime_nets, sms, kind, size):
    """``StaticEngine`` on a whole net in one regime: production-route logits (pools fused) and parity-route taps equal
    ``int_ops.static_forward`` bit for bit on a sample of the batch, with the same number of launches as the calibrated
    net at that batch."""
    from convnet_quantization_b200 import _lib
    from convnet_quantization_b200.engine import StaticEngine
    qp, qp_np = regime_nets[kind]
    b = _net_batch(size, sms)
    x = R.net_input(kind, b, seed=b)
    idx = R.net_sample(b, sms, seed=b)
    want, want_taps = _oracle(qp_np, x[torch.from_numpy(idx)])
    lib = _lib.load()
    eng, ref = StaticEngine(qp, "cuda"), StaticEngine(qparams, "cuda")
    xd = x.cuda()
    counts = []
    for e in (eng, ref):
        e.forward(xd, graph=False)  # first launches outside the count
        n0 = lib.b200q_launch_count()
        logits = e.forward(xd, graph=False)
        counts.append(lib.b200q_launch_count() - n0)
        if e is eng:
            got = logits
    assert counts[0] == counts[1], f"{kind} b={b}: {counts[0]} launches, the calibrated net {counts[1]}"
    what = f"{kind} net b={b}"
    _assert_equal(got[torch.from_numpy(idx).cuda()].cpu().numpy(), want, what + " logits")
    _, taps = eng.forward(xd, taps=True)
    for k, t in taps.items():
        a = t[torch.from_numpy(idx).cuda()].cpu().numpy()
        if k == "quant":
            a = a[..., :3]
        _assert_equal(a, want_taps[k], f"{what} tap {k}")
        if len(idx) >= 32:
            assert len(np.unique(want_taps[k])) >= 16, f"{what}: tap {k} has {len(np.unique(want_taps[k]))} values"


@gpu
@pytest.mark.parametrize("pdl", [False, True])
@pytest.mark.parametrize("b", [1, 32])
@pytest.mark.parametrize("kind", R.NETS)
def test_regime_net_graph(regime_nets, kind, b, pdl):
    """The whole-network executor (CUDA graph, with and without programmatic dependent launch) on each regime net:
    logits equal the integer oracle and the eager forward, across replays with different inputs."""
    from convnet_quantization_b200.engine import StaticEngine
    qp, qp_np = regime_nets[kind]
    eng = StaticEngine(qp, "cuda", pdl=pdl)
    buf = torch.empty(b, 3, 32, 32, device="cuda")
    for rep in range(3):
        x = R.net_input(kind, b, seed=100 * b + rep)
        buf.copy_(x)
        y = eng.forward(buf, graph=True)
        _assert_equal(y.cpu().numpy(), _oracle(qp_np, x)[0], f"{kind} net b={b} pdl={pdl} rep={rep}")
        assert torch.equal(eng.forward(buf, graph=False), y)


# ---------------------------------------------------------------------------------------------- single-CTA conv2 + pool
SINGLE_CTA_SIZES = ("band_first", "band_odd", "many")


def single_cta_kernels():
    """conv2 + pool on one CTA per band (``conv_halo_kernel<32,64,64,1,true,...>``): the product's fall-back where the
    device has no room for a CTA pair, selected here through the development library's ``B200Q_NO_CTA2=1``."""
    return [(f"conv2 pool=True {size} {regime} single CTA",
             f"conv_halo_kernel<32,64,64,1,true,{R._check_arg(R.REGIMES[regime][0])},8>")
            for regime in R.REGIMES for size in SINGLE_CTA_SIZES]


def _single_cta_cases():
    """Run in a child process with the development library and ``B200Q_NO_CTA2=1``: each case against the oracle,
    then one profiler pass; returns (mismatch messages, kernel names)."""
    from torch.profiler import ProfilerActivity, profile
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    errors, runs = [], []
    for regime in R.REGIMES:
        for size in SINGLE_CTA_SIZES:
            try:
                _check_conv("conv2", True, size, regime, sms, mirrors=True)
            except AssertionError as e:
                errors.append(str(e)[:300])
            _, c = _packed("conv2", regime)
            b = R._conv_batch("conv2", size, sms)
            x = torch.zeros((b, 32, 32, 64), dtype=torch.uint8, device="cuda")
            runs.append(lambda x=x, b=b, c=c: _run_conv(x, c, b, True, 32, 64))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for run in runs:
            run()
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                      and not e.name.startswith(("Memcpy", "Memset"))), key=lambda e: e.time_range.start)
    return errors, [R._plain_kernel_name(e.name) for e in kernels]


@gpu
def test_regime_conv2_pool_single_cta():
    """conv2 + fused pool on the single-CTA halo kernel (what ``b200q_conv3x3_tc`` runs where no CTA pair fits) in
    every regime, at the first band batch, an odd one and one where every CTA walks several bands: bit-exact against
    the oracle (the conv2 + pool cases of ``test_regime_conv_layer``, with the one-CTA kernel), and each launches that
    kernel with the ``CHECK`` argument its flags select."""
    from convnet_quantization_b200 import _lib
    env = dict(os.environ, B200Q_LIB=str(_lib.build(dev=True)), B200Q_NO_CTA2="1")
    code = ("import json, tests.test_gpu_requant_regimes as T; "
            "print('RESULT ' + json.dumps(T._single_cta_cases()))")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-3000:]
    errors, names = json.loads(next(l for l in r.stdout.splitlines() if l.startswith("RESULT "))[7:])
    assert not errors, "\n".join(errors)
    want = single_cta_kernels()
    assert len(names) == len(want), f"{len(want)} cases, {len(names)} kernels: {names}"
    wrong = [(label, kernel, name) for (label, kernel), name in zip(want, names) if f"::{kernel}(" not in name]
    assert not wrong, "cases that did not run the kernel they claim:\n" + "\n".join(map(str, wrong))
