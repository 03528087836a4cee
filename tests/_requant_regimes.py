"""Test helpers shared by the per-layer kernel tests: which kernel ``b200q_conv3x3_tc`` / ``b200q_linear_tc`` select for a
batch (``csrc/igemm_tc.cu``, ``csrc/conv_halo.cu``, ``csrc/conv_halo2.cu``, ``csrc/conv_pair.cu``, ``csrc/conv_small.cu``),
the image sample compared with the oracle, and layers built directly in each requantisation regime that
``packing.requant_flags`` can select.

Every tensor-core epilogue runs one of three arithmetic forms, chosen at pack time by the layer's flags
(``include/b200q.h``):

* ``BOUNDED | ACC22``: conversion-free form, no range test (the halo / pair kernels, and ``igemm_tc_kernel`` with
  ``COUT`` 64, are launched with ``CHECK = false``);
* ``BOUNDED`` only: conversion-free form; a warp with any accumulator outside +-2^22 redoes its chunk in the exact
  I2F/F2I form;
* not ``BOUNDED``: exact form only.

``regime_layer`` builds each regime from seeded integers (no calibration, so nothing depends on the host's float
arithmetic); ``regime_input`` builds inputs that make the regime do what it is meant to do."""
from __future__ import annotations

import numpy as np
import torch

WHOLE = 160   # up to this many images every output is compared with the oracle; above it, a sample
SAMPLE = 48
B200_SMS = 148  # SM count the case tables are enumerated for when no device is present (coverage test)

RQ_BOUNDED, RQ_ACC22 = 1, 2  # include/b200q.h (the CPU tests must not need the library)
FAST = RQ_BOUNDED | RQ_ACC22

# regime -> (flags it must get, ReLU fused, input zero-point, output zero-point)
REGIMES = {
    "acc22": (FAST, True, 131, 100),
    "range_mixed": (RQ_BOUNDED, False, 3, 128),
    "mult": (0, False, 77, 0),
    "mult_many": (0, False, 0, 255),
    "bdiv_edge": (RQ_BOUNDED, True, 128, 60),
    "bdiv_over": (0, True, 128, 60),
    "corr": (0, False, 255, 128),
}
S_X, S_OUT = 2.0 ** -6, 2.0 ** -3   # powers of two: mult and bdiv of chosen channels come out exact
LINEARS = {"fc1": (4096, 512), "lin512": (512, 64)}  # (k, n)


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
        "160": 160,
        "nbi3_below": 3 * sms - 1, "nbi3_above": 3 * sms + 1,
        "many": 9 * sms + 5,                 # every persistent CTA (pair) walks three or more bands
    }[size]


def _check_arg(flags, cout=None):
    """Demangled ``CHECK`` template argument the launcher picks: false exactly for ``BOUNDED | ACC22`` layers (for
    ``igemm_tc_kernel`` only when ``COUT`` is 64); ``flags=None`` matches either."""
    if flags is None:
        return "(true|false)"
    fast = (flags & FAST) == FAST and cout in (None, 64)
    return "false" if fast else "true"


def _conv_plan(layer, pool, b, sms, flags=None, mirrors=True):
    """(kernel-name pattern, images per band, bands in flight at once) that ``b200q_conv3x3_tc`` selects.  Patterns
    are matched against demangled names with the spaces and ``(int)`` / ``(bool)`` casts removed.  With ``flags`` the
    pattern names the ``CHECK`` argument too; ``mirrors=False``: the layer has no host copies of its constants, so the
    band-resident kernels are not eligible and the large-batch shifted-TMA kernel runs."""
    cin, cout, img = _geom(layer)
    p = "true" if pool else "false"
    if b <= 2:
        return rf"conv3x3_tiny_kernel<{img},{cin},{cout},{p}>", 1, b
    if b <= _small_last(layer, sms):
        return rf"igemm_tc_kernel<{img},{cin},{cout},false,{p},{_check_arg(flags, cout)},64>", 1, b
    if not mirrors or (layer == "conv3" and pool):
        # weights resident in shared memory for the 32 x 32 and 16 x 16 layers, streamed for the 8 x 8 ones
        per_round = {32: sms // 8, 16: sms // 2, 8: 2 * sms}[img]
        return rf"igemm_tc_kernel<{img},{cin},{cout},{'true' if img > 8 else 'false'},{p},{_check_arg(flags, cout)},0>", \
            1, per_round
    c = _check_arg(flags)
    if layer == "conv2" and pool:
        return rf"conv_halo2_kernel<{c},8>", 2, sms // 2
    if layer == "conv2":
        return rf"conv_halo_kernel<32,64,64,1,false,{c},8>", 1, sms
    if layer == "conv3":
        nbi = 1 if b < 3 * sms else 3
        return rf"conv_halo_kernel<16,64,128,{nbi},false,{c},8>", nbi, sms
    if layer == "conv4":
        return rf"conv_halo_kernel<16,128,128,1,{p},{c},8>", 1, sms
    return rf"conv_pair_kernel<{cin},{p},{c}>", 4, sms // 2


def _fc1_batch(size, sms):
    narrow_last = 128 * (sms // 8)  # eight 64-column CTA tiles per 128 rows while they fit on the SMs
    return {"1": 1, "7": 7, "narrow_last": narrow_last, "wide_first": narrow_last + 1}[size]


def _fc1_kernel(b, sms):
    return rf"igemm_tc_kernel<0,4096,512,false,false,true,{64 if b <= 128 * (sms // 8) else 0}>"


def _linear_kernel(name, b, sms, flags):
    if name == "fc1":
        return _fc1_kernel(b, sms)
    return rf"igemm_tc_kernel<0,512,64,false,false,{_check_arg(flags, 64)},0>"


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


def _plain_kernel_name(name):
    return (name.replace(" ", "").replace("(int)", "").replace("(bool)0", "false").replace("(bool)1", "true"))


# ---------------------------------------------------------------------------------------------- regimes
def _dims(name):
    """(output channels, K, weight shape) of a conv layer or of a linear one (``LINEARS``)."""
    if name in LINEARS:
        k, n = LINEARS[name]
        return n, k, (n, k)
    cin, cout, _ = _geom(name)
    return cout, 9 * cin, (cout, cin, 3, 3)


def _input_range(regime):
    """Byte range of the bulk of a regime's inputs: small bytes where the range test must fire only on the saturated
    images; for ``corr`` bytes that keep the raw ``sum x*w`` inside +-2^22 (no fall-back) while ``|acc|`` stays below
    2^21 (``bdiv`` can centre it)."""
    return {"range_mixed": (0, 7), "corr": (140, 160)}.get(regime, (0, 255))


def _weights(regime, name, g):
    cout, k, shape = _dims(name)
    w = torch.zeros((cout, k), dtype=torch.int64)
    sign = torch.randint(0, 2, (cout, 1), generator=g) * 2 - 1
    if regime == "acc22":
        m = (2 ** 22 - 1) // (255 * k)  # 255 * sum|w| < 2^22 for every channel and every input
        w = torch.randint(-m, m + 1, (cout, k), generator=g)
    elif regime == "range_mixed":
        # single-signed channels: |sum x*w| reaches 255 * 127 * K; one channel in four with small weights stays in range
        big = torch.randint(100, 128, (cout, k), generator=g)
        small = torch.randint(8, 17, (cout, k), generator=g)
        w = torch.where((torch.arange(cout) % 4 == 3).view(-1, 1), small, big) * sign
    elif regime == "corr":
        # even channels: positive weights summing to 16 600..18 000, so zp_x * sum w >= 2^22 with zp_x = 255 (and
        # MAGIC_F + corr is not exact in fp32 for odd sums, which only the exact form gets right)
        w = torch.randint(-20, 21, (cout, k), generator=g)
        for c in range(0, cout, 2):
            s = int(torch.randint(16600, 18001, (1,), generator=g))
            row = torch.full((k,), s // k, dtype=torch.int64)
            row[torch.randperm(k, generator=g)[: s % k]] += 1
            w[c] = row
    else:
        w = torch.randint(-127, 128, (cout, k), generator=g)
    if regime == "mult_many":
        # channels 1 mod 4 (mult 4): negative weights summing to -14 000 .. -16 300, so a saturated image drives the
        # accumulator to -3.6M .. -4.16M, inside the range test, and t = 4 * acc below -1.5 * 2^23, where the
        # conversion-free rounding (t + 1.5 * 2^23 as an integer) wraps around
        for c in range(1, cout, 4):
            s = int(torch.randint(14000, 16301, (1,), generator=g))
            row = torch.full((k,), s // k, dtype=torch.int64)
            row[torch.randperm(k, generator=g)[: s % k]] += 1
            w[c] = -row
    if regime in ("mult", "mult_many"):
        # the channels that get mult > 0.5 have three non-zero weights, so that their outputs do not all clamp
        sparse = [0] if regime == "mult" else list(range(0, cout, 2))
        for c in sparse:
            row = torch.zeros(k, dtype=torch.int64)
            pos = torch.randperm(k, generator=g)[:3]
            row[pos] = torch.randint(1, 4, (3,), generator=g) * (torch.randint(0, 2, (3,), generator=g) * 2 - 1)
            w[c] = row
    return w.to(torch.int8).reshape(shape)


def _f32(v):
    return np.float32(v)


def regime_layer(name, regime, seed=0):
    """``(layer, s_x, zp_x)``: a layer dict in the ``ptq.calibrate_static`` form (``w_int8``, ``w_scales`` float64,
    ``bias`` float32, ``out_scale``, ``out_zp``) for conv ``name`` or linear ``fc1`` / ``lin512`` in ``regime``
    (``REGIMES``), and the input scale and zero-point to pack it with.

    Typical channels get ``bdiv`` that centres the regime's bulk input on output 128 and ``mult`` that spreads the
    central 98 % of it over about 200 output steps.  Then per regime: ``range_mixed`` channels 2 mod 4 at ``mult`` =
    2^-p, ``bdiv`` = -2^21 (unclamped outputs for accumulators beyond 2^22); ``mult`` one channel at 0.51; ``mult_many``
    every even channel in (0.5, 4] and channels 1 mod 4 at 4 with heavy negative weights; ``bdiv_edge`` channels 0 mod
    8 at ``mult`` = 2^-15 and ``bdiv`` = +-2^21 exactly; ``bdiv_over`` the same with channel 0 one float step above
    2^21, and channel 1 at ``bdiv`` = -2^25.  The last two (and ``corr``) give bytes that only the exact form gets
    right, so a kernel that takes the conversion-free form without ``BOUNDED`` fails."""
    from oracle import int_ops as IO
    flags, relu, zp_x, zp_out = REGIMES[regime]
    g = torch.Generator().manual_seed(1000 * seed + 17 * list(REGIMES).index(regime) + sum(map(ord, name)))
    w = _weights(regime, name, g)
    cout, k, _ = _dims(name)
    # per-channel centre and spread of the accumulator on a few images of the regime's bulk input
    lo, hi = _input_range(regime)
    rng = np.random.default_rng(seed + 7)
    wn = w.numpy()
    if name in LINEARS:
        acc = IO.linear_acc(rng.integers(lo, hi + 1, (64, k)).astype(np.uint8), zp_x, wn)
    else:
        cin, _, img = _geom(name)
        acc = IO.conv3x3_acc(rng.integers(lo, hi + 1, (2, img, img, cin)).astype(np.uint8), zp_x, wn)
        acc = acc.reshape(-1, cout)
    q01, q50, q99 = np.percentile(acc.astype(np.float64), [1, 50, 99], axis=0)
    mult = np.minimum(200.0 / np.maximum(q99 - q01, 1.0), 0.45)
    bdiv = np.clip(-q50 + (128 - zp_out) / mult, -0.95 * 2 ** 21, 0.95 * 2 ** 21)
    if regime == "mult":
        mult[0] = 0.51
    elif regime == "mult_many":
        mult[0::2] = np.linspace(0.5, 4.0, cout // 2 + 1)[1:]
        mult[1::4] = 4.0
        bdiv[1::4] = 0.0
    elif regime == "range_mixed":
        # channels 2 mod 4 map accumulators of 2^21 .. ~2^21 + 255 * 2^p onto the output range (mult = 2^-p, bdiv =
        # -2^21): the saturated border pixels, beyond 2^22, give unclamped outputs that only the exact form gets right
        p = int(np.ceil(np.log2(252 * 113 * k / 100)))
        mult[2::4] = 2.0 ** -p
        bdiv[2::4] = -2.0 ** 21
    elif regime in ("bdiv_edge", "bdiv_over"):
        mult[0::8] = 2.0 ** -15
        bdiv[0::8] = np.where(np.arange(0, cout, 8) % 16 == 0, 2.0 ** 21, -2.0 ** 21)
        if regime == "bdiv_over":
            # t = (acc - 2^25) * 0.45 lies below -1.5 * 2^23 for every in-range accumulator: the exact form clamps it,
            # the conversion-free rounding wraps around
            mult[1], bdiv[1] = 0.45, -2.0 ** 25
    ws = mult * S_OUT / S_X
    atw = (_f32(S_X) * ws.astype(np.float32)).astype(np.float32)
    bias = (bdiv * atw.astype(np.float64)).astype(np.float32)
    if regime == "bdiv_over":
        bias[0] = np.nextafter(bias[0], np.float32(np.inf))
    layer = {"w_int8": w, "w_scales": torch.from_numpy(ws.astype(np.float64)), "bias": torch.from_numpy(bias),
             "out_scale": S_OUT, "out_zp": zp_out}
    return layer, S_X, zp_x


def regime_relu(regime):
    return REGIMES[regime][1]


def regime_flags(name, regime, seed=0):
    """``packing.requant_flags`` of the layer as ``PackedConv`` / ``PackedLinear`` pack it."""
    from convnet_quantization_b200 import packing
    layer, s_x, zp_x = regime_layer(name, regime, seed)
    mult, bdiv = packing.requant_constants(s_x, layer["w_scales"], layer["bias"], layer["out_scale"])
    return packing.requant_flags(mult, bdiv, layer["w_int8"], zp_x)


SATURATE_EVERY = 7  # range_mixed: every 7th image saturated (odd, so that both accumulator slots of a CTA see one)


def regime_input(regime, shape, seed, device="cpu"):
    """uint8 input of ``shape`` (NHWC images, or ``[b, k]`` rows): seeded bytes in the regime's bulk range, image 0
    saturated and the last image's top half zero; a single image gets two saturated top rows and a zero bottom half.
    A single row of a linear layer gets its first eighth saturated and its last eighth zero.  ``range_mixed`` also
    saturates every ``SATURATE_EVERY``-th image and only the top quarter of image 1 (a single image: its top rows, a
    single row: its first half, and nothing zeroed), so that the run-time range test fires in some warps of a launch and
    not in others."""
    lo, hi = _input_range(regime)
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randint(lo, hi + 1, shape, generator=g, device=device, dtype=torch.int32).to(torch.uint8)
    rows = shape[1]
    b = shape[0]
    mixed = regime == "range_mixed"
    if b == 1 and len(shape) == 2:
        x[0, : rows // 2 if mixed else rows // 8] = 255
        if not mixed:
            x[0, -(rows // 8):] = 0
    elif b == 1:
        x[0, :2] = 255
        if not mixed:  # zero bytes are far from range_mixed's bulk: its only image would clamp
            x[0, rows // 2:] = 0
    else:
        x[0] = 255
        x[-1, : rows // 2] = 0
    if mixed and b > 1:
        x[SATURATE_EVERY::SATURATE_EVERY] = 255
        x[1, : rows // 4] = 255
    return x.contiguous()


def range_tested(x_u8, zp_x, w_int8, band_kernel):
    """int64 quantity the conversion-free epilogue range-tests, per output element: the raw ``sum x*w`` over all nine
    taps with the pads holding ``zp_x`` in the halo / halo2 / pair kernels (``band_kernel``), the zero-point-corrected
    accumulator in ``igemm_tc_kernel`` (its TMA zero-fills the pads and the correction comes from the border-class
    table).  The test passes for values in [-2^22, 2^22)."""
    from oracle import int_ops as IO
    w = np.asarray(w_int8)
    if w.ndim == 2:
        acc = IO.linear_acc(x_u8, zp_x, w)
        return acc + zp_x * w.astype(np.int64).sum(1) if band_kernel else acc
    acc = IO.conv3x3_acc(x_u8, zp_x, w)
    return acc + zp_x * w.astype(np.int64).reshape(w.shape[0], -1).sum(1) if band_kernel else acc


def out_of_range(q):
    return (q >= 2 ** 22) | (q < -2 ** 22)


# ---------------------------------------------------------------------------------------------- whole net
NET_LAYERS = ("conv1", "conv2", "conv3", "conv4", "conv5", "conv6", "fc1", "fc2")
NETS = ("acc22", "fires", "unbounded")


def regime_net(qp, kind):
    """The static-PTQ parameters ``qp`` (``ptq.calibrate_static`` form) turned into a whole net in one regime:
    ``acc22`` every layer's integer weights divided (toward zero) by the smallest d >= 4 that bounds its accumulators
    below 2^22, ``w_scales`` times d; ``fires`` conv4-conv6's integer weights x4 clamped to +-127, ``w_scales`` / 4
    (they keep ``BOUNDED`` but lose ``ACC22``, so the net runs ``CHECK = false`` kernels for conv2 / conv3 and
    range-tested ones from conv4 on; scaling every layer leaves fc1's output fewer than 16 distinct values);
    ``unbounded`` channel 0 of every layer at ``mult`` = 0.51 (same ``bdiv``)."""
    import copy
    from convnet_quantization_b200 import packing
    qp = copy.deepcopy(qp)
    s = float(qp["in_scale"])
    for name in NET_LAYERS:
        L = qp[name]
        w = L["w_int8"].to(torch.int64)
        if kind == "acc22":
            d = 4
            while packing.acc_bound(torch.div(w, d, rounding_mode="trunc"), 255) >= 2 ** 22:
                d += 1
            L["w_int8"] = torch.div(w, d, rounding_mode="trunc").to(torch.int8)
            L["w_scales"] = L["w_scales"] * d
        elif kind == "fires" and name in ("conv4", "conv5", "conv6"):
            L["w_int8"] = (w * 4).clamp(-127, 127).to(torch.int8)
            L["w_scales"] = L["w_scales"] / 4
        elif kind == "unbounded":
            ws = L["w_scales"].clone()
            new = 0.51 * float(L["out_scale"]) / s
            L["bias"] = L["bias"].clone()
            L["bias"][0] = float(L["bias"][0]) * new / float(ws[0])
            ws[0] = new
            L["w_scales"] = ws
        s = float(L["out_scale"])
    return qp


def net_flags(qp):
    """``packing.requant_flags`` of every layer of a static net, as ``PackedStaticNet`` packs it."""
    from convnet_quantization_b200 import packing
    out, s, zp = {}, float(qp["in_scale"]), int(qp["in_zp"])
    for name in NET_LAYERS:
        L = qp[name]
        mult, bdiv = packing.requant_constants(s, L["w_scales"], L["bias"], L["out_scale"])
        out[name] = packing.requant_flags(mult, bdiv, L["w_int8"], zp)
        s, zp = float(L["out_scale"]), int(L["out_zp"])
    return out


def net_input(kind, b, seed):
    """fp32 NCHW images: synthetic images (x3 for ``fires``), image 0 saturated high."""
    from convnet_quantization_b200 import synth
    x = synth.images_f32(b, seed=seed) * (3.0 if kind == "fires" else 1.0)
    x[0] = 1.0e3
    return x


def net_sample(b, sms, seed):
    """Every image up to ``SAMPLE``; above, the first two, the last, both sides of the SM-count boundaries and seeded
    random images, ``SAMPLE`` in all."""
    if b <= SAMPLE:
        return np.arange(b)
    idx = {0, 1, b - 1} | {i for lo in (sms, 2 * sms, 3 * sms) for i in (lo - 1, lo) if lo < b}
    rest = np.setdiff1d(np.arange(b), np.fromiter(idx, dtype=np.int64))
    fill = np.random.default_rng(seed).choice(rest, size=SAMPLE - len(idx), replace=False)
    return np.sort(np.concatenate([np.fromiter(idx, dtype=np.int64), fill]))
