"""CPU checks of the requantisation regimes the GPU sweep (``tests/test_gpu_requant_regimes.py``) runs: each regime gets
the pack-time flags it is meant to get, for the reason it is meant to get them; the integer oracle equals the live
fbgemm ops on each regime's constants; and every kernel instantiation compiled into the product library is named by at
least one GPU case, or listed here with the reason no product path reaches it."""
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from tests import _requant_regimes as R

LAYERS = ("conv2", "conv3", "conv4", "conv5", "conv6", "fc1", "lin512")


def _conditions(name, regime):
    """Which of the four ``B200Q_RQ_BOUNDED`` conditions the layer meets, and whether it meets ``ACC22``."""
    from convnet_quantization_b200 import packing
    layer, s_x, zp_x = R.regime_layer(name, regime)
    mult, bdiv = packing.requant_constants(s_x, layer["w_scales"], layer["bias"], layer["out_scale"])
    w = layer["w_int8"].to(torch.int64).reshape(layer["w_int8"].shape[0], -1)
    return {"mult": bool(((mult >= 0) & (mult <= 0.5)).all()), "bdiv": bool((bdiv.abs() <= 2.0 ** 21).all()),
            "corr": bool(((zp_x * w.sum(1)).abs() < 2 ** 22).all()),
            "acc22": packing.acc_bound(layer["w_int8"], zp_x) < 2 ** 22}, mult, bdiv


# the one bound each unbounded regime breaks
BREAKS = {"mult": "mult", "mult_many": "mult", "bdiv_over": "bdiv", "corr": "corr"}


@pytest.mark.parametrize("regime", list(R.REGIMES))
@pytest.mark.parametrize("name", LAYERS)
def test_regime_flags(name, regime):
    """``packing.requant_flags`` gives each regime its flags on every layer it is used on, and an unbounded regime
    breaks exactly the bound it is named for."""
    flags = R.regime_flags(name, regime)
    assert flags == R.REGIMES[regime][0], (name, regime, flags)
    cond, mult, bdiv = _conditions(name, regime)
    broken = {k for k in ("mult", "bdiv", "corr") if not cond[k]}
    assert broken == ({BREAKS[regime]} if regime in BREAKS else set()), (name, regime, broken)
    assert cond["acc22"] == (regime == "acc22"), (name, regime)
    if regime == "mult":
        assert mult[0].item() == np.float32(0.51) and bool((mult[1:] <= 0.5).all())
    if regime == "mult_many":
        assert bool((mult[0::2] > 0.5).all() & (mult[0::2] <= 4.0).all())
    if regime in ("bdiv_edge", "bdiv_over"):
        edge = bdiv[0::8].abs()
        exact = edge[1:] if regime == "bdiv_over" else edge
        assert bool((exact == 2.0 ** 21).all()), exact
        assert (bdiv[0].item() > 2.0 ** 21) == (regime == "bdiv_over")
        assert bool((bdiv[0::16] > 0).all()) and bool((bdiv[8::16] < 0).all())


def test_regimes_span_the_output_clamps():
    zps = {zp for _, _, _, zp in R.REGIMES.values()}
    assert {0, 255} <= zps
    assert sum(not relu for _, relu, _, _ in R.REGIMES.values()) >= 2


def _torch_qparams(layer, s_x, zp_x):
    from oracle import int_ops as IO
    w = layer["w_int8"]
    qw = torch._make_per_channel_quantized_tensor(w, layer["w_scales"].double(), torch.zeros(w.shape[0], dtype=torch.int64), 0)
    mult, bdiv = IO.requant_params(s_x, layer["w_scales"].numpy(), layer["bias"].numpy(), layer["out_scale"])
    return qw, mult, bdiv


@pytest.mark.parametrize("regime", list(R.REGIMES))
@pytest.mark.parametrize("name", ["fc1", "conv6"])
def test_oracle_pinned_on_regime_constants(name, regime):
    """``int_ops.linear_q`` / ``int_ops.conv2d_q`` == live ``quantized::linear`` / ``quantized::conv2d`` (and their
    ``_relu`` forms) on each regime's constants: ``mult`` > 0.5, ``|bdiv|`` at and above 2^21, input zero-point 255,
    accumulators beyond 2^24 (where ``f32(acc)`` rounds).  Inputs stay in 0..127, the range ``reduce_range``
    calibration gives, so fbgemm's 16-bit pair sums cannot saturate."""
    from oracle import int_ops as IO
    torch.backends.quantized.engine = "fbgemm"
    layer, s_x, zp_x = R.regime_layer(name, regime)
    qw, mult, bdiv = _torch_qparams(layer, s_x, zp_x)
    g = torch.Generator().manual_seed(5)
    w = layer["w_int8"].numpy()
    hi = 7 if regime == "range_mixed" else 127  # range_mixed's constants are set for small bytes
    if name == "fc1":
        x = torch.randint(0, hi + 1, (48, 4096), generator=g, dtype=torch.uint8)
        x[0] = 127
        x[1, :2048] = 127
        x[1, 2048:] = 0
        acc = IO.linear_acc(x.numpy(), zp_x, w)
    else:
        x = torch.randint(0, hi + 1, (3, 8, 8, 256), generator=g, dtype=torch.uint8)
        x[0] = 127
        x[1, :4] = 0
        acc = IO.conv3x3_acc(x.numpy(), zp_x, w)
    assert np.abs((acc.astype(np.float64) + bdiv) * mult).max() < 2.0 ** 31
    if regime == "range_mixed":
        assert np.abs(acc).max() > 2 ** 24  # f32(acc) rounds
    qx_dims = x if name == "fc1" else x.permute(0, 3, 1, 2).contiguous()
    qx = torch._make_per_tensor_quantized_tensor(qx_dims, s_x, zp_x)
    for relu in (False, True):
        if name == "fc1":
            packed = torch.ops.quantized.linear_prepack(qw, layer["bias"])
            op = torch.ops.quantized.linear_relu if relu else torch.ops.quantized.linear
            want = op(qx, packed, layer["out_scale"], layer["out_zp"]).int_repr().numpy()
            got = IO.linear_q(x.numpy(), s_x, zp_x, w, layer["w_scales"].numpy(), layer["bias"].numpy(),
                              layer["out_scale"], layer["out_zp"], relu=relu)
        else:
            packed = torch.ops.quantized.conv2d_prepack(qw, layer["bias"], [1, 1], [1, 1], [1, 1], 1)
            op = torch.ops.quantized.conv2d_relu if relu else torch.ops.quantized.conv2d
            want = op(qx, packed, layer["out_scale"], layer["out_zp"]).int_repr().numpy().transpose(0, 2, 3, 1)
            got = IO.conv2d_q(x.numpy(), s_x, zp_x, w, layer["w_scales"].numpy(), layer["bias"].numpy(),
                              layer["out_scale"], layer["out_zp"], relu=relu)
        bad = got != want
        assert not bad.any(), f"{name} {regime} relu={relu}: {int(bad.sum())} / {bad.size} differ"
        if not (relu and layer["out_zp"] == 255):  # there ReLU clamps every output to 255
            assert len(np.unique(want)) >= 16, (name, regime, relu, np.unique(want))


# ---------------------------------------------------------------------------------------------- coverage
KERNELS = ("igemm_tc_kernel", "conv_halo_kernel", "conv_halo2_kernel", "conv_pair_kernel", "conv3x3_tiny_kernel")

# instantiations compiled into the product library that no product path selects
UNREACHABLE = {
    r"conv_halo2_kernel<(true|false),4>": "four accumulator slots: only the development switch B200Q_H2_SLOTS=4 selects it",
    r"igemm_tc_kernel<(32,64,64|16,64,128|16,128,128),false,(true|false),(true|false),0>":
        "streamed weights for the layers whose weights fit in shared memory: only the development switch "
        "B200Q_TC_STREAM_WEIGHTS=1 selects it",
}


def _library_instantiations():
    from convnet_quantization_b200 import _lib
    tools = [shutil.which(t) or f"/usr/local/cuda/bin/{t}" for t in ("cuobjdump", "cu++filt")]
    lib = _lib.LIB_PATH
    if _lib._stale(lib):
        _lib.build()
    elf = subprocess.run([tools[0], "-elf", str(lib)], capture_output=True, text=True, check=True).stdout
    syms = sorted(set(re.findall(r"\.text\.(_Z[0-9A-Za-z_]+)", elf)))
    names = subprocess.run([tools[1]], input="\n".join(syms), capture_output=True, text=True, check=True).stdout
    out = set()
    for n in names.splitlines():
        plain = R._plain_kernel_name(n.split(">(")[0] + ">")
        m = re.search(r"(%s)<.*>$" % "|".join(KERNELS), plain)
        if m:
            out.add(m.group(0))
    return out


def test_every_compiled_instantiation_has_a_case():
    """Each tensor-core / small-batch conv and linear instantiation in ``libb200q.so`` is the expected kernel of at
    least one GPU case (case tables enumerated for a 148-SM B200), or is listed in ``UNREACHABLE``."""
    from tests import test_gpu_requant_regimes as G
    have = _library_instantiations()
    assert len(have) == 70, sorted(have)
    expected = {name for _, name in G.expected_kernels(R.B200_SMS) + G.single_cta_kernels()}
    unexplained = sorted(k for k in have if k not in expected and not any(re.fullmatch(p, k) for p in UNREACHABLE))
    assert not unexplained, "instantiations no case runs:\n" + "\n".join(unexplained)
    listed = sorted(k for k in have if any(re.fullmatch(p, k) for p in UNREACHABLE))
    assert len(listed) == 10 and not set(listed) & expected, listed
    stale = sorted(e for e in expected if e not in have)
    assert not stale, f"cases expect kernels the library does not contain: {stale}"
