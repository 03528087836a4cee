"""The drop-in surface (SURVEY 8b) without a GPU: class names, methods, attributes and the pre-``quantize()`` behaviour of
the model classes mirror the reference's (`models/*.py`, as listed in SURVEY.md 8(b))."""
import inspect

import pytest
import torch

from convnet_quantization_b200 import synth
from convnet_quantization_b200.models.baseline_model import SimpleConvNet
from convnet_quantization_b200.models.custom_quantization_model import (CustomQuantizationModel, CustomQuantizedConv2d,
                                                                         CustomQuantizedLinear, CustomQuantizedSimpleConvNet)
from convnet_quantization_b200.models.dynamic_ptq_model import DynamicPTQModel
from convnet_quantization_b200.models.optimized_custom_quantization import OptimizedCustomQuantization
from convnet_quantization_b200.models.static_ptq_model import StaticPTQModel

SURFACE = {  # SURVEY.md 8(b), "Python surface a replacement must keep"
    DynamicPTQModel: ["load_state_dict", "quantize", "forward", "__call__", "eval", "cpu", "to", "get_model_size"],
    StaticPTQModel: ["quantize", "get_model_size"],
    CustomQuantizationModel: ["load_state_dict", "quantize", "forward"],
    OptimizedCustomQuantization: ["quantize", "get_model_size"],
}


def test_methods_and_attributes():
    for cls, names in SURFACE.items():
        for n in names:
            assert callable(getattr(cls, n, None)), f"{cls.__name__}.{n}"
    d = DynamicPTQModel()
    assert isinstance(d.fp32_model, SimpleConvNet) and d.quantized_model is None
    s = StaticPTQModel()
    assert isinstance(s.fp32_model, SimpleConvNet) and s.quantized_model is None
    assert list(inspect.signature(s.quantize).parameters)[0] == "calibration_data_loader"
    c = CustomQuantizationModel()
    assert isinstance(c.model, SimpleConvNet) and c.quantized_model is None and c.is_custom_quantized is True
    assert list(inspect.signature(OptimizedCustomQuantization.quantize).parameters)[:2] == ["self", "model"]


def test_behaviour_before_quantize_is_the_fp32_net():
    sd = synth.make_state_dict(0)
    x = synth.images_f32(4, seed=2)
    net = SimpleConvNet()
    net.load_state_dict(sd)
    want = net.eval()(x)
    d = DynamicPTQModel()
    d.load_state_dict(sd)
    assert d.eval() is d and d.cpu() is d and d.to("cpu") is d
    with torch.no_grad():
        assert torch.equal(d(x), want) and torch.equal(d.forward(x), want)
    c = CustomQuantizationModel()
    c.load_state_dict(sd)
    with torch.no_grad():
        assert torch.equal(c.eval()(x), want)
        q = c.quantize()  # as written: BN folded, identity stubs - runs on the CPU like the reference
        assert isinstance(q, CustomQuantizedSimpleConvNet) and isinstance(q.conv1, CustomQuantizedConv2d)
        assert isinstance(q.fc1, CustomQuantizedLinear) and q.is_custom_quantized
        torch.testing.assert_close(q(x), want, rtol=1e-4, atol=1e-4)
    with pytest.raises(ValueError):
        StaticPTQModel(mode="nope")
    with pytest.raises(ValueError):
        CustomQuantizationModel(mode="nope")

