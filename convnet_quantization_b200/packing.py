"""Weight pre-pack for the CUDA engine (host side, once per model).

Turns the static-PTQ parameter dict of ``ptq.calibrate_static`` into device buffers in the layouts the
kernels read, plus the ctypes structs of ``include/b200q.h``:

* conv weights int8 ``[Cout][kh][kw][Cin]`` (K-major, K = 9*Cin; conv1's Cin 3 -> 4 with a zero channel);
* fc1 weight columns permuted from the reference's NCHW flatten order ``c*16+h*4+w``
  (``x.view(-1, 256*4*4)``, ``models/baseline_model.py:78``) to the engine's NHWC order ``(h*4+w)*256+c``;
* per-channel fp32 requant constants ``mult = (s_x*s_w)/s_out`` and ``bdiv = bias/(s_x*s_w)`` computed in
  fp32 on the host exactly as fbgemm does (SURVEY.md Appendix A);
* the zero-point correction table ``corr[9][Cout] = zp_x * sum(w over the taps that are inside the image)``
  for the 3x3 border classes (TMA zero-fills out-of-image taps, but quantized zero is ``zp_x``, not 0).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib

CONV_GEOMETRY = {  # layer -> (cin, cout, img)
    "conv1": (3, 64, 32), "conv2": (64, 64, 32), "conv3": (64, 128, 16),
    "conv4": (128, 128, 16), "conv5": (128, 256, 8), "conv6": (256, 256, 8),
}


def requant_constants(s_x: float, w_scales: torch.Tensor, bias: torch.Tensor, s_out: float):
    """fp32 (mult, bdiv) per output channel; every step rounds to binary32 like the CPU kernels."""
    f32 = torch.float32
    atw = torch.tensor(s_x, dtype=f32) * w_scales.detach().cpu().to(f32)
    mult = atw / torch.tensor(s_out, dtype=f32)
    bdiv = bias.detach().cpu().to(f32) / atw
    return mult.contiguous(), bdiv.contiguous()


def acc_bound(w_int8: torch.Tensor, zp_x: int) -> int:
    """Largest magnitude, over output channels and all uint8 inputs, of the raw accumulator ``sum x*w``, of the
    zero-point-corrected one ``sum (x-zp_x)*w`` and of the correction ``zp_x*sum w`` itself."""
    w = w_int8.detach().cpu().to(torch.int64).reshape(w_int8.shape[0], -1)
    pos, neg = w.clamp(min=0).sum(1), (-w).clamp(min=0).sum(1)
    raw = 255 * torch.maximum(pos, neg)
    acc = torch.maximum((255 - zp_x) * pos + zp_x * neg, zp_x * pos + (255 - zp_x) * neg)
    corr = (zp_x * (pos - neg)).abs()
    return int(torch.stack([raw, acc, corr]).max())


def requant_flags(mult: torch.Tensor, bdiv: torch.Tensor, w_int8: torch.Tensor, zp_x: int) -> int:
    """``B200Q_RQ_BOUNDED`` when every channel satisfies the bounds under which the conversion-free requantisation of
    the tensor-core epilogue is exact, ``B200Q_RQ_ACC22`` when no input can push an accumulator past 2^22
    (``include/b200q.h``)."""
    flags = 0
    w = w_int8.detach().cpu().to(torch.int64).reshape(w_int8.shape[0], -1)
    corr_ok = bool(((zp_x * w.sum(1)).abs() < 2 ** 22).all())
    if corr_ok and bool((mult >= 0).all() and (mult <= 0.5).all() and (bdiv.abs() <= 2.0 ** 21).all()
                        and torch.isfinite(mult).all() and torch.isfinite(bdiv).all()):
        flags |= _lib.RQ_BOUNDED
    if acc_bound(w_int8, zp_x) < 2 ** 22:
        flags |= _lib.RQ_ACC22
    return flags


def conv_border_corr(w_int8: torch.Tensor, zp_x: int) -> torch.Tensor:
    """``corr[3*rc+cc][co]``: rc/cc = 0 first row/col, 1 interior, 2 last row/col."""
    wsum_tap = w_int8.to(torch.int64).sum(dim=1)  # [Cout, 3, 3]
    rows = []
    for rc in range(3):
        for cc in range(3):
            khs = [k for k in range(3) if not (rc == 0 and k == 0) and not (rc == 2 and k == 2)]
            kws = [k for k in range(3) if not (cc == 0 and k == 0) and not (cc == 2 and k == 2)]
            rows.append(wsum_tap[:, khs][:, :, kws].sum(dim=(1, 2)) * int(zp_x))
    return torch.stack(rows).to(torch.int32).contiguous()


def input_lut(in_scale: float, in_zp: int, mean=None, std=None) -> torch.Tensor:
    """uint8 ``[3][256]`` table for the uint8 data path: ``lut[c][v]`` is what the reference pipeline makes of a raw
    pixel value ``v`` in channel ``c`` — ``ToTensor`` (``v/255``), ``Normalize(mean, std)``
    (``utils/dataset_manager.py:41-44``) and the model's ``QuantStub`` (``aten::quantize_per_tensor``) — computed here
    with those very torch CPU ops, so the GPU look-up is bit-identical to quantising the fp32 tensor."""
    from . import synth
    v = torch.arange(256, dtype=torch.uint8).view(256, 1, 1, 1).expand(256, 3, 1, 1).contiguous()
    if mean is None and std is None:
        x = synth.normalize(v)
    else:
        m = torch.tensor(mean, dtype=torch.float32).view(1, 3, 1, 1)
        sd = torch.tensor(std, dtype=torch.float32).view(1, 3, 1, 1)
        x = ((v.to(torch.float32) / 255.0) - m) / sd
    q = torch.quantize_per_tensor(x, float(in_scale), int(in_zp), torch.quint8).int_repr()
    return q.view(256, 3).t().contiguous()  # [3][256]


class PackedConv:
    def __init__(self, name, layer, s_x, zp_x, device, relu=True):
        cin, cout, img = CONV_GEOMETRY[name]
        w = layer["w_int8"].detach().cpu()
        assert tuple(w.shape) == (cout, cin, 3, 3), (name, w.shape)
        cin_p = 4 if cin == 3 else cin
        wk = torch.zeros(cout, 3, 3, cin_p, dtype=torch.int8)
        wk[..., :cin] = w.permute(0, 2, 3, 1)
        mult, bdiv = requant_constants(s_x, layer["w_scales"], layer["bias"], layer["out_scale"])
        self.name, self.cin, self.cout, self.img = name, cin_p, cout, img
        self.zp_x, self.zp_out, self.s_out = int(zp_x), int(layer["out_zp"]), float(layer["out_scale"])
        self.w = wk.contiguous().to(device)
        # host mirrors stay alive with the object: the C struct points at them (kernel-parameter constants)
        self.corr_host = conv_border_corr(w, zp_x)
        self.mult_host, self.bdiv_host = mult, bdiv
        self.corr = self.corr_host.to(device)
        self.mult, self.bdiv = mult.to(device), bdiv.to(device)
        self.c = _lib.Conv3x3(cin_p, cout, img, self.zp_x, self.w.data_ptr(), self.corr.data_ptr(),
                              self.corr_host.data_ptr(),
                              _lib.Requant(self.mult.data_ptr(), self.bdiv.data_ptr(), self.zp_out, int(relu),
                                           requant_flags(mult, bdiv, w, zp_x), 0, self.mult_host.data_ptr(),
                                           self.bdiv_host.data_ptr()))

    def ptr(self):
        return C.byref(self.c)


class PackedLinear:
    def __init__(self, name, layer, s_x, zp_x, device, relu, nhwc_from=None):
        w = layer["w_int8"].detach().cpu()
        n, k = w.shape
        if nhwc_from is not None:  # (c, h, w) of the NCHW-flattened producer
            c, h, wd = nhwc_from
            w = w.view(n, c, h, wd).permute(0, 2, 3, 1).reshape(n, k)
        mult, bdiv = requant_constants(s_x, layer["w_scales"], layer["bias"], layer["out_scale"])
        self.name, self.k, self.n = name, k, n
        self.zp_x, self.zp_out, self.s_out = int(zp_x), int(layer["out_zp"]), float(layer["out_scale"])
        self.w = w.contiguous().to(device)
        self.corr_host = (w.to(torch.int64).sum(dim=1) * int(zp_x)).to(torch.int32).contiguous()
        self.mult_host, self.bdiv_host = mult, bdiv
        self.corr = self.corr_host.to(device)
        self.mult, self.bdiv = mult.to(device), bdiv.to(device)
        self.c = _lib.Linear(k, n, self.zp_x, self.w.data_ptr(), self.corr.data_ptr(), self.corr_host.data_ptr(),
                             _lib.Requant(self.mult.data_ptr(), self.bdiv.data_ptr(), self.zp_out, int(relu),
                                          requant_flags(mult, bdiv, w, zp_x), 0, self.mult_host.data_ptr(),
                                          self.bdiv_host.data_ptr()))

    def ptr(self):
        return C.byref(self.c)


class PackedStaticNet:
    """All device-resident constants of the static-PTQ net + the ``b200q_static_net`` struct."""

    def __init__(self, qp: dict, device):
        self.device = torch.device(device)
        self.in_scale, self.in_zp = float(qp["in_scale"]), int(qp["in_zp"])
        # 1/scale in fp32, as aten::quantize_per_tensor computes it
        self.in_inv_scale = float(torch.tensor(1.0, dtype=torch.float32) / torch.tensor(self.in_scale, dtype=torch.float32))
        s, zp = self.in_scale, self.in_zp
        self.convs = []
        for i in range(1, 7):
            L = qp[f"conv{i}"]
            self.convs.append(PackedConv(f"conv{i}", L, s, zp, self.device, relu=True))
            s, zp = float(L["out_scale"]), int(L["out_zp"])
        self.fc1 = PackedLinear("fc1", qp["fc1"], s, zp, self.device, relu=True, nhwc_from=(256, 4, 4))
        s, zp = float(qp["fc1"]["out_scale"]), int(qp["fc1"]["out_zp"])
        self.fc2 = PackedLinear("fc2", qp["fc2"], s, zp, self.device, relu=False)
        self.out_scale, self.out_zp = float(qp["fc2"]["out_scale"]), int(qp["fc2"]["out_zp"])
        self.input_lut = input_lut(self.in_scale, self.in_zp)  # host uint8 [3][256] (uint8 data path)
        net = _lib.StaticNet()
        net.in_inv_scale, net.in_zp = self.in_inv_scale, self.in_zp
        for i, pc in enumerate(self.convs):
            net.conv[i] = pc.c
        net.fc1, net.fc2, net.out_scale = self.fc1.c, self.fc2.c, self.out_scale
        self.c = net

    def ptr(self):
        return C.byref(self.c)

    def weight_bytes(self) -> int:
        return sum(p.w.numel() for p in self.convs) + self.fc1.w.numel() + self.fc2.w.numel()


class PackedSandwichNet:
    """Device constants of the per-layer sandwich net (``ptq.calibrate_sandwich``) + the ``b200q_sandwich_net`` struct.

    conv1..conv6 and fc1 are packed as in the static net with ReLU fusion off and each layer's own QuantStub
    (``in_scale`` / ``in_zp``); ``luts[i]`` is the boundary table (DeQuantStub -> ReLU -> next QuantStub) after layer i
    (``ptq.sandwich_boundary_lut``); fc2 stays fp32."""

    def __init__(self, sp: dict, device):
        from . import ptq
        self.device = torch.device(device)
        names = ptq.SANDWICH_LAYERS
        self.convs = [PackedConv(n, sp[n], sp[n]["in_scale"], sp[n]["in_zp"], self.device, relu=False) for n in names[:6]]
        self.fc1 = PackedLinear("fc1", sp["fc1"], sp["fc1"]["in_scale"], sp["fc1"]["in_zp"], self.device, relu=False,
                                nhwc_from=(256, 4, 4))
        self.fc1_scale, self.fc1_zp = float(sp["fc1"]["out_scale"]), int(sp["fc1"]["out_zp"])
        self.fc2_w = sp["fc2"]["weight"].detach().to(self.device, torch.float32).contiguous()
        self.fc2_b = sp["fc2"]["bias"].detach().to(self.device, torch.float32).contiguous()
        if tuple(self.fc2_w.shape) != (10, 512) or tuple(self.fc2_b.shape) != (10,):
            raise _lib.B200QError(f"sandwich fc2 must be fp32 [10,512] + [10], got {tuple(self.fc2_w.shape)} + "
                                  f"{tuple(self.fc2_b.shape)}")
        self.luts = [ptq.sandwich_boundary_lut(sp[a]["out_scale"], sp[a]["out_zp"], sp[b]["in_scale"], sp[b]["in_zp"])
                     for a, b in zip(names[:-1], names[1:])]
        s_in = float(sp["conv1"]["in_scale"])
        net = _lib.SandwichNet()
        net.in_inv_scale = float(torch.tensor(1.0, dtype=torch.float32) / torch.tensor(s_in, dtype=torch.float32))
        for i, pc in enumerate(self.convs):
            net.conv[i] = pc.c
        net.fc1 = self.fc1.c
        for i, lut in enumerate(self.luts):
            C.memmove(net.lut_host[i], lut.numpy().tobytes(), 256)
        net.fc1_scale = self.fc1_scale
        net.fc2_w, net.fc2_b = self.fc2_w.data_ptr(), self.fc2_b.data_ptr()
        self.c = net

    def ptr(self):
        return C.byref(self.c)
