"""Host side of the convolution engine: ctypes descriptor, weight packing and layer-level helpers.

Activations inside the engine are NHWC fp32 torch tensors; every helper launches kernels of libmonorec_b200.so on the
current CUDA stream through the C ABI (include/monorec_b200.h: mr_conv_desc).  Nothing here computes on the CPU and
nothing falls back to torch ops.
"""
import ctypes
import math
from ctypes import c_float, c_int, c_void_p

import torch

from . import _lib

import os

MAX_SRC = 3
ACT_NONE, ACT_LEAKY, ACT_SIGMOID, ACT_ABSTANH = 0, 1, 2, 3
LEAKY_SLOPE = 0.1  # model/layers.py:290, 318, 381
KC = 32            # channels per K chunk of the tensor-core kernel (csrc/conv_tc.cu)

# Arithmetic of the dense-contraction layers: "tf32" = tcgen05 tensor cores (kind::tf32, fp32 accumulate, fp32 storage),
# "f16" = tcgen05 kind::f16 with half NHWC activations and weights (fp32 accumulate; BASELINE config 3),
# "fp32" = CUDA-core FMA kernel (bit-level parity path).  1-channel heads always use the CUDA-core dot-product kernel.
MODE = os.environ.get("MONOREC_B200_CONV", "tf32").lower()
# half sources of <= 32 channels: 32-channel K chunks (SWIZZLE_64B rows), in the tap-refetch kernel and inside the halo box alike
# (round 2: 429 -> 203 us on the 32->32 3x3 layer over the single-frame volumes).
K32 = os.environ.get("MONOREC_B200_TC_K32", "1") != "0"
HALO_F16 = os.environ.get("MONOREC_B200_TC_HALO_F16", "1") != "0" and os.environ.get("MONOREC_B200_TC_HALO", "") != "0"
# the single-channel layers (1x1 mask classifier, the four 3x3 depth heads) run on the tensor cores too in the tf32 / f16
# modes (Cout padded to 16): 5.93 -> 5.83 ms per half-mode forward at B=8 against the CUDA-core per-pixel kernel (round 2)
TC_HEADS = True
DT_F32, DT_F16 = 0, 1
FLOPS = None       # set to [0] to count the conv stacks' flops during a forward (bench.py's tensor roofline)


def set_mode(mode):
    global MODE
    assert mode in ("tf32", "fp32", "f16")
    MODE = mode


def act_dtype():
    """torch dtype of the NHWC activations inside the engine for the current MODE."""
    return torch.float16 if MODE == "f16" else torch.float32


def _dt(t):
    return DT_F16 if t.dtype == torch.float16 else DT_F32


class ConvDesc(ctypes.Structure):
    """Mirror of `struct mr_conv_desc` (include/monorec_b200.h)."""
    _fields_ = [("n_src", c_int), ("src", c_void_p * MAX_SRC), ("src_c", c_int * MAX_SRC),
                ("B", c_int), ("Hs", c_int), ("Ws", c_int), ("upsample2", c_int),
                ("kh", c_int), ("kw", c_int), ("sy", c_int), ("sx", c_int), ("pad_t", c_int), ("pad_l", c_int),
                ("Ho", c_int), ("Wo", c_int), ("Cout", c_int),
                ("weight", c_void_p), ("bias", c_void_p), ("dst", c_void_p),
                ("dst_H", c_int), ("dst_W", c_int), ("dst_c", c_int), ("dst_coff", c_int),
                ("oy_step", c_int), ("ox_step", c_int), ("oy_off", c_int), ("ox_off", c_int),
                ("act", c_int), ("act_a", c_float), ("act_b", c_float), ("src_dtype", c_int), ("dst_dtype", c_int)]


def same_pad_before(n, k, s):
    """Leading zero padding of PadSameConv2d (model/layers.py:249-251); the trailing part is implicit (zero fill)."""
    total = s * (math.ceil(n / s) - 1) + k - n
    return total // 2


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def pack_conv_weight(w):
    """nn.Conv2d weight (Cout, Cin, kh, kw) -> [kh][kw][Cin][Cout] contiguous fp32."""
    return w.detach().to(torch.float32).permute(2, 3, 1, 0).contiguous()


def pack_convT_k4s2(w):
    """nn.ConvTranspose2d(k=4, s=2) weight (Cin, Cout, 4, 4) -> four sub-pixel 2x2 kernels [py][px] -> [2][2][Cin][Cout].

    With the reference's centre crop of one pixel (model/layers.py:269-286, oversize = -2) output pixel (Y, X) of the
    cropped 2H x 2W map receives input rows i with 2 i + ky = Y + 1:
        Y even (py = 0): (i, ky) = (Y/2 - 1, 3), (Y/2, 1)          Y odd (py = 1): (i, ky) = ((Y-1)/2, 2), ((Y+1)/2, 0)
    i.e. a 2-tap filter along each axis on the input grid with taps ordered by increasing i.
    """
    w = w.detach().to(torch.float32)
    taps = {0: (3, 1), 1: (2, 0)}
    out = {}
    for py in (0, 1):
        for px in (0, 1):
            sub = w[:, :, list(taps[py]), :][:, :, :, list(taps[px])]      # (Cin, Cout, 2, 2)
            out[(py, px)] = sub.permute(2, 3, 0, 1).contiguous()           # [2][2][Cin][Cout]
    return out


def conv2d(srcs, weight, bias, kh, kw, stride=(1, 1), act=ACT_NONE, act_a=0.0, act_b=1.0, upsample2=False,
           out=None, out_coff=0, pad=None, out_hw=None, out_step=(1, 1), out_off=(0, 0)):
    """One fused convolution launch.

    srcs: list of NHWC tensors [B, Hs, Ws, C_i] (concatenated along C in this order).  weight: packed [kh][kw][Cin][Cout].
    Returns the NHWC output tensor (allocated unless `out` is given; then the channel slice at `out_coff` is written).
    """
    lib = _lib.load()
    x0 = srcs[0]
    B, Hs, Ws, _ = x0.shape
    Hv, Wv = (2 * Hs, 2 * Ws) if upsample2 else (Hs, Ws)
    sy, sx = stride
    Cout = weight.shape[-1]
    if pad is None:
        pad = (same_pad_before(Hv, kh, sy), same_pad_before(Wv, kw, sx))
    if out_hw is None:
        out_hw = (math.ceil(Hv / sy), math.ceil(Wv / sx))
    Ho, Wo = out_hw
    if out is None:
        out = torch.empty(B, Ho * out_step[0], Wo * out_step[1], Cout, device=x0.device, dtype=torch.float32)
    d = ConvDesc()
    d.n_src = len(srcs)
    cin = 0
    for i, s in enumerate(srcs):
        assert s.is_cuda and s.dtype == x0.dtype and s.is_contiguous(), "conv sources must be contiguous CUDA tensors of one dtype"
        assert s.shape[:3] == x0.shape[:3], "concatenated sources must share B, H, W"
        d.src[i] = s.data_ptr()
        d.src_c[i] = s.shape[3]
        cin += s.shape[3]
    assert weight.shape == (kh, kw, cin, Cout), f"packed weight {tuple(weight.shape)} != {(kh, kw, cin, Cout)}"
    d.B, d.Hs, d.Ws, d.upsample2 = B, Hs, Ws, int(upsample2)
    d.kh, d.kw, d.sy, d.sx, d.pad_t, d.pad_l = kh, kw, sy, sx, pad[0], pad[1]
    d.Ho, d.Wo, d.Cout = Ho, Wo, Cout
    d.weight = weight.data_ptr()
    d.bias = bias.data_ptr() if bias is not None else None
    d.dst = out.data_ptr()
    d.dst_H, d.dst_W, d.dst_c, d.dst_coff = out.shape[1], out.shape[2], out.shape[3], out_coff
    d.oy_step, d.ox_step, d.oy_off, d.ox_off = out_step[0], out_step[1], out_off[0], out_off[1]
    d.act, d.act_a, d.act_b = act, act_a, act_b
    d.src_dtype, d.dst_dtype = _dt(x0), _dt(out)
    with torch.cuda.device(x0.device):
        _lib.check(lib.mr_conv2d_nhwc(ctypes.byref(d), _stream(x0)), "mr_conv2d_nhwc")
    return out


def conv_transpose_k4s2_crop(srcs, sub_weights, bias, act=ACT_LEAKY, act_a=LEAKY_SLOPE):
    """Refine (model/layers.py:380-400): ConvTranspose2d(k4, s2) + LeakyReLU + centre crop, as 4 sub-pixel 2x2 convs."""
    x0 = srcs[0]
    B, Hs, Ws, _ = x0.shape
    Cout = sub_weights[(0, 0)].shape[-1]
    out = torch.empty(B, 2 * Hs, 2 * Ws, Cout, device=x0.device, dtype=torch.float32)
    for py in (0, 1):
        for px in (0, 1):
            conv2d(srcs, sub_weights[(py, px)], bias, 2, 2, act=act, act_a=act_a, out=out,
                   pad=(1 - py, 1 - px), out_hw=(Hs, Ws), out_step=(2, 2), out_off=(py, px))
    return out


def nchw_to_nhwc(x, out=None, out_coff=0, one_minus=None, dtype=None):
    """fp32 (B,C,H,W) -> NHWC fp32 / half (optionally into a channel slice of `out`, optionally scaled by
    (1 - one_minus[b,0,h,w]))."""
    lib = _lib.load()
    dtype = (out.dtype if out is not None else dtype) or torch.float32
    if out is None and one_minus is None and x.dim() == 4 and x.dtype == torch.float32 and x.permute(0, 2, 3, 1).is_contiguous():
        v = x.permute(0, 2, 3, 1)             # already channels-last in memory (e.g. cuDNN NHWC output): a view, no kernel
        if dtype == torch.float32:
            return v
        o = torch.empty(v.shape, device=x.device, dtype=torch.float16)
        with torch.cuda.device(x.device):
            _lib.check(lib.mr_cast_f32_to_f16(v.data_ptr(), o.data_ptr(), v.numel(), _stream(x)), "mr_cast_f32_to_f16")
        return o
    x = x.contiguous()
    B, C, H, W = x.shape
    if out is None:
        out = torch.empty(B, H, W, C, device=x.device, dtype=dtype)
    om_t = None
    if one_minus is not None:    # the kernel reads fp32 [B,1,H,W]: any other dtype / shape would be read out of bounds
        om_t = one_minus.to(device=x.device, dtype=torch.float32).contiguous()
        assert om_t.numel() == B * H * W, f"one_minus must hold one value per pixel (B,1,H,W), got {tuple(one_minus.shape)}"
    fn, name = (lib.mr_nchw_to_nhwc_f16, "mr_nchw_to_nhwc_f16") if out.dtype == torch.float16 else (lib.mr_nchw_to_nhwc, "mr_nchw_to_nhwc")
    with torch.cuda.device(x.device):
        _lib.check(fn(x.data_ptr(), out.data_ptr(), B, C, H, W, out.shape[3], out_coff,
                      om_t.data_ptr() if om_t is not None else None, _stream(x)), name)
    return out        # (om_t stays referenced until the launch has been queued; the caching allocator is stream-ordered)


def as_nhwc(x, dtype):
    """(B,C,H,W) feature map -> NHWC tensor of `dtype`: a view when the memory is already channels-last in that type."""
    v = x.permute(0, 2, 3, 1)
    if x.dtype == dtype and v.is_contiguous():
        return v
    return nchw_to_nhwc(x.to(torch.float32), dtype=dtype)


def maxpool2(x):
    lib = _lib.load()
    B, H, W, C = x.shape
    out = torch.empty(B, H // 2, W // 2, C, device=x.device, dtype=x.dtype)
    fn, name = (lib.mr_maxpool2_nhwc_f16, "mr_maxpool2_nhwc_f16") if x.dtype == torch.float16 else (lib.mr_maxpool2_nhwc, "mr_maxpool2_nhwc")
    with torch.cuda.device(x.device):
        _lib.check(fn(x.data_ptr(), out.data_ptr(), B, H, W, C, _stream(x)), name)
    return out


def max_over_frames(x, frames):
    """x: [frames*B, ...] -> [B, ...] element-wise max over the leading frame axis."""
    if frames == 1:
        return x
    lib = _lib.load()
    B = x.shape[0] // frames
    out = torch.empty((B,) + tuple(x.shape[1:]), device=x.device, dtype=x.dtype)
    fn, name = (lib.mr_max_over_frames_f16, "mr_max_over_frames_f16") if x.dtype == torch.float16 else (lib.mr_max_over_frames, "mr_max_over_frames")
    with torch.cuda.device(x.device):
        _lib.check(fn(x.data_ptr(), out.data_ptr(), frames, out.numel(), _stream(x)), name)
    return out


def maxpool3s2_channels_last(x):
    """MaxPool2d(3, stride 2, padding 1) on an NCHW-shaped channels-last tensor (the ResNet stem pool); returns the same kind."""
    lib = _lib.load()
    B, Cc, H, W = x.shape
    xn = x.permute(0, 2, 3, 1)
    assert xn.is_contiguous()
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.empty(B, Ho, Wo, Cc, device=x.device, dtype=x.dtype)
    with torch.cuda.device(x.device):
        _lib.check(lib.mr_maxpool3s2_nhwc(xn.data_ptr(), out.data_ptr(), _dt(x), B, H, W, Cc, _stream(x)), "mr_maxpool3s2_nhwc")
    return out.permute(0, 3, 1, 2)


def pool_and_frame_max(x, frames):
    """x: [frames*B,H,W,C] -> (maxpool2(x) [frames*B,H/2,W/2,C], max over the frames [B,H,W,C]) in one pass over x."""
    lib = _lib.load()
    FB, H, W, Cc = x.shape
    B = FB // frames
    pooled = torch.empty(FB, H // 2, W // 2, Cc, device=x.device, dtype=x.dtype)
    fmax = torch.empty(B, H, W, Cc, device=x.device, dtype=x.dtype)
    with torch.cuda.device(x.device):
        _lib.check(lib.mr_pool_and_frame_max(x.data_ptr(), pooled.data_ptr(), fmax.data_ptr(), _dt(x), frames, B, H, W, Cc, _stream(x)),
                   "mr_pool_and_frame_max")
    return pooled, fmax


def mask_volume(volume, mask):
    """cost_volume * (1 - cv_mask) on NCHW tensors (model/monorec/monorec_model.py:713)."""
    lib = _lib.load()
    volume = volume.contiguous()
    mask = mask.to(torch.float32).contiguous()
    B, D, H, W = volume.shape
    out = torch.empty_like(volume)
    with torch.cuda.device(volume.device):
        _lib.check(lib.mr_mask_volume(volume.data_ptr(), mask.data_ptr(), out.data_ptr(), B, D, H * W, _stream(volume)),
                   "mr_mask_volume")
    return out


# --------------------------------------------------------------------------------------------------------------------
# layer objects: weights packed once for both kernels, dispatch by MODE
# --------------------------------------------------------------------------------------------------------------------
def _round_tf32(w):
    """Round-to-nearest onto the TF32 grid (10 explicit mantissa bits); the tensor core truncates the rest."""
    bits = w.contiguous().view(torch.int32)
    return ((bits + 0x1000) & ~0x1FFF).view(torch.float32)


def pack_tc_weight(w, src_c, half=False, allow_k32=True):
    """Correlation kernel (Cout, Cin, kh, kw) -> [kh*kw][n_pad][k_pad] K-major through the library's host-side packer
    (include/monorec_b200.h: mr_pack_conv_weights): every source padded to a whole number of K chunks (32 fp32 / 64 half
    channels = one 128-byte swizzle row, or 32 half channels = one 64-byte row when every source has <= 32 channels; zero
    rows), Cout padded to a multiple of 16; values rounded to TF32 (fp32 storage) or converted to half.
    allow_k32=False / MONOREC_B200_TC_K32=0 (experiments) force 64-channel chunks by packing in torch instead."""
    import ctypes
    Cout, Cin, kh, kw = w.shape
    assert sum(src_c) == Cin
    if half and not (K32 and allow_k32) and all(c <= 32 for c in src_c):
        return _pack_tc_weight_torch(w, src_c, half, kc=64)
    lib = _lib.load()
    wc = w.detach().to("cpu", torch.float32).contiguous()
    sc = (ctypes.c_int * len(src_c))(*[int(c) for c in src_c])
    n_pad, k_pad = ctypes.c_int(0), ctypes.c_int(0)
    dt = DT_F16 if half else DT_F32
    nbytes = lib.mr_pack_conv_weights_bytes(Cout, len(src_c), sc, kh, kw, dt, ctypes.byref(n_pad), ctypes.byref(k_pad))
    assert nbytes > 0
    out = torch.empty(kh * kw, n_pad.value, k_pad.value, dtype=torch.float16 if half else torch.float32)
    _lib.check(lib.mr_pack_conv_weights(wc.data_ptr(), Cout, len(src_c), sc, kh, kw, dt, out.data_ptr()), "mr_pack_conv_weights")
    return out.to(w.device), n_pad.value, k_pad.value


def _pack_tc_weight_torch(w, src_c, half, kc=None):
    """The same layout written with torch ops (the packer's restatement: tests compare the two)."""
    Cout, Cin, kh, kw = w.shape
    if kc is None:
        kc = (32 if all(c <= 32 for c in src_c) else 64) if half else KC
    n_pad = ((Cout + 15) // 16) * 16
    k_pad = sum(((c + kc - 1) // kc) * kc for c in src_c)
    out = torch.zeros(kh * kw, n_pad, k_pad, device=w.device, dtype=torch.float32)
    wt = w.detach().to(torch.float32).permute(2, 3, 0, 1).reshape(kh * kw, Cout, Cin)
    ci = ko = 0
    for c in src_c:
        out[:, :Cout, ko:ko + c] = wt[:, :, ci:ci + c]
        ci += c
        ko += ((c + kc - 1) // kc) * kc
    return (out.to(torch.float16).contiguous() if half else _round_tf32(out)), n_pad, k_pad


class PackedConv:
    """One convolution of the engine with its weights in both kernel layouts."""

    def __init__(self, weight, bias, src_c, stride=(1, 1), act=ACT_NONE, act_a=0.0, act_b=1.0, pad=None, out_step=(1, 1),
                 out_off=(0, 0), allow_tc=True):
        w = weight.detach().to(torch.float32)
        self.cout, self.cin, self.kh, self.kw = w.shape
        self.src_c = tuple(int(c) for c in src_c)
        self.stride, self.pad, self.out_step, self.out_off = stride, pad, out_step, out_off
        self.act, self.act_a, self.act_b = act, act_a, act_b
        self.bias = None if bias is None else bias.detach().to(torch.float32).contiguous()
        self.w32 = pack_conv_weight(w)
        self.tc_ok = (allow_tc or TC_HEADS) and self.cout <= 256 and (self.cout >= 8 or TC_HEADS) and all(c % 4 == 0 for c in self.src_c)
        self.tc_ok_f16 = self.tc_ok and all(c % 8 == 0 for c in self.src_c)
        self._wtc = {}
        self._w_src = w

    def wtc(self, half=False):
        if half not in self._wtc:
            self._wtc[half] = pack_tc_weight(self._w_src, self.src_c, half=half, allow_k32=True)
        return self._wtc[half]

    def __call__(self, srcs, out=None, out_hw=None, final=False, out_coff=0):
        """out_coff: first channel of the slice of `out` this layer writes (tensor-core path)."""
        assert tuple(s.shape[3] for s in srcs) == self.src_c, (tuple(s.shape[3] for s in srcs), self.src_c)
        if FLOPS is not None:      # bench.py: multiply-adds of this layer (2 flops each), counted on one eager forward
            Bn, Hs, Ws, _ = srcs[0].shape
            ho, wo = out_hw if out_hw is not None else (math.ceil(Hs / self.stride[0]), math.ceil(Ws / self.stride[1]))
            FLOPS[0] += 2 * Bn * ho * wo * self.cout * sum(self.src_c) * self.kh * self.kw
        if MODE == "f16" and srcs[0].dtype == torch.float16:
            if self.tc_ok_f16:
                return conv2d_tc(srcs, self, out=out, out_hw=out_hw, round_out=False, half=True, out_f32=final, out_coff=out_coff)
            assert self.cout == 1, "f16 mode: only the single-channel heads run on the CUDA-core kernel"
        if MODE == "tf32" and self.tc_ok:
            return conv2d_tc(srcs, self, out=out, out_hw=out_hw, round_out=not final, out_coff=out_coff)
        if out_coff:
            raise NotImplementedError("monorec_b200.conv: channel-slice outputs need the tensor-core path")
        return conv2d(srcs, self.w32, self.bias, self.kh, self.kw, stride=self.stride, act=self.act, act_a=self.act_a,
                      act_b=self.act_b, out=out, pad=self.pad, out_hw=out_hw, out_step=self.out_step, out_off=self.out_off)


def _tc_out(srcs, L, out, out_hw, half, out_f32):
    """(destination, output grid) of a PackedConv on the tensor cores: `out` or a new NHWC tensor."""
    x0 = srcs[0]
    B, Hs, Ws, _ = x0.shape
    if out_hw is None:
        out_hw = (math.ceil(Hs / L.stride[0]), math.ceil(Ws / L.stride[1]))
    if out is None:
        out = torch.empty(B, out_hw[0] * L.out_step[0], out_hw[1] * L.out_step[1], L.cout, device=x0.device,
                          dtype=torch.float16 if (half and not out_f32) else torch.float32)
    return out, out_hw


def _tc_descs(srcs, subs, out, out_hw, half, out_coff=0):
    """Descriptors of one tensor-core launch over the PackedConvs `subs` (one, or the sub-pixel phases of a layer, which share
    the first one's bias), with their packed weights' n_pad / k_pad."""
    descs = (ConvDesc * len(subs))()
    n_pad = k_pad = None
    for d, L in zip(descs, subs):
        wtc, n_pad_i, k_pad_i = L.wtc(half)
        assert n_pad in (None, n_pad_i) and k_pad in (None, k_pad_i)
        n_pad, k_pad = n_pad_i, k_pad_i
        Hs, Ws = srcs[0].shape[1:3]
        pad = L.pad if L.pad is not None else (same_pad_before(Hs, L.kh, L.stride[0]), same_pad_before(Ws, L.kw, L.stride[1]))
        _fill_desc(d, srcs, L, out, out_hw, pad, wtc, half, out_coff)
        d.bias = subs[0].bias.data_ptr() if subs[0].bias is not None else None
    return descs, n_pad, k_pad


def conv2d_tc(srcs, L, out=None, out_hw=None, round_out=True, half=False, out_f32=False, out_coff=0):
    """Tensor-core launch (csrc/conv_tc.cu) of a PackedConv."""
    lib = _lib.load()
    x0 = srcs[0]
    assert all(s.is_cuda for s in srcs)
    out, out_hw = _tc_out(srcs, L, out, out_hw, half, out_f32)
    descs, n_pad, k_pad = _tc_descs(srcs, [L], out, out_hw, half, out_coff)
    with torch.cuda.device(x0.device):
        _lib.check(lib.mr_conv2d_nhwc_tc(descs, n_pad, k_pad, int(round_out), _stream(x0)), "mr_conv2d_nhwc_tc")
    return out


def _fill_desc(d, srcs, L, out, out_hw, pad, wtc, half, out_coff=0):
    x0 = srcs[0]
    B, Hs, Ws, _ = x0.shape
    sy, sx = L.stride
    Ho, Wo = out_hw
    d.n_src = len(srcs)
    for i, s in enumerate(srcs):
        assert s.dtype == (torch.float16 if half else torch.float32) and s.is_contiguous()
        assert s.shape[:3] == x0.shape[:3]
        d.src[i] = s.data_ptr()
        d.src_c[i] = s.shape[3]
    d.B, d.Hs, d.Ws, d.upsample2 = B, Hs, Ws, 0
    d.kh, d.kw, d.sy, d.sx, d.pad_t, d.pad_l = L.kh, L.kw, sy, sx, pad[0], pad[1]
    d.Ho, d.Wo, d.Cout = Ho, Wo, L.cout
    d.weight = wtc.data_ptr()
    d.bias = L.bias.data_ptr() if L.bias is not None else None
    d.dst = out.data_ptr()
    d.dst_H, d.dst_W, d.dst_c, d.dst_coff = out.shape[1], out.shape[2], out.shape[3], int(out_coff)
    d.oy_step, d.ox_step, d.oy_off, d.ox_off = L.out_step[0], L.out_step[1], L.out_off[0], L.out_off[1]
    d.act, d.act_a, d.act_b = L.act, L.act_a, L.act_b
    d.src_dtype, d.dst_dtype = (DT_F16 if half else DT_F32), _dt(out)


def conv2d_tc_phases(srcs, subs, out, out_hw, round_out=True, half=False):
    """The sub-pixel convolutions of one Refine / Upconv layer in ONE launch (mr_conv2d_nhwc_tc_phases): same sources and
    destination, per-phase filter / padding / output offset; the phases of a spatial tile run side by side, so the input is
    read from HBM once instead of once per phase."""
    lib = _lib.load()
    x0 = srcs[0]
    assert all(s.is_cuda for s in srcs) and all(L.pad is not None for L in subs)
    descs, n_pad, k_pad = _tc_descs(srcs, subs, out, out_hw, half)
    with torch.cuda.device(x0.device):
        _lib.check(lib.mr_conv2d_nhwc_tc_phases(descs, len(subs), n_pad, k_pad, int(round_out), _stream(x0)), "mr_conv2d_nhwc_tc_phases")
    return out


class TcPlan(ctypes.Structure):
    """Mirror of `struct mr_conv_tc_plan` (include/monorec_b200.h)."""
    _fields_ = [(n, c_int) for n in ("kernel", "ctas_per_sm", "stages", "b_stream", "row_bytes", "kc", "tmem_cols", "smem_bytes",
                                     "total_tiles", "grid", "epilogue")]


TC_KERNELS = ("refetch", "halo", "halo_stream")          # MR_TC_REFETCH, MR_TC_HALO, MR_TC_HALO_STREAM
TC_EPILOGUES = ("staged", "one_column", "generic")       # MR_TC_EPI_*


def tc_plan(layer, srcs, out=None, out_hw=None, round_out=True, half=False, out_f32=False, out_coff=0, sms=None):
    """Launch plan (mr_conv2d_nhwc_tc_plan) of `conv2d_tc(srcs, layer, out, out_hw, round_out, half, out_f32, out_coff)` for a
    PackedConv, or of the one-launch call a PackedSubpixel makes (`out`: its (2H, 2W) destination), as a dict.  Host code only:
    the sources may be CPU tensors.  sms: SM count the grid is sized for (default: that of the sources' device)."""
    lib = _lib.load()
    x0 = srcs[0]
    if isinstance(layer, PackedSubpixel):
        subs = layer.subs
        if out is None:
            out = torch.empty(x0.shape[0], 2 * x0.shape[1], 2 * x0.shape[2], subs[0].cout, device=x0.device, dtype=x0.dtype)
        out_hw = tuple(x0.shape[1:3])
    else:
        subs = [layer]
        out, out_hw = _tc_out(srcs, layer, out, out_hw, half, out_f32)
    if sms is None:
        sms = torch.cuda.get_device_properties(x0.device).multi_processor_count
    descs, n_pad, k_pad = _tc_descs(srcs, subs, out, out_hw, half, out_coff)
    p = TcPlan()
    _lib.check(lib.mr_conv2d_nhwc_tc_plan(descs, len(subs), n_pad, k_pad, int(round_out), int(sms), ctypes.byref(p)),
               "mr_conv2d_nhwc_tc_plan")
    r = {n: getattr(p, n) for n, _ in TcPlan._fields_}
    r["kernel"], r["epilogue"], r["n_phases"] = TC_KERNELS[p.kernel], TC_EPILOGUES[p.epilogue], len(subs)
    return r


# MONOREC_B200_SUBPIXEL_ONE_LAUNCH=0: one launch per sub-pixel phase (A/B measurements)
SUBPIXEL_ONE_LAUNCH = os.environ.get("MONOREC_B200_SUBPIXEL_ONE_LAUNCH", "1") != "0"


class PackedSubpixel:
    """Four sub-pixel convolutions writing the (2H, 2W) output with step 2: Refine's ConvTranspose2d(k4, s2) + crop
    (model/layers.py:380-400) and Upconv's nearest-x2 + pad(0,1,0,1) + 2x2 conv (:338-356)."""

    def __init__(self, subs):
        self.subs = subs   # list of PackedConv

    def __call__(self, srcs):
        x0 = srcs[0]
        B, Hs, Ws, _ = x0.shape
        out = torch.empty(B, 2 * Hs, 2 * Ws, self.subs[0].cout, device=x0.device, dtype=x0.dtype)
        L0 = self.subs[0]
        half = MODE == "f16" and x0.dtype == torch.float16 and L0.tc_ok_f16
        if SUBPIXEL_ONE_LAUNCH and (half or (MODE == "tf32" and L0.tc_ok)) and all(L.pad is not None for L in self.subs):
            if FLOPS is not None:
                FLOPS[0] += sum(2 * B * Hs * Ws * L.cout * sum(L.src_c) * L.kh * L.kw for L in self.subs)
            return conv2d_tc_phases(srcs, self.subs, out, (Hs, Ws), round_out=not half, half=half)
        for L in self.subs:
            L(srcs, out=out, out_hw=(Hs, Ws))
        return out


def refine_layer(conv2d_t, src_c, act=ACT_LEAKY, act_a=LEAKY_SLOPE):
    w = conv2d_t.weight.detach().to(torch.float32)       # (Cin, Cout, 4, 4)
    taps = {0: (3, 1), 1: (2, 0)}                        # see pack_convT_k4s2
    subs = []
    for py in (0, 1):
        for px in (0, 1):
            sub = w[:, :, list(taps[py]), :][:, :, :, list(taps[px])].permute(1, 0, 2, 3).contiguous()  # (Cout,Cin,2,2)
            subs.append(PackedConv(sub, conv2d_t.bias, src_c, act=act, act_a=act_a, pad=(1 - py, 1 - px),
                                   out_step=(2, 2), out_off=(py, px)))
    return PackedSubpixel(subs)


def upconv_layer(conv, src_c):
    """out[2oy+py, 2ox+px] of nearest-x2 + 2x2 conv: even phases see both taps on the same input pixel (weights add up),
    odd phases see input pixels o and o+1 (zero beyond the border = the reference's trailing pad)."""
    w = conv.weight.detach().to(torch.float32)           # (Cout, Cin, 2, 2)
    subs = []
    for py in (0, 1):
        wy = w if py == 1 else w.sum(2, keepdim=True)
        for px in (0, 1):
            wyx = wy if px == 1 else wy.sum(3, keepdim=True)
            subs.append(PackedConv(wyx.contiguous(), conv.bias, src_c, pad=(0, 0), out_step=(2, 2), out_off=(py, px)))
    return PackedSubpixel(subs)
