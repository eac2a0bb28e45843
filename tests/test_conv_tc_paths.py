"""Every launch path of the tensor-core convolution (csrc/conv_tc.cu) against a float64 convolution of the exact operands.

The host rule (mr_conv2d_nhwc_tc_plan, `conv.tc_plan`) picks, per call, one of three kernels -- tap-refetch (1, 2 or 4 CTAs
per SM, 1 to 4 sub-pixel phases per launch), halo with resident weights (2 or 3 CTAs per SM, 128- or 64-byte rows), halo with
streamed weights (a ring of 3 to 8 weight stages) -- and one of three epilogues (staged, one-column for Cout == 1, generic).
Each case of CASES names the plan it must get, in tf32 and in f16 mode; the CPU test holds the rule to that, the GPU tests run
the case and compare every output element with

    |out - act(ref)| <= L * c * 2^-24 * sqrt(K) * S + r * |act(ref)| + tiny

where ref and S = conv(|x|, |w|) + |bias| are float64 convolutions of the operands the kernel multiplies (inputs on the TF32
grid or half, weights rounded the way the packer rounds them), K = Cin * kh * kw, L the Lipschitz constant of the activation,
r = 2^-11 for TF32-rounded or half outputs and 0 for fp32 outputs, tiny = 2^-24 (half subnormal spacing) plus the evaluation
error of sigmoid / |tanh|.  The products are exact in fp32 (11-bit mantissas), so the first term is the fp32 accumulation.
The same cases, with the same gate, run through the fp32 CUDA-core kernel.

C_GATE: measured on a B200 (148 SMs, 1000 W power limit), the worst c of any case and variant was 0.374 in tf32 (cout200),
0.212 in f16 (cout200) and 0.549 on the CUDA-core kernel (halo_1x1_c20); `-s` prints it per case.  Values below 1 are what fp32
accumulation gives.  The gate is 2, under 4x the worst measured value.
"""
import math

import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"
C_GATE = 2.0
MODES = ("tf32", "f16", "fp32")
TC_MODES = ("tf32", "f16")
SMS = 148   # SM count of a B200; the CPU test plans for it, the GPU tests for the device they run on


def _leaky_ref(y, a):
    return torch.where(y >= 0, y, a * y)


class Case:
    """One layer: kind "conv" (PackedConv), "refine" (4 sub-pixel 2x2 phases) or "upconv" (1x1 / 1x2 / 2x1 / 2x2 phases).
    H, W: source size; plan: mode -> (kernel, ctas_per_sm, row_bytes, epilogue[, b_stream]); persistent: at least 3 tiles per
    CTA on the device."""

    def __init__(self, cid, kind, src_c, cout, kh, kw, stride, B, H, W, act, a, b, final, plan, persistent=False, src_c_f16=None):
        self.cid, self.kind, self.src_c, self.cout, self.kh, self.kw, self.stride = cid, kind, src_c, cout, kh, kw, stride
        self.B, self.H, self.W, self.act, self.a, self.b, self.final = B, H, W, act, a, b, final
        self.plan, self.persistent = plan, persistent
        self.src_c_f16 = src_c_f16 or src_c     # f16 sources need channel counts that are multiples of 8

    def channels(self, mode):
        return self.src_c_f16 if mode == "f16" else self.src_c

    def __repr__(self):
        return self.cid


LK, SG, AT = 1, 2, 3   # conv.ACT_LEAKY, ACT_SIGMOID, ACT_ABSTANH
CASES = [
    # ---- tap-refetch: strided k x 1 / 1 x k layers at 1, 2 and 4 CTAs per SM, sub-pixel phases ----
    Case("refetch_3x1_s2_c256", "conv", (128,), 256, 3, 1, (2, 1), 3, 61, 75, LK, 0.1, 1.0, False,
         {"tf32": ("refetch", 1, 128, "staged"), "f16": ("refetch", 1, 128, "staged")}),
    Case("refetch_1x5_s2_c192", "conv", (64,), 192, 1, 5, (1, 2), 3, 21, 97, LK, 0.1, 1.0, False,
         {"tf32": ("refetch", 1, 128, "staged"), "f16": ("refetch", 1, 128, "staged")}),
    Case("refetch_7x1_s2_c128", "conv", (48,), 128, 7, 1, (2, 1), 3, 45, 35, LK, 0.1, 1.0, False,
         {"tf32": ("refetch", 2, 128, "staged"), "f16": ("refetch", 2, 128, "staged")}),
    Case("refetch_1x7_s2_c40", "conv", (32,), 40, 1, 7, (1, 2), 3, 123, 1179, LK, 0.1, 1.0, False,
         {"tf32": ("refetch", 4, 128, "staged"), "f16": ("refetch", 4, 64, "staged")}, persistent=True),
    Case("refetch_5x1_s2_c64_final", "conv", (64,), 64, 5, 1, (2, 1), 3, 37, 27, LK, 0.1, 1.0, True,
         {"tf32": ("refetch", 4, 128, "staged"), "f16": ("refetch", 4, 128, "staged")}),
    Case("refine_3src", "refine", (192, 128, 256), 128, 2, 2, (1, 1), 3, 15, 21, LK, 0.1, 1.0, False,
         {"tf32": ("refetch", 2, 128, "staged"), "f16": ("refetch", 2, 128, "staged")}),
    Case("refine_c256", "refine", (256,), 256, 2, 2, (1, 1), 3, 9, 14, LK, 0.1, 1.0, False,
         {"tf32": ("refetch", 1, 128, "staged"), "f16": ("refetch", 1, 128, "staged")}),
    Case("upconv_unequal_phases", "upconv", (64, 32), 48, 2, 2, (1, 1), 3, 29, 580, 0, 0.0, 1.0, False,
         {"tf32": ("refetch", 4, 128, "staged"), "f16": ("refetch", 4, 128, "staged")}, persistent=True),
    # ---- halo kernel, resident weights: 2 / 3 CTAs per SM, 128- / 64-byte rows, kh or kw up to 7, 1x1 ----
    Case("halo_3x3_c32", "conv", (32,), 32, 3, 3, (1, 1), 3, 190, 293, LK, 0.1, 1.0, False,
         {"tf32": ("halo", 2, 128, "staged"), "f16": ("halo", 3, 64, "staged")}, persistent=True),
    Case("halo_1x7_c16", "conv", (16,), 16, 1, 7, (1, 1), 3, 37, 53, LK, 0.1, 1.0, False,
         {"tf32": ("halo", 2, 128, "staged"), "f16": ("halo", 3, 64, "staged")}),
    Case("halo_7x1_c24", "conv", (24,), 24, 7, 1, (1, 1), 3, 45, 29, LK, 0.1, 1.0, False,
         {"tf32": ("halo", 2, 128, "staged"), "f16": ("halo", 3, 64, "staged")}),
    Case("halo_1x1_c20", "conv", (32,), 20, 1, 1, (1, 1), 3, 35, 43, LK, 0.1, 1.0, False,
         {"tf32": ("halo", 3, 128, "staged"), "f16": ("halo", 3, 64, "generic")}),
    Case("halo_3x3_c48", "conv", (48,), 48, 3, 3, (1, 1), 3, 33, 47, LK, 0.1, 1.0, False,
         {"tf32": ("halo_stream", 2, 128, "staged", 8), "f16": ("halo", 2, 128, "staged")}),
    Case("halo_3x1_c48", "conv", (48,), 48, 3, 1, (1, 1), 3, 29, 37, LK, 0.1, 1.0, False,
         {"tf32": ("halo", 2, 128, "staged"), "f16": ("halo", 3, 128, "staged")}),
    # ---- halo kernel, streamed weights: 3 sources with tail chunks, ring depths 8 and 3 ----
    Case("stream_3src_tails", "conv", (36, 44, 20), 48, 3, 3, (1, 1), 3, 131, 291, LK, 0.1, 1.0, False,
         {"tf32": ("halo_stream", 2, 128, "staged", 8), "f16": ("halo_stream", 2, 128, "staged", 8)}, persistent=True,
         src_c_f16=(40, 48, 24)),
    Case("stream_7x7_c40", "conv", (32,), 40, 7, 7, (1, 1), 3, 27, 35, LK, 0.1, 1.0, False,
         {"tf32": ("halo_stream", 2, 128, "staged", 3), "f16": ("halo_stream", 2, 64, "staged", 8)}),
    Case("stream_3x3_c128", "conv", (128,), 128, 3, 3, (1, 1), 3, 23, 41, LK, 0.1, 1.0, False,
         {"tf32": ("halo_stream", 2, 128, "staged", 3), "f16": ("halo_stream", 2, 128, "staged", 3)}),
    # ---- channel counts (n_pad > Cout) and epilogues ----
    Case("cout200", "conv", (32,), 200, 3, 3, (1, 1), 3, 19, 27, LK, 0.1, 1.0, True,
         {"tf32": ("refetch", 1, 128, "staged"), "f16": ("refetch", 1, 64, "staged")}),
    Case("cout256", "conv", (256,), 256, 1, 3, (1, 1), 3, 13, 22, LK, 0.1, 1.0, False,
         {"tf32": ("refetch", 1, 128, "staged"), "f16": ("refetch", 1, 128, "staged")}),
    Case("cout6_generic", "conv", (32,), 6, 3, 3, (1, 1), 3, 21, 30, LK, 0.1, 1.0, False,
         {"tf32": ("halo", 2, 128, "generic"), "f16": ("halo", 3, 64, "generic")}),
    Case("sigmoid_cout16_generic", "conv", (32,), 16, 3, 3, (1, 1), 3, 19, 25, SG, 0.0, 1.0, False,
         {"tf32": ("halo", 2, 128, "generic"), "f16": ("halo", 3, 64, "generic")}),
    Case("head_sigmoid_1x1", "conv", (48,), 1, 1, 1, (1, 1), 3, 35, 51, SG, 0.0, 1.0, True,
         {"tf32": ("halo", 3, 128, "one_column"), "f16": ("halo", 3, 128, "one_column")}),
    Case("head_abstanh_3x3", "conv", (24,), 1, 3, 3, (1, 1), 3, 33, 45, AT, 0.25, 2.5, True,
         {"tf32": ("halo", 2, 128, "one_column"), "f16": ("halo", 3, 64, "one_column")}),
    Case("head_abstanh_c128", "conv", (128,), 1, 3, 3, (1, 1), 3, 17, 29, AT, -0.5, 0.75, True,
         {"tf32": ("halo_stream", 2, 128, "one_column", 8), "f16": ("halo", 2, 128, "one_column")}),
    Case("head_abstanh_c256", "conv", (256,), 1, 3, 3, (1, 1), 3, 11, 19, AT, 0.25, 2.5, True,
         {"tf32": ("halo_stream", 2, 128, "one_column", 8), "f16": ("halo_stream", 2, 128, "one_column", 8)}),
]
CASE_IDS = [c.cid for c in CASES]
BY_ID = dict(zip(CASE_IDS, CASES))


def _layer(case, mode, act_a=None, device="cpu", seed=0):
    """The case's layer object (weights ~ N(0, 1/K), bias ~ N(0, 1)) for `mode`'s channel counts."""
    from monorec_b200 import conv as C
    src_c = case.channels(mode)
    g = torch.Generator().manual_seed(1000 + seed + sum(map(ord, case.cid)))
    cin = sum(src_c)
    a = case.a if act_a is None else act_a
    if case.kind == "conv":
        w = torch.randn(case.cout, cin, case.kh, case.kw, generator=g) / math.sqrt(cin * case.kh * case.kw)
        bias = torch.randn(case.cout, generator=g)
        return C.PackedConv(w.to(device), bias.to(device), src_c, stride=case.stride, act=case.act, act_a=a, act_b=case.b)
    if case.kind == "refine":
        ct = torch.nn.ConvTranspose2d(cin, case.cout, 4, stride=2)
        with torch.no_grad():
            ct.weight.copy_(torch.randn(ct.weight.shape, generator=g) / math.sqrt(cin * 4))
            ct.bias.copy_(torch.randn(case.cout, generator=g))
        return C.refine_layer(ct.to(device), src_c, act=case.act, act_a=a)
    up = torch.nn.Conv2d(cin, case.cout, 2)
    with torch.no_grad():
        up.weight.copy_(torch.randn(up.weight.shape, generator=g) / math.sqrt(cin * 4))
        up.bias.copy_(torch.randn(case.cout, generator=g))
    return C.upconv_layer(up.to(device), src_c)


def _sources(case, mode, device, B=None, seed=0):
    """Inputs on the TF32 grid (tf32 / fp32) or half, N(0, 1), NHWC."""
    from monorec_b200 import conv as C
    g = torch.Generator().manual_seed(seed + 7)
    out = []
    for c in case.channels(mode):
        x = torch.randn(B or case.B, case.H, case.W, c, generator=g)
        out.append(x.half().to(device) if mode == "f16" else C._round_tf32(x).to(device))
    return out


def _out_hw(case, L):
    if case.kind != "conv":
        return case.H, case.W
    return math.ceil(case.H / case.stride[0]), math.ceil(case.W / case.stride[1])


def _plan_kwargs(mode, final):
    """How PackedConv.__call__ calls conv2d_tc in `mode`."""
    return dict(round_out=not final, half=False) if mode == "tf32" else dict(round_out=False, half=True, out_f32=final)


def _plan(case, mode, srcs, L, out=None, out_coff=0, sms=SMS):
    from monorec_b200 import conv as C
    if case.kind == "conv":
        return C.tc_plan(L, srcs, out=out, out_hw=_out_hw(case, L), out_coff=out_coff, sms=sms, **_plan_kwargs(mode, case.final))
    return C.tc_plan(L, srcs, out=out, round_out=mode == "tf32", half=mode == "f16", sms=sms)


def _signature(p):
    return (p["kernel"], p["ctas_per_sm"], p["row_bytes"], p["n_phases"] > 1, p["epilogue"])


def _check_plan(case, mode, p):
    exp = case.plan[mode]
    got = (p["kernel"], p["ctas_per_sm"], p["row_bytes"], p["epilogue"])
    assert got == exp[:4], f"{case.cid} {mode}: plan {got} != {exp[:4]} ({p})"
    if len(exp) > 4:
        assert p["b_stream"] == exp[4], f"{case.cid} {mode}: weight ring of {p['b_stream']} stages, expected {exp[4]}"
    if case.kind != "conv":
        assert p["n_phases"] == 4


# ---------------------------------------------------------------------------------------------------------------------
# host only: the dispatch rule keeps every case on its path; the argument checks that need no driver
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", TC_MODES)
@pytest.mark.parametrize("cid", CASE_IDS)
def test_case_plans_on_the_host(cid, mode):
    case = BY_ID[cid]
    L = _layer(case, mode)
    srcs = [torch.empty(case.B, case.H, case.W, c, dtype=torch.float16 if mode == "f16" else torch.float32)
            for c in case.channels(mode)]
    p = _plan(case, mode, srcs, L)
    _check_plan(case, mode, p)
    assert p["grid"] == min(SMS * p["ctas_per_sm"], p["total_tiles"]) and p["smem_bytes"] <= 212 * 1024
    assert p["tmem_cols"] * p["ctas_per_sm"] <= 512
    if case.persistent:
        assert p["total_tiles"] >= 3 * p["grid"], (cid, mode, p)


def test_plan_argument_checks_without_gpu():
    import ctypes
    from monorec_b200 import _lib
    from monorec_b200 import conv as C
    lib = _lib.load()
    case = BY_ID["halo_3x3_c32"]
    L = _layer(case, "tf32")
    x = torch.empty(1, 16, 24, 32)
    out = torch.empty(1, 16, 24, 32)
    descs, n_pad, k_pad = C._tc_descs([x], [L], out, (16, 24), False)
    p = C.TcPlan()

    def rc(descs=descs, n_phases=1, n_pad=n_pad, k_pad=k_pad, sms=SMS, plan=ctypes.byref(p)):
        return lib.mr_conv2d_nhwc_tc_plan(descs, n_phases, n_pad, k_pad, 0, sms, plan), lib.mr_last_error().decode()

    assert rc()[0] == 0 and C.TC_KERNELS[p.kernel] == "halo"
    assert rc(descs=None) == (-1, "mr_conv2d_nhwc_tc: null descriptor")
    assert rc(plan=None)[0] == -1
    assert rc(n_phases=5)[0] == -1 and "phases" in rc(n_phases=5)[1]
    assert rc(sms=0)[0] == -1
    assert rc(k_pad=k_pad + 32)[0] == -1 and "does not match" in rc(k_pad=k_pad + 32)[1]
    assert rc(n_pad=24)[0] == -1 and rc(n_pad=272)[0] == -1
    d = descs[0]
    for field, bad, msg in [("src_c", None, "multiple of 4"), ("dst_coff", 1, "channel slice"), ("act", 7, "activation"),
                            ("Ho", 17, "placement"), ("upsample2", 1, "upsample"), ("sy", 5, "stride"), ("src_dtype", 3, "src_dtype")]:
        saved = getattr(d, field) if field != "src_c" else d.src_c[0]
        if field == "src_c":
            d.src_c[0] = 30
        else:
            setattr(d, field, bad)
        r, m = rc()
        assert r == -1 and msg in m, (field, r, m)
        if field == "src_c":
            d.src_c[0] = saved
        else:
            setattr(d, field, saved)
    assert rc()[0] == 0
    # the launch runs the same checks before it needs the driver
    d.dst_coff = 1
    assert lib.mr_conv2d_nhwc_tc(descs, n_pad, k_pad, 0, None) == -1 and b"channel slice" in lib.mr_last_error()
    d.dst_coff = 0
    # sub-pixel phases must agree on everything but filter, padding, weights and output offset
    sub = _layer(BY_ID["refine_3src"], "tf32")
    xs = [torch.empty(1, 4, 6, c) for c in (192, 128, 256)]
    o = torch.empty(1, 8, 12, 128)
    descs4, n_pad4, k_pad4 = C._tc_descs(xs, sub.subs, o, (4, 6), False)
    assert lib.mr_conv2d_nhwc_tc_plan(descs4, 4, n_pad4, k_pad4, 1, SMS, ctypes.byref(p)) == 0 and p.total_tiles == 4
    descs4[2].act_a = 0.5
    assert lib.mr_conv2d_nhwc_tc_plan(descs4, 4, n_pad4, k_pad4, 1, SMS, ctypes.byref(p)) == -1
    assert b"phase 2 differs" in lib.mr_last_error()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: run the cases, gate every element against float64
# ---------------------------------------------------------------------------------------------------------------------
WORST = {}   # (case, mode, variant) -> worst c, printed at the end of the module


@pytest.fixture(scope="module", autouse=True)
def _report_worst_c():
    yield
    if WORST:
        print("\nworst c = (|out - act(ref)| - r |act(ref)| - tiny) / (L 2^-24 sqrt(K) S) per case:")
        for k in sorted(WORST):
            print(f"  {' '.join(k):60s} {WORST[k]:.3f}")
        print(f"  max {max(WORST.values()):.3f} (gate c = {C_GATE})")


def _act64(y, act, a, b):
    if act == LK:
        return _leaky_ref(y, a)
    if act == SG:
        return torch.sigmoid(y)
    if act == AT:
        return a + b * torch.tanh(y).abs()
    return y


def _lipschitz(act, a, b):
    if act == LK:
        return 1.0 if abs(a) <= 1 else max(1.0, abs(a))
    if act == SG:
        return 0.25
    if act == AT:
        return abs(b)
    return 1.0


def _phase_refs(case, mode, L, srcs, act_a):
    """[(py_slice, px_slice, ref, S, K)] in float64 for each phase (a conv is one phase at offset 0, step 1)."""
    from monorec_b200 import conv as C
    x = torch.cat([s.double() for s in srcs], 3).permute(0, 3, 1, 2)      # NCHW float64, exact copy of the operands
    subs = [L] if case.kind == "conv" else L.subs
    Hs, Ws = x.shape[2:]
    out_hw = _out_hw(case, L)
    res = []
    for P in subs:
        w = P._w_src.to(x.device, torch.float32)
        w = (w.half() if mode == "f16" else C._round_tf32(w) if mode == "tf32" else w).double()
        b = P.bias.to(x.device).double() if P.bias is not None else torch.zeros(P.cout, device=x.device, dtype=torch.float64)
        sy, sx = P.stride
        pt, pl = P.pad if P.pad is not None else (C.same_pad_before(Hs, P.kh, sy), C.same_pad_before(Ws, P.kw, sx))
        Ho, Wo = out_hw
        pb, pr = (Ho - 1) * sy + P.kh - Hs - pt, (Wo - 1) * sx + P.kw - Ws - pl
        xp = F.pad(x, (pl, max(pr, 0), pt, max(pb, 0)))
        y = F.conv2d(xp, w, None, (sy, sx))[:, :, :Ho, :Wo] + b.view(1, -1, 1, 1)
        S = F.conv2d(xp.abs(), w.abs(), None, (sy, sx))[:, :, :Ho, :Wo] + b.abs().view(1, -1, 1, 1)
        ref = _act64(y, P.act, act_a, P.act_b)
        oy, ox = P.out_off
        ys, xs_ = P.out_step
        res.append((slice(oy, oy + (Ho - 1) * ys + 1, ys), slice(ox, ox + (Wo - 1) * xs_ + 1, xs_),
                    ref.permute(0, 2, 3, 1), S.permute(0, 2, 3, 1), w.shape[1] * P.kh * P.kw))
    return res


def _run(case, mode, L, srcs, out, out_coff=0):
    """The layer through the engine's own dispatch for `mode`, into the caller's (NaN-filled) destination."""
    from monorec_b200 import conv as C
    old = C.MODE
    C.set_mode(mode)
    try:
        if case.kind == "conv":
            L(srcs, out=out, out_hw=_out_hw(case, L), final=case.final, out_coff=out_coff)
        elif mode == "fp32":
            for P in L.subs:
                P(srcs, out=out, out_hw=(case.H, case.W))
        else:
            C.conv2d_tc_phases(srcs, L.subs, out, (case.H, case.W), round_out=mode == "tf32", half=mode == "f16")
    finally:
        C.set_mode(old)
    return out


def _out_dtype(case, mode):
    return torch.float16 if (mode == "f16" and not case.final) else torch.float32


def _gate(case, mode, out, refs, act_a, coff, variant):
    """Every element of every phase within the bound; returns the worst c."""
    L_act = _lipschitz(case.act, act_a, case.b)
    rounded = not case.final and mode != "fp32"
    r = 2.0 ** -11 if rounded else 0.0
    tiny = 2.0 ** -24 + (2.0 ** -21 * (1 + abs(act_a) + abs(case.b)) if case.act in (SG, AT) else 0.0)
    worst = 0.0
    for ys, xs_, ref, S, K in refs:
        o = out[:, ys, xs_, coff:coff + case.cout]
        assert not torch.isnan(o).any(), f"{case.cid} {mode}: output pixels left unwritten"
        err = (o.double() - ref).abs()
        unit = L_act * 2.0 ** -24 * math.sqrt(K) * S
        excess = err - r * ref.abs() - tiny
        c = (excess / unit).max().item()
        worst = max(worst, c)
        if c > C_GATE:
            idx = torch.nonzero(excess > C_GATE * unit)[0].tolist()
            pytest.fail(f"{case.cid} {mode} {variant}: c = {c:.2f} > {C_GATE} at (b, y, x, ch) = {idx}: out {o[tuple(idx)].item()!r}, "
                        f"ref {ref[tuple(idx)].item()!r}, S {S[tuple(idx)].item():.3e}, K {K}")
        if rounded and out.dtype == torch.float32:   # stored activations are on the TF32 grid
            assert int((o.contiguous().view(torch.int32) & 0x1FFF).abs().max()) == 0
    WORST[(case.cid, mode, variant)] = max(WORST.get((case.cid, mode, variant), 0.0), worst)
    return worst


def _assert_nan_outside(out, case, coff, refs):
    """Every element the layer does not own is still the NaN it was filled with, bit for bit."""
    mask = torch.ones(out.shape, dtype=torch.bool, device=out.device)
    for ys, xs_, *_ in refs:
        mask[:, ys, xs_, coff:coff + case.cout] = False
    bits = out.view(torch.int16 if out.dtype == torch.float16 else torch.int32)
    nan_bits = torch.full((), float("nan"), dtype=out.dtype).view(bits.dtype).item()
    assert bool((bits[mask] == nan_bits).all()), f"{case.cid}: the kernel wrote outside its output region"


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cid", CASE_IDS)
def test_case_matches_float64(cid, mode):
    case = BY_ID[cid]
    L = _layer(case, mode, device=DEV)
    srcs = _sources(case, mode, DEV)
    Ho, Wo = _out_hw(case, L)
    step = 1 if case.kind == "conv" else 2
    out = torch.full((case.B, Ho * step, Wo * step, case.cout), float("nan"), device=DEV, dtype=_out_dtype(case, mode))
    if mode in TC_MODES:
        p = _plan(case, mode, srcs, L, out=out, sms=torch.cuda.get_device_properties(DEV).multi_processor_count)
        _check_plan(case, mode, p)
        if case.persistent:
            assert p["total_tiles"] >= 3 * p["grid"], p
    _run(case, mode, L, srcs, out)
    torch.cuda.synchronize()
    _gate(case, mode, out, _phase_refs(case, mode, L, srcs, case.a), case.a, 0, "")


SLOPE_CASES = ["refetch_1x7_s2_c40", "halo_3x3_c32", "stream_3x3_c128", "cout6_generic", "refine_3src"]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("slope", [0.1, 0.0, -0.3, 1.7])
@pytest.mark.parametrize("cid", SLOPE_CASES)
def test_leaky_slope(cid, slope, mode):
    """LeakyReLU is x >= 0 ? x : slope * x for any slope, in the staged and the generic epilogue (a slope above 1 is where
    max(x, slope * x) differs)."""
    case = BY_ID[cid]
    L = _layer(case, mode, act_a=slope, device=DEV)
    srcs = _sources(case, mode, DEV, seed=3)
    Ho, Wo = _out_hw(case, L)
    step = 1 if case.kind == "conv" else 2
    out = torch.full((case.B, Ho * step, Wo * step, case.cout), float("nan"), device=DEV, dtype=_out_dtype(case, mode))
    _run(case, mode, L, srcs, out)
    torch.cuda.synchronize()
    _gate(case, mode, out, _phase_refs(case, mode, L, srcs, slope), slope, 0, f"slope={slope}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", TC_MODES)
@pytest.mark.parametrize("coff,extra_c", [(8, 16), (3, 11)])
@pytest.mark.parametrize("cid", ["refetch_7x1_s2_c128", "halo_3x3_c32", "stream_3src_tails", "halo_1x1_c20"])
def test_guard_bands(cid, coff, extra_c, mode):
    """A channel slice (aligned: staged epilogue; unaligned: generic) of a NaN-filled destination larger than the output grid:
    the slice is gated like the plain output, every other element stays NaN bit for bit."""
    case = BY_ID[cid]
    L = _layer(case, mode, device=DEV)
    srcs = _sources(case, mode, DEV, seed=5)
    Ho, Wo = _out_hw(case, L)
    out = torch.full((case.B, Ho + 3, Wo + 5, case.cout + extra_c), float("nan"), device=DEV, dtype=_out_dtype(case, mode))
    p = _plan(case, mode, srcs, L, out=out, out_coff=coff, sms=torch.cuda.get_device_properties(DEV).multi_processor_count)
    aligned = coff % (8 if out.dtype == torch.float16 else 4) == 0 and (case.cout + extra_c) % (8 if out.dtype == torch.float16 else 4) == 0
    assert p["kernel"] == case.plan[mode][0]
    assert p["epilogue"] == (case.plan[mode][3] if aligned else "generic")
    _run(case, mode, L, srcs, out, out_coff=coff)
    torch.cuda.synchronize()
    refs = _phase_refs(case, mode, L, srcs, case.a)
    _gate(case, mode, out, refs, case.a, coff, f"coff={coff}")
    _assert_nan_outside(out, case, coff, refs)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", TC_MODES)
@pytest.mark.parametrize("cid", ["upconv_unequal_phases", "halo_3x3_c32", "stream_3src_tails"])
def test_bitwise_batch_and_repeat(cid, mode):
    """Each tile's arithmetic does not depend on which CTA runs it: batch element b alone equals element b of the B=3 batch
    (the tile -> CTA assignment differs), and two launches of the same layer are bitwise identical."""
    case = BY_ID[cid]
    L = _layer(case, mode, device=DEV)
    srcs = _sources(case, mode, DEV, seed=9)
    Ho, Wo = _out_hw(case, L)
    step = 1 if case.kind == "conv" else 2

    def run(ss):
        out = torch.full((ss[0].shape[0], Ho * step, Wo * step, case.cout), float("nan"), device=DEV, dtype=_out_dtype(case, mode))
        return _run(case, mode, L, ss, out)

    full, again = run(srcs), run(srcs)
    torch.cuda.synchronize()
    assert torch.equal(full.view(torch.int16 if full.dtype == torch.float16 else torch.int32),
                       again.view(torch.int16 if full.dtype == torch.float16 else torch.int32))
    for b in range(case.B):
        one = run([s[b:b + 1].contiguous() for s in srcs])
        torch.cuda.synchronize()
        assert torch.equal(one[0], full[b]), f"{cid} {mode}: batch element {b} differs when run alone"


@pytest.mark.gpu
@pytest.mark.parametrize("mode", TC_MODES)
def test_model_paths_are_in_the_matrix(mode, monkeypatch):
    """Every (kernel, CTAs per SM, row bytes, phases > 1, epilogue) one forward of MonoRecModel at 256x512, B=8, F=4 launches
    is a path some case above runs."""
    from monorec_b200 import conv as C
    from monorec_b200.model import MonoRecModel
    from monorec_b200.synthetic import make_inputs, seeded_state_dict, to_device
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    used = {}
    orig_tc, orig_ph = C.conv2d_tc, C.conv2d_tc_phases

    def conv2d_tc(srcs, L, out=None, out_hw=None, round_out=True, half=False, out_f32=False, out_coff=0):
        p = C.tc_plan(L, srcs, out=out, out_hw=out_hw, round_out=round_out, half=half, out_f32=out_f32, out_coff=out_coff, sms=sms)
        used.setdefault(_signature(p), (L.cout, L.src_c, L.kh, L.kw, L.stride))
        return orig_tc(srcs, L, out=out, out_hw=out_hw, round_out=round_out, half=half, out_f32=out_f32, out_coff=out_coff)

    def conv2d_tc_phases(srcs, subs, out, out_hw, round_out=True, half=False):
        p = C.tc_plan(C.PackedSubpixel(subs), srcs, out=out, round_out=round_out, half=half, sms=sms)
        used.setdefault(_signature(p), (subs[0].cout, subs[0].src_c, "phases"))
        return orig_ph(srcs, subs, out, out_hw, round_out=round_out, half=half)

    monkeypatch.setattr(C, "conv2d_tc", conv2d_tc)
    monkeypatch.setattr(C, "conv2d_tc_phases", conv2d_tc_phases)
    old = C.MODE
    C.set_mode(mode)
    try:
        model = MonoRecModel()
        model.load_state_dict(seeded_state_dict(model, seed=7, gain=0.7))
        model = model.to(DEV).eval()
        with torch.no_grad():
            model(to_device(make_inputs(8, 4, 256, 512, seed=1), DEV))
        torch.cuda.synchronize()
    finally:
        C.set_mode(old)
    matrix = set()
    for case in CASES:
        srcs = [torch.empty(case.B, case.H, case.W, c, dtype=torch.float16 if mode == "f16" else torch.float32)
                for c in case.channels(mode)]
        matrix.add(_signature(_plan(case, mode, srcs, _layer(case, mode), sms=sms)))
    print(f"\n{mode}: {len(used)} tensor-core paths in the model forward:", *sorted(used), sep="\n  ")
    missing = {s: used[s] for s in used if s not in matrix}
    assert not missing, f"paths the model takes that no case covers: {missing}"
