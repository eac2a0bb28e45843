"""Host-side logic that needs no GPU: checkpoint contract, padding arithmetic, descriptor ABI, weight packing."""
import ctypes

import pytest
import torch


def test_reference_checkpoint_loads(tmp_path):
    """Checkpoint contract (base/base_trainer.py:142-150, utils/util.py:244-248): DataParallel-prefixed state_dict."""
    from monorec_b200.model import MonoRecModel
    from monorec_b200.synthetic import seeded_state_dict
    src = MonoRecModel()
    sd = seeded_state_dict(src, seed=3, gain=1.0)
    torch.save({"arch": "DataParallel", "state_dict": {"module." + k: v for k, v in sd.items()}}, tmp_path / "cp.pth")
    m = MonoRecModel(checkpoint_location=[tmp_path / "cp.pth"])
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]), k
    torch.save({"arch": "MonoRecModel", "state_dict": sd}, tmp_path / "cp2.pth")
    m2 = MonoRecModel(mask_cp_loc=tmp_path / "cp2.pth", depth_cp_loc=tmp_path / "cp2.pth")
    assert torch.equal(m2.att_module.classifier[0].weight, sd["att_module.classifier.0.weight"])
    assert torch.equal(m2.depth_module.dec[4][2].bias, sd["depth_module.dec.4.2.bias"])


def test_same_padding_matches_reference_formula():
    from monorec_b200.conv import same_pad_before
    from oracle.convnet_oracle import same_pad
    for n in (16, 17, 32, 33, 64, 255, 256):
        for k in (1, 2, 3, 5, 7):
            for s in (1, 2):
                assert same_pad_before(n, k, s) == same_pad(n, k, s)[0]


def test_conv_desc_abi_matches_library():
    from monorec_b200 import _lib
    from monorec_b200.conv import ConvDesc
    assert ctypes.sizeof(ConvDesc) == _lib.load().mr_sizeof_conv_desc()


def test_convT_subkernels_reproduce_conv_transpose():
    """The four sub-pixel 2x2 kernels of pack_convT_k4s2 == ConvTranspose2d(k4,s2) + centre crop (layers.py:380-400)."""
    import torch.nn.functional as F
    from monorec_b200.conv import pack_convT_k4s2
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 5, 6, 7, generator=g)
    w = torch.randn(5, 4, 4, 4, generator=g)
    ref = F.conv_transpose2d(x, w, stride=2)[:, :, 1:-1, 1:-1]
    out = torch.zeros_like(ref)
    for (py, px), sub in pack_convT_k4s2(w).items():          # sub: [2][2][Cin][Cout]
        wk = sub.permute(3, 2, 0, 1)                           # (Cout, Cin, 2, 2) correlation kernel
        xp = F.pad(x, (1 - px, px, 1 - py, py))
        out[:, :, py::2, px::2] = F.conv2d(xp, wk)
    assert torch.allclose(out, ref, atol=1e-5)


def test_unsupported_reference_options_raise():
    from monorec_b200.model import MonoRecModel
    for kw in ({"simple_mask": True}, {"depth_large_model": True}, {"augmentation": "depth"}, {"use_ssim": False},
               {"cv_patch_size": 5}, {"sfcv_mult_mask": False}):
        with pytest.raises(NotImplementedError):
            MonoRecModel(**kw)
    m = MonoRecModel(pretrain_mode=2)
    assert hasattr(m, "att_module") and not hasattr(m, "depth_module")
    m = MonoRecModel(pretrain_mode=1)
    assert hasattr(m, "depth_module") and not hasattr(m, "att_module")


def test_trunk_batchnorm_folding_matches_unfolded_eval():
    """ResnetEncoder's inference path folds eval-mode BatchNorm into the convolutions (monorec_model.py:118-129 semantics);
    the folded copy must track parameter updates."""
    from monorec_b200.model import ResnetEncoder
    torch.manual_seed(0)
    enc = ResnetEncoder(18, pretrained=False).eval()
    for m in enc.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0, 0.5)
            m.running_var.uniform_(0.5, 2.0)
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.normal_(0, 0.2)
    x = torch.rand(2, 3, 64, 128)
    with torch.enable_grad():
        ref = [t.detach().clone() for t in enc(x)]          # module-by-module path
    with torch.no_grad():
        out = [t.clone() for t in enc(x)]                    # folded path
    assert len(out) == 5
    for a, b in zip(ref, out):
        assert a.shape == b.shape and float((a - b).abs().max()) <= 1e-5 * float(a.abs().max())
    sd = {k: v.clone() for k, v in enc.state_dict().items()}
    sd["encoder.bn1.bias"] += 1.0
    enc.load_state_dict(sd)
    with torch.no_grad():
        out2 = enc(x)[0]
    with torch.enable_grad():
        ref2 = enc(x)[0].detach()
    assert float((out2 - ref2).abs().max()) < 1e-4 and float((out2 - out[0]).abs().max()) > 0.5


def test_tc_weight_packing_chunk_widths():
    """Packed tensor-core weights: [taps][n_pad][k_pad], every source padded to whole K chunks; half sources of <= 32
    channels use 32-channel chunks (64-byte swizzle rows; the library derives the chunk width from k_pad:
    include/monorec_b200.h)."""
    from monorec_b200 import conv as C
    w = torch.randn(24, 32, 3, 3)
    wt, n_pad, k_pad = C.pack_tc_weight(w, (32,), half=False)
    assert wt.dtype == torch.float32 and wt.shape == (9, 32, 32) and (n_pad, k_pad) == (32, 32)
    assert torch.equal(wt[4, :24, :], C._round_tf32(w[:, :, 1, 1])) and float(wt[:, 24:].abs().max()) == 0.0
    wt, n_pad, k_pad = C.pack_tc_weight(w, (32,), half=True, allow_k32=True)
    assert wt.dtype == torch.float16 and k_pad == (32 if C.K32 else 64) and wt.shape == (9, 32, k_pad)
    wt, n_pad, k_pad = C.pack_tc_weight(w, (32,), half=True, allow_k32=False)
    assert k_pad == 64 and float(wt[:, :, 32:].abs().max()) == 0.0
    w2 = torch.randn(48, 96, 3, 3)
    wt, n_pad, k_pad = C.pack_tc_weight(w2, (32, 64), half=True)          # a 64-channel source keeps 64-channel chunks
    assert (n_pad, k_pad) == (48, 128) and torch.equal(wt[0, :, 64:128], w2[:, 32:, 0, 0].half())
    assert float(wt[:, :, 32:64].abs().max()) == 0.0
    s1 = C.PackedConv(w, None, (32,), stride=(1, 1))
    s2 = C.PackedConv(w, None, (32,), stride=(2, 1))
    assert s1.wtc(True)[2] == (32 if C.K32 else 64) and s2.wtc(True)[2] == (32 if C.K32 else 64)


def test_c_packer_matches_torch_restatement():
    """mr_pack_conv_weights (host-side C, include/monorec_b200.h) == the torch restatement of the layout, fp32/TF32 and half,
    one to three concatenated sources, ragged channel counts; padding rows and columns are zero."""
    from monorec_b200 import conv as C
    g = torch.Generator().manual_seed(3)
    for cout, src_c, kh, kw in [(24, (32,), 3, 3), (48, (32, 64), 3, 3), (96, (64, 64, 96), 1, 1), (1, (24,), 3, 3), (13, (40,), 7, 1)]:
        w = torch.randn(cout, sum(src_c), kh, kw, generator=g)
        for half in (False, True):
            got, n_pad, k_pad = C.pack_tc_weight(w, src_c, half=half)
            ref, n_ref, k_ref = C._pack_tc_weight_torch(w, src_c, half)
            assert (n_pad, k_pad) == (n_ref, k_ref) and got.dtype == ref.dtype and torch.equal(got, ref), (cout, src_c, half)


def test_c_subpixel_kernels_reproduce_reference_layers():
    """mr_subpixel_convt_k4s2 / mr_subpixel_upconv2: the four phase kernels reproduce ConvTranspose2d(k4, s2) + crop (Refine,
    model/layers.py:380-400) and Upsample(x2) + pad(0,1,0,1) + Conv2d(k2) (Upconv, :338-356)."""
    import ctypes
    import torch.nn.functional as F
    from monorec_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 5, 6, 7, generator=g)
    wt = torch.randn(5, 4, 4, 4, generator=g).contiguous()           # (Cin, Cout, 4, 4)
    ref = F.conv_transpose2d(x, wt, stride=2)[:, :, 1:-1, 1:-1]
    out = torch.zeros_like(ref)
    for py in (0, 1):
        for px in (0, 1):
            sub = torch.empty(4, 5, 2, 2)
            pt, pl = ctypes.c_int(-1), ctypes.c_int(-1)
            assert lib.mr_subpixel_convt_k4s2(wt.data_ptr(), 5, 4, py, px, sub.data_ptr(), ctypes.byref(pt), ctypes.byref(pl)) == 0
            assert (pt.value, pl.value) == (1 - py, 1 - px)
            xp = F.pad(x, (pl.value, 1 - pl.value, pt.value, 1 - pt.value))
            out[:, :, py::2, px::2] = F.conv2d(xp, sub)
    assert torch.allclose(out, ref, atol=1e-5)
    wu = torch.randn(3, 5, 2, 2, generator=g).contiguous()           # (Cout, Cin, 2, 2)
    up = F.interpolate(x, scale_factor=2, mode="nearest")
    ref = F.conv2d(F.pad(up, (0, 1, 0, 1)), wu)
    out = torch.zeros_like(ref)
    for py in (0, 1):
        for px in (0, 1):
            kh, kw = ctypes.c_int(0), ctypes.c_int(0)
            sub = torch.empty(3 * 5 * 4)
            assert lib.mr_subpixel_upconv2(wu.data_ptr(), 3, 5, py, px, sub.data_ptr(), ctypes.byref(kh), ctypes.byref(kw)) == 0
            sub = sub[:3 * 5 * kh.value * kw.value].view(3, 5, kh.value, kw.value)
            xp = F.pad(x, (0, kw.value - 1, 0, kh.value - 1))          # pixel o + 1 beyond the border is the reference's zero pad
            out[:, :, py::2, px::2] = F.conv2d(xp, sub)
    assert torch.allclose(out, ref, atol=1e-5)


def test_integration_monkey_patch_resolves_through_reference_config_parser(golden_dir):
    """INTEGRATION.md section 2: the reference builds its models by class name -- evaluate.py:29-31 calls
    ConfigParser.initialize_list("models", model.model), which looks every entry's "type" up in model.model and calls it
    with the entry's "args".  After the two-line patch that lookup yields the drop-in; fed the "models" block of
    configs/evaluate/eval_monorec.json, it must build monorec_b200's model, accept the reference constructor's keywords in
    the reference's order, and end up with the settings the reference's own model has (tests/golden/integration.json,
    written by `make_golden.py --only-integration` from the unmodified reference)."""
    import inspect
    import json
    import types
    import monorec_b200.model as fast
    g = json.loads((golden_dir / "integration.json").read_text())
    assert [n for n in inspect.signature(fast.MonoRecModel.__init__).parameters if n != "self"] == g["reference_init_keywords"]
    module_arch = types.ModuleType("model.model")          # the reference's model/model.py registry ...
    module_arch.MonoRecModel = fast.MonoRecModel            # ... after INTEGRATION.md's patch
    assert g["models"] and len(g["models"]) == len(g["reference_settings"])
    for entry, ref in zip(g["models"], g["reference_settings"]):
        model = getattr(module_arch, entry["type"])(**entry["args"])
        assert type(model) is fast.MonoRecModel and type(model).__module__ == "monorec_b200.model"
        got = {n: getattr(model, n) for n in ref}
        assert {n: (list(v) if isinstance(v, tuple) else v) for n, v in got.items()} == ref
        assert model.use_mono is True and model.use_stereo is False and model.pretrain_mode == 0
        assert tuple(model.inv_depth_min_max) == (0.33, 0.0025)


def test_trunk_unused_level_is_lazy_and_identical():
    """The 512-channel trunk level has no consumer in the reference (monorec_model.py:372-380, :545 read levels 0-3): it is
    evaluated on first use.  Slices / indices the Mask and Depth modules use do not trigger it; index 4, iteration and
    concatenation do, with the same values as the eager evaluation."""
    import monorec_b200.model as M
    enc = M.ResnetEncoder(18, pretrained=False).eval()
    x = torch.rand(2, 3, 64, 128)
    old = M.TRUNK_LAZY_LEVEL4
    try:
        with torch.no_grad():
            M.TRUNK_LAZY_LEVEL4 = False
            eager = enc(x)
            M.TRUNK_LAZY_LEVEL4 = True
            lazy = enc(x)
        assert type(eager) is list and isinstance(lazy, M._TrunkFeatures) and len(lazy) == 5
        assert len(lazy[:4]) == 4 and lazy[3].shape[1] == 256 and list.__getitem__(lazy, 4) is None      # not evaluated yet
        assert torch.equal(lazy[4], eager[4]) and torch.equal(lazy[-1], eager[4])
        with torch.no_grad():
            lazy2 = enc(x)
        assert all(torch.equal(a, b) for a, b in zip(lazy2, eager))                                        # iteration evaluates
        lazy2.reset_tail()
        assert list.__getitem__(lazy2, 4) is None and torch.equal((lazy2 + [])[4], eager[4])
    finally:
        M.TRUNK_LAZY_LEVEL4 = old
