#!/usr/bin/env python
"""Generates tests/golden/*.npz by running the UNMODIFIED reference from /root/reference on CPU fp32.

Run in the dev container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

The reference has no tests or golden vectors of its own (SURVEY.md §4), so these files are the pin for
both the oracle (oracle/*.py) and the CUDA path.  Nothing is copied from the reference: it is imported
in-place with the two shims of SURVEY.md Appendix B (kornia stub, torchvision weight download disabled).

Files written
  kitti_sample.npz        bundled KITTI sample (example/test_monorec.py: keyframe 169, frames 168/170):
                          uint8 inputs + reference CostVolumeModule outputs (sub-sampled volumes, full argmax,
                          valid masks, per-plane float64 checksums)
  cv_synth_small.npz      full reference cost-volume tensors for small seeded synthetic configs
  cv_synth_d64f6.npz      the same for 64 planes x 6 source frames (`--only-d64f6`)
  cv_config2.npz          BASELINE config 2's geometry at full size (256x512, 32 planes, 4 source frames, seed 100 of the
                          synthetic generator): sub-sampled volumes, rows, arg-max, validity, checksums (`--only-config2`)
  model_kitti_sample.npz  full MonoRecModel forward on the bundled KITTI sample, seeded weights (`--only-kitti-model`)
  model_synth_small.npz   full MonoRecModel forward (seeded weights, 2 gains) on a small synthetic config:
                          cv_mask, 4 depth maps, image_features checksums
  pointcloud.npz          the reference's PLYSaver.add_depthmap + mask dilation / vote on seeded inputs (`--only-pointcloud`)
  metrics.npz             the reference's seven sparse depth metrics on seeded inputs, four parameter sets (`--only-metrics`)
  reprojection.npz        the reference's reprojection_loss (model/loss_functions/common_losses.py) and its autograd gradient
                          w.r.t. the predicted inverse depth on seeded inputs, three argument sets (`--only-reprojection`)
  model_fp64.npz          the same two model configurations evaluated by the reference in float64 (`--only-model-fp64`):
                          the reference's own fp32 rounding noise on `result` / `cv_mask`, which sizes the GPU gates
  integration.json        the "models" block of configs/evaluate/eval_monorec.json, the reference MonoRecModel's constructor
                          keywords, and the settings of the models the reference's ConfigParser builds from that block
                          (`--only-integration`)
"""
import os
import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
REPO = HERE.parent.parent
REF = Path(os.environ.get("MONOREC_REFERENCE", "/root/reference"))
sys.path.insert(0, str(REPO))

from monorec_b200.synthetic import make_inputs, seeded_state_dict  # noqa: E402



def import_reference():
    """SURVEY.md Appendix B shims, then import the reference's model module."""
    for name in ["kornia", "kornia.augmentation", "kornia.geometry", "kornia.geometry.camera", "kornia.geometry.depth"]:
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["kornia.augmentation"].RandomHorizontalFlip = object
    sys.modules["kornia.augmentation"].RandomResizedCrop = object
    sys.modules["kornia.geometry.camera"].pixel2cam = None
    sys.modules["kornia.geometry.depth"].DepthWarper = None
    sys.modules["kornia"].augmentation = sys.modules["kornia.augmentation"]
    import torchvision
    orig = torchvision.models.resnet18
    torchvision.models.resnet18 = lambda pretrained=False, **kw: orig(weights=None)
    sys.path.insert(0, str(REF))
    import model.monorec.monorec_model as ref_mod  # noqa
    return ref_mod


def load_kitti_sample():
    """Restates the example loader for the single bundled sample.

    reference: example/test_monorec.py:18-45, data_loader/kitti_odometry_dataset.py:120-134 (crop, resize, /255-.5),
    :253-269 (frame selection), :318-374 (intrinsics).  Returns uint8 CHW images + float32 matrices.
    """
    from PIL import Image
    root = REF / "example" / "data" / "kitti"
    calib = {}
    for line in open(root / "sequences" / "07" / "calib.txt"):
        k, v = line.split(":", 1)
        calib[k] = np.array([float(x) for x in v.split()])
    P2 = calib["P2"].reshape(3, 4)
    H, W = 256, 512
    img0 = Image.open(root / "sequences" / "07" / "image_2" / "000169.png")
    ow, oh = img0.size
    r_orig, r_target = oh / ow, H / W
    assert r_orig < r_target
    new_w = oh / r_target
    box = ((ow - new_w) // 2, 0, ow - (ow - new_w) // 2, oh)
    c_x = (P2[0, 2] - (ow - new_w) / 2) / new_w
    c_y = P2[1, 2] / oh
    rescale = oh / H
    f_x = P2[0, 0] / W / rescale
    f_y = P2[1, 1] / H / rescale
    K = np.zeros((4, 4), np.float32)
    K[0, 0], K[1, 1], K[0, 2], K[1, 2], K[2, 2], K[3, 3] = f_x * W, f_y * H, c_x * W, c_y * H, 1, 1
    poses_all = np.loadtxt(root / "poses_dvso" / "07.txt").reshape(-1, 3, 4)

    def pose(i):
        p = np.eye(4, dtype=np.float32)
        p[:3] = poses_all[i]
        return p

    def image(i):
        im = Image.open(root / "sequences" / "07" / "image_2" / f"{i:06d}.png").crop(box)
        im = im.resize((W, H), resample=Image.BILINEAR)
        return np.array(im).transpose(2, 0, 1).copy()  # uint8 CHW

    return {"keyframe_u8": image(169), "frames_u8": np.stack([image(168), image(170)]), "K": K,
            "keyframe_pose": pose(169), "poses": np.stack([pose(168), pose(170)]), "crop_box": np.array(box)}


def sample_to_dict(s):
    to_t = lambda u8: (torch.from_numpy(u8.astype(np.float32)) / 255 - .5)
    nF = s["frames_u8"].shape[0]
    return {"keyframe": to_t(s["keyframe_u8"]).unsqueeze(0),
            "keyframe_pose": torch.from_numpy(s["keyframe_pose"]).unsqueeze(0),
            "keyframe_intrinsics": torch.from_numpy(s["K"]).unsqueeze(0),
            "frames": [to_t(s["frames_u8"][i]).unsqueeze(0) for i in range(nF)],
            "poses": [torch.from_numpy(s["poses"][i]).unsqueeze(0) for i in range(nF)],
            "intrinsics": [torch.from_numpy(s["K"]).unsqueeze(0) for _ in range(nF)]}


def run_ref_cv(ref_mod, data, steps=32, inv=(0.33, 0.0025)):
    cvm = ref_mod.CostVolumeModule()
    d = dict(data)
    key = d["keyframe"]
    d["inv_depth_min"] = key.new_tensor([inv[0]])
    d["inv_depth_max"] = key.new_tensor([inv[1]])
    d["cv_depth_steps"] = key.new_tensor([steps], dtype=torch.int32)
    with torch.no_grad():
        d = cvm(d)
    return d["cost_volume"], d["single_frame_cvs"]


def top2_margin(cv):
    t = torch.topk(cv, 2, dim=1)[0]
    return (t[:, 0] - t[:, 1])


def write_small(path, ref_mod, configs):
    """Full reference cost-volume tensors for small seeded synthetic configs {tag: (B, F, D, H, W, seed)}."""
    small = {}
    for tag, (B, nF, D, H, W, seed) in configs.items():
        d = make_inputs(B, nF, H, W, seed=seed)
        cv, sf = run_ref_cv(ref_mod, d, steps=D)
        small[f"{tag}_cfg"] = np.array([B, nF, D, H, W, seed])
        small[f"{tag}_cv"] = cv.numpy()
        small[f"{tag}_sf"] = np.stack([v.numpy() for v in sf])
        small[f"{tag}_key_u8"] = np.round((d["keyframe"].numpy() + 0.5) * 255).astype(np.uint8)
        small[f"{tag}_frames_u8"] = np.round((torch.stack(d["frames"]).numpy() + 0.5) * 255).astype(np.uint8)
        small[f"{tag}_poses"] = torch.stack(d["poses"]).numpy()
        small[f"{tag}_K"] = d["keyframe_intrinsics"].numpy()
    np.savez_compressed(path, **small)


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    ref_mod = import_reference()
    if "--only-kitti-model" in sys.argv:
        # the north-star sentence literally: full MonoRecModel on the bundled example sample (256x512, 2 source frames);
        # no pretrained weights exist offline, so seeded weights (two gains) as in model_synth_small.npz
        s = load_kitti_sample()
        out = {}
        for gain_tag, gain in (("g1", 1.0), ("g07", 0.7)):
            model = ref_mod.MonoRecModel()
            model.load_state_dict(seeded_state_dict(model, seed=7, gain=gain))
            model.eval()
            with torch.no_grad():
                r = model(sample_to_dict(s))
            out[f"{gain_tag}_cv_mask"] = r["cv_mask"].numpy().astype(np.float16)        # values in (0,1): 5e-4 quantisation
            out[f"{gain_tag}_result"] = r["result"].numpy()                             # fp32: the gated quantity
            for i, p in enumerate(r["predicted_inverse_depths"][1:], start=1):
                out[f"{gain_tag}_depth{i}"] = p.numpy()
            print(gain_tag, "result range", float(r["result"].min()), float(r["result"].max()),
                  "mask range", float(r["cv_mask"].min()), float(r["cv_mask"].max()))
        out["wseed"] = np.array([7])
        np.savez_compressed(HERE / "model_kitti_sample.npz", **out)
        return
    if "--only-model-fp64" in sys.argv:
        # The reference's OWN fp32 rounding noise on the gated quantities: the same model and inputs evaluated in float64.
        # |result32 - result64| is what any fp32 implementation can be told apart from another by; the GPU tests gate the
        # drop-in at max(1e-3, 4 x that) (tests/test_convnet_gpu.py).  Written to a separate small file.
        to64 = lambda d: {k: ([t.double() for t in v] if isinstance(v, list) else v.double()) for k, v in d.items()}
        out = {}
        s = load_kitti_sample()
        for cfg, data in (("kitti", sample_to_dict(s)), ("synth", make_inputs(1, 2, 64, 128, seed=5))):
            for gain_tag, gain in (("g1", 1.0), ("g07", 0.7)):
                model = ref_mod.MonoRecModel()
                model.load_state_dict(seeded_state_dict(model, seed=7, gain=gain))
                model.eval()
                with torch.no_grad():
                    r32 = model(dict(data))
                    torch.set_default_dtype(torch.float64)      # the reference creates its grids / patch kernel with the default dtype
                    model64 = ref_mod.MonoRecModel()
                    model64.load_state_dict({k: (v.double() if v.is_floating_point() else v) for k, v in model.state_dict().items()})
                    r64 = model64.eval()(to64(data))
                    torch.set_default_dtype(torch.float32)
                d_res = (r32["result"].double() - r64["result"]).abs().max().item()
                d_mask = (r32["cv_mask"].double() - r64["cv_mask"]).abs().max().item()
                d_heads = [(a.double() - b).abs().max().item() for a, b in zip(r32["predicted_inverse_depths"], r64["predicted_inverse_depths"])]
                out[f"{cfg}_{gain_tag}_noise"] = np.array([d_res, d_mask] + d_heads)
                out[f"{cfg}_{gain_tag}_result64"] = r64["result"].float().numpy()
                out[f"{cfg}_{gain_tag}_cv_mask64"] = r64["cv_mask"].float().numpy().astype(np.float16)
                print(cfg, gain_tag, "reference fp32 vs fp64: result", d_res, "mask", d_mask, "heads", d_heads, flush=True)
        np.savez_compressed(HERE / "model_fp64.npz", **out)
        return
    if "--only-config2" in sys.argv:
        # BASELINE config 2's geometry at full size (256x512, 32 planes, 4 source frames, one keyframe of the synthetic
        # KITTI-shaped generator bench.py uses): sub-sampled volumes, rows, full arg-max / validity maps and per-plane
        # checksums, like kitti_sample.npz
        d = make_inputs(1, 4, 256, 512, seed=100)
        cv, sf = run_ref_cv(ref_mod, d)
        sub = (slice(None), slice(None), slice(2, None, 4), slice(1, None, 8))
        np.savez_compressed(
            HERE / "cv_config2.npz", cfg=np.array([1, 4, 32, 256, 512, 100]),
            cv_sub=cv[sub].numpy(), sf_sub=np.stack([v[sub].numpy() for v in sf]),
            cv_rows=cv[:, :, 100:104].numpy(), sf_rows=np.stack([v[:, :, 100:104].numpy() for v in sf]),
            argmax=cv.argmax(1).numpy().astype(np.uint8), margin=top2_margin(cv).numpy().astype(np.float16),
            cv_zero=np.packbits((cv == 0).all(1).numpy()),
            sf_zero=np.packbits(np.stack([(v == 0).all(1).numpy() for v in sf])),
            cv_plane_sum=cv.double().sum((2, 3)).numpy(), sf_plane_sum=np.stack([v.double().sum((2, 3)).numpy() for v in sf]))
        print("config 2 golden: valid share per frame", [float(1 - (v == 0).all(1).float().mean()) for v in sf])
        return
    if "--only-metrics" in sys.argv:
        # the reference's own sparse metric functions (model/metric_functions/sparse_metrics.py) on small seeded inputs:
        # inverse-depth predictions, LiDAR-like sparse targets (~8 % of the pixels), a moving-object mask
        sys.path.insert(0, str(REF))
        sys.modules.setdefault("kornia.geometry.camera", types.ModuleType("kornia.geometry.camera"))
        import model.metric_functions.sparse_metrics as SM  # noqa
        g = torch.Generator().manual_seed(11)
        B, H, W = 3, 48, 80
        pred = torch.rand(B, 1, H, W, generator=g) * 0.3 + 0.002
        pred[torch.rand(B, 1, H, W, generator=g) < 0.02] = 0.0                      # predictions that are exactly 0
        gt = (pred * (1 + 0.25 * torch.randn(B, 1, H, W, generator=g))).clamp_min(1e-3)
        gt[torch.rand(B, 1, H, W, generator=g) > 0.08] = 0.0                        # sparse
        mv = (torch.rand(B, 1, H, W, generator=g) > 0.6).float()
        out = {"pred": pred.numpy(), "gt": gt.numpy(), "mvobj": mv.numpy()}
        names = ("a1", "a2", "a3", "rmse", "rmse_log", "abs_rel", "sq_rel")
        cases = {"plain": dict(), "roi_md": dict(roi=[4, 44, 8, 72], max_distance=80.0),
                 "onlyvalid": dict(roi=None, max_distance=50.0, pred_all_valid=False),
                 "onlydynamic": dict(roi=None, max_distance=80.0, use_cvmask=True)}   # (the reference does not crop mvobj_mask: roi must be None)
        for tag, kw in cases.items():
            vals = []
            for n in names:
                d = {"result": pred.clone(), "target": gt.clone(), "mvobj_mask": mv.clone()}
                vals.append(float(getattr(SM, f"{n}_sparse_metric")(d, **kw)))
            out[f"case_{tag}"] = np.array(vals, dtype=np.float64)
            print(tag, dict(zip(names, vals)))
        np.savez_compressed(HERE / "metrics.npz", **out)
        return
    if "--only-pointcloud" in sys.argv:
        # the unmodified PLYSaver (utils/ply_utils.py) + the mask lines of create_pointcloud.py:77-78, :93-95 on seeded inputs
        import torch.nn.functional as F
        sys.path.insert(0, str(REF))
        from utils.ply_utils import PLYSaver  # noqa
        g = torch.Generator().manual_seed(23)
        B, H, W, NW = 2, 40, 64, 5
        inv_depth = torch.rand(B, 1, H, W, generator=g) * 0.3 + 0.002
        image = torch.rand(B, 3, H, W, generator=g) - 0.5
        K = torch.eye(4).repeat(B, 1, 1)
        K[:, 0, 0] = 61.0; K[:, 1, 1] = 60.0; K[:, 0, 2] = 31.0; K[:, 1, 2] = 19.5
        ang = torch.tensor([0.05, -0.08])
        pose = torch.eye(4).repeat(B, 1, 1)
        pose[:, 0, 0] = ang.cos(); pose[:, 0, 2] = ang.sin(); pose[:, 2, 0] = -ang.sin(); pose[:, 2, 2] = ang.cos()
        pose[:, :3, 3] = torch.tensor([[1.0, -0.2, 12.0], [3.0, 0.1, 14.5]])
        cv_masks = [torch.rand(B, 1, H, W, generator=g) * 0.09 for _ in range(NW)]          # below the 0.1 threshold ...
        cv_masks[0][0, 0, 3, 5] = 0.5; cv_masks[2][1, 0, 30, 50] = 0.11; cv_masks[4][0, 0, 39, 63] = 0.1   # ... except three hits
        keeps = []
        for m in cv_masks:                                                                   # create_pointcloud.py:77-78
            mask = (m >= .1).to(dtype=torch.float32)
            keeps.append((F.conv2d(mask, mask.new_ones((1, 1, 33, 33)), padding=16) < 1).to(dtype=torch.float32))
        voted = (torch.sum(torch.stack(keeps), dim=0) > NW - 1).to(dtype=torch.float32)       # :93
        out = {"inv_depth": inv_depth.numpy(), "image": image.numpy(), "K": K.numpy(), "pose": pose.numpy(),
               "cv_masks": torch.stack(cv_masks).numpy(), "keeps": torch.stack(keeps).numpy()}
        for tag, roi, use_vote in (("plain", None, False), ("roi_vote", [4, 36, 6, 60], True)):
            saver = PLYSaver(H, W, min_d=3, max_d=30, batch_size=B, roi=roi, dropout=0)
            depth = inv_depth.clone()
            if use_vote:
                depth *= voted                                                               # :95
            saver.add_depthmap(depth, image.clone(), K.clone(), pose.clone())
            v = np.array(saver.data, dtype=np.float32).reshape(-1, 6)
            out[f"vertices_{tag}"] = v
            print(tag, v.shape, "kept share", v.shape[0] / (B * H * W))
        np.savez_compressed(HERE / "pointcloud.npz", **out)
        return
    if "--only-reprojection" in sys.argv:
        # the unmodified reprojection_loss (model/loss_functions/common_losses.py:16-114) with the argument sets the reference's
        # losses use (monorec_loss.py:185-188, :355, :361), reduce=False, and torch autograd of sum(weights * errors) w.r.t.
        # the predicted inverse depth
        sys.path.insert(0, str(REF))
        from model.loss_functions.common_losses import reprojection_loss, compute_errors  # noqa
        from tests.helpers import REPROJ_CFG, reprojection_inputs  # noqa
        d, invd, wts = reprojection_inputs()
        out = {"cfg": np.array(REPROJ_CFG), "invd": invd.numpy(), "weights": wts.numpy()}
        cases = {"plain": dict(use_mono=True, use_stereo=False, automasking=False),
                 "auto": dict(use_mono=True, use_stereo=True, automasking=True),
                 "stereo_border": dict(use_mono=False, use_stereo=True, automasking=False, border=3)}
        for tag, kw in cases.items():
            pred = invd.clone().requires_grad_(True)
            err = reprojection_loss(pred, {k: (list(v) if isinstance(v, list) else v) for k, v in d.items()},
                                    error_function=compute_errors, reduce=False, combine_frames="min", mono_auto=False, **kw)
            inf = torch.isinf(err)
            (torch.where(inf, torch.zeros_like(err), err) * wts).sum().backward()
            red = reprojection_loss(invd.clone(), {k: (list(v) if isinstance(v, list) else v) for k, v in d.items()},
                                    error_function=compute_errors, reduce=True, combine_frames="min", mono_auto=False, **kw)
            out[f"errors_{tag}"] = err.detach().numpy()
            out[f"grad_{tag}"] = pred.grad.numpy()
            out[f"reduced_{tag}"] = np.array(float(red))
            print(tag, "inf share", float(inf.float().mean()), "mean finite error", float(err[~inf].mean()),
                  "max |grad|", float(pred.grad.abs().max()), "reduced", float(red))
        np.savez_compressed(HERE / "reprojection.npz", **out)
        return
    if "--only-integration" in sys.argv:
        # INTEGRATION.md section 2 on the reference side: evaluate.py:29-31 builds its models with
        # ConfigParser.initialize_list("models", model.model) from the config's "models" block.  The checkpoint path is
        # dropped (no checkpoint offline); the parser is created without its run directories and logging set-up.
        import inspect
        import json
        import model.model as module_arch  # noqa
        from utils.parse_config import ConfigParser  # noqa
        cfg = json.loads((REF / "configs" / "evaluate" / "eval_monorec.json").read_text())
        models = [dict(m, args={k: v for k, v in m["args"].items() if k != "checkpoint_location"}) for m in cfg["models"]]
        parser = ConfigParser.__new__(ConfigParser)
        parser._config = {"models": models}
        keywords = [n for n in inspect.signature(ref_mod.MonoRecModel.__init__).parameters if n != "self"]
        settings = []
        for m in parser.initialize_list("models", module_arch):
            vals = {n: getattr(m, n) for n in keywords if hasattr(m, n)}
            settings.append({n: (list(v) if isinstance(v, tuple) else v) for n, v in vals.items()
                             if isinstance(v, (bool, int, float, str, list, tuple, type(None)))})
        out = {"config": "configs/evaluate/eval_monorec.json", "models": models, "reference_init_keywords": keywords,
               "reference_settings": settings}
        (HERE / "integration.json").write_text(json.dumps(out, indent=1) + "\n")
        print(json.dumps(settings))
        return
    if "--only-d64f6" in sys.argv:
        # BASELINE config 5's plane and frame counts (64 planes, 6 source frames) at a small size; added after the other
        # files, which are left untouched
        write_small(HERE / "cv_synth_d64f6.npz", ref_mod, {"d": (1, 6, 64, 40, 72, 4)})
        return

    # ---- 1. bundled KITTI sample --------------------------------------------------------------
    s = load_kitti_sample()
    data = sample_to_dict(s)
    cv, sf = run_ref_cv(ref_mod, data)
    # the same reference in float64 (for the tie-margin rule of SURVEY.md §8c)
    data64 = {k: ([t.double() for t in v] if isinstance(v, list) else v.double()) for k, v in data.items()}
    torch.set_default_dtype(torch.float64)
    cv64, sf64 = run_ref_cv(ref_mod, data64)
    torch.set_default_dtype(torch.float32)
    print("kitti sample: fp32 vs fp64 reference max|d| =", float((cv.double() - cv64).abs().max()),
          "argmax agree =", float((cv.argmax(1) == cv64.argmax(1)).float().mean()))
    sub = (slice(None), slice(None), slice(2, None, 4), slice(1, None, 8))
    np.savez_compressed(
        HERE / "kitti_sample.npz",
        keyframe_u8=s["keyframe_u8"], frames_u8=s["frames_u8"], K=s["K"], keyframe_pose=s["keyframe_pose"],
        poses=s["poses"],
        cv_sub=cv[sub].numpy(), sf_sub=np.stack([v[sub].numpy() for v in sf]),
        cv_rows=cv[:, :, 100:104].numpy(), sf_rows=np.stack([v[:, :, 100:104].numpy() for v in sf]),
        argmax=cv.argmax(1).numpy().astype(np.uint8),
        margin=top2_margin(cv).numpy().astype(np.float16),
        margin64=top2_margin(cv64).numpy().astype(np.float16),
        argmax64=cv64.argmax(1).numpy().astype(np.uint8),
        cv_zero=np.packbits((cv == 0).all(1).numpy()),
        sf_zero=np.packbits(np.stack([(v == 0).all(1).numpy() for v in sf])),
        cv_plane_sum=cv.double().sum((2, 3)).numpy(), sf_plane_sum=np.stack([v.double().sum((2, 3)).numpy() for v in sf]),
        cv_plane_sqsum=(cv.double() ** 2).sum((2, 3)).numpy(),
    )

    # ---- 2. small synthetic cost volumes (full tensors) ---------------------------------------
    small = {}
    for tag, (B, nF, D, H, W, seed) in {"a": (2, 2, 32, 32, 64, 1), "b": (1, 3, 16, 40, 72, 2),
                                        "c": (1, 4, 32, 48, 64, 3)}.items():
        d = make_inputs(B, nF, H, W, seed=seed)
        cv, sf = run_ref_cv(ref_mod, d, steps=D)
        small[f"{tag}_cfg"] = np.array([B, nF, D, H, W, seed])
        small[f"{tag}_cv"] = cv.numpy()
        small[f"{tag}_sf"] = np.stack([v.numpy() for v in sf])
        small[f"{tag}_key_u8"] = np.round((d["keyframe"].numpy() + 0.5) * 255).astype(np.uint8)
        small[f"{tag}_frames_u8"] = np.round((torch.stack(d["frames"]).numpy() + 0.5) * 255).astype(np.uint8)
        small[f"{tag}_poses"] = torch.stack(d["poses"]).numpy()
        small[f"{tag}_K"] = d["keyframe_intrinsics"].numpy()
    np.savez_compressed(HERE / "cv_synth_small.npz", **small)

    # ---- 3. full model on a small synthetic config --------------------------------------------
    out = {}
    B, nF, H, W, seed = 1, 2, 64, 128, 5
    for gain_tag, gain in (("g1", 1.0), ("g07", 0.7)):
        model = ref_mod.MonoRecModel()
        model.load_state_dict(seeded_state_dict(model, seed=7, gain=gain))
        model.eval()
        d = make_inputs(B, nF, H, W, seed=seed)
        with torch.no_grad():
            r = model(d)
        out[f"{gain_tag}_cv_mask"] = r["cv_mask"].numpy()
        for i, p in enumerate(r["predicted_inverse_depths"]):
            out[f"{gain_tag}_depth{i}"] = p.numpy()
        for i, p in enumerate(r["image_features"]):
            out[f"{gain_tag}_feat{i}_sum"] = np.array([p.double().sum().item(), p.double().abs().sum().item()])
        out[f"{gain_tag}_cost_volume_masked_sum"] = np.array([r["cost_volume"].double().sum().item()])
        q = torch.tensor([0.01, 0.25, 0.5, 0.75, 0.99])
        print(gain_tag, "result q", torch.quantile(r["result"].flatten(), q), "mask q", torch.quantile(r["cv_mask"].flatten(), q))
        print(gain_tag, "result range", float(r["result"].min()), float(r["result"].max()),
              "mask range", float(r["cv_mask"].min()), float(r["cv_mask"].max()))
    out["cfg"] = np.array([B, nF, 32, H, W, seed, 7])
    # the checkpoint contract: every key and shape of the reference model's state_dict (SURVEY.md §8b)
    ref_sd = ref_mod.MonoRecModel().state_dict()
    out["state_keys"] = np.array(list(ref_sd.keys()))
    out["state_shapes"] = np.array([",".join(str(int(v)) for v in t.shape) for t in ref_sd.values()])
    np.savez_compressed(HERE / "model_synth_small.npz", **out)
    for f in sorted(HERE.glob("*.npz")):
        print(f.name, f.stat().st_size // 1024, "KiB")


if __name__ == "__main__":
    main()
