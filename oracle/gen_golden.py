"""ORACLE — TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by importing the UNMODIFIED reference modules from
/root/reference (read-only, never copied).  Run in the build container only (the GPU box has no /root/reference):

    python oracle/gen_golden.py

Each fixture stores the reference's OUTPUTS (and small inputs); large inputs are regenerated from seeds by
oracle.avatar_oracle.seeded_pop_params / gaussianavatar_b200.synthetic so the fixtures stay small.
"""
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
OUT = os.path.join(ROOT, "tests", "golden")

from model.network import POP_no_unet                     # noqa: E402  (reference)
from submodules.smplx.lbs import lbs                      # noqa: E402  (reference)
from utils.general_utils import getIdxMap_torch           # noqa: E402  (reference)
from utils.graphics_utils import focal2fov, getProjectionMatrix, getWorld2View2   # noqa: E402  (reference)
from utils.loss_utils import l1_loss_w, ssim              # noqa: E402  (reference)

from gaussianavatar_b200 import synthetic as syn          # noqa: E402
from oracle.avatar_oracle import seeded_pop_params, seeded_unet_params        # noqa: E402


def gen_test_pose_subset():
    s = torch.load(os.path.join(REF, "assets/test_pose/smpl_parms.pth"))
    c = np.load(os.path.join(REF, "assets/test_pose/cam_parms.npz"))
    idx = np.arange(0, 480, 15)                          # 32 of the 480 shipped poses
    np.savez_compressed(os.path.join(OUT, "test_pose_subset.npz"), beta=s["beta"].numpy(), body_pose=s["body_pose"].numpy()[idx],
                        trans=s["trans"].numpy()[idx], frame_index=idx, intrinsic=c["intrinsic"], extrinsic=c["extrinsic"])


def _reference_dataset_items(stage2, every_item):
    """Items of the reference's own dataset classes (scene/dataset_mono.py) on the synthetic folder tests/dataset_fixture.py writes:
    the first and last item of each dataset, or every item."""
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from dataset_fixture import write_synthetic_dataset
    from scene import dataset_mono as ref
    _orig = ref.getProjectionMatrix      # numpy-1.x semantics of the reference env (python float / np.float32 -> float64 scalar): see gen_camera
    ref.getProjectionMatrix = lambda **kw: _orig(**{**kw, "K": np.asarray(kw["K"]).astype(np.float64)})
    fields = ("original_image", "world_view_transform", "projection_matrix", "full_proj_transform", "camera_center")
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        mp = write_synthetic_dataset(tmp, stage2=stage2)
        mp.no_mask = 1      # the reference's masked branch (dataset_mono.py:214) feeds an int8 array to PIL, which the Pillow of this image rejects
        sets = dict(train=ref.MonoDataset_train(mp, device="cpu"), test=ref.MonoDataset_test(mp, device="cpu"),
                    novel_pose=ref.MonoDataset_novel_pose(mp, device="cpu"))
        for name, dset in sets.items():
            out[f"{name}/len"] = np.array(len(dset))
            for i in (range(len(dset)) if every_item else (0, len(dset) - 1)):
                item = dset[i]
                for k in fields:
                    if k in item:
                        out[f"{name}/{i}/{k}"] = np.asarray(item[k], dtype=np.float32)
                out[f"{name}/{i}/scalars"] = np.array([item["FovX"], item["FovY"], item["width"], item["height"], item["pose_idx"]], dtype=np.float64)
                for k in ("pose_data", "transl_data", "inp_pos_map"):
                    if k in item:
                        out[f"{name}/{i}/{k}"] = np.asarray(item[k], dtype=np.float32)
    return out


def gen_dataset_items():
    np.savez_compressed(os.path.join(OUT, "dataset_items.npz"), **_reference_dataset_items(stage2=True, every_item=False))


def gen_dataset_items_stage1():
    """Every item of the stage-1 datasets (no input position maps)."""
    np.savez_compressed(os.path.join(OUT, "dataset_items_stage1.npz"), **_reference_dataset_items(stage2=False, every_item=True))


def gen_smpl_A():
    body = syn.make_body(0)
    d = np.load(os.path.join(OUT, "test_pose_subset.npz"))
    pose = torch.tensor(d["body_pose"][:16]); transl = torch.tensor(d["trans"][:16])
    pose = torch.cat([pose, torch.zeros(1, 72)], 0); transl = torch.cat([transl, torch.zeros(1, 3)], 0)   # + T-pose
    B = pose.shape[0]
    _, _, A = lbs(body.betas.expand(B, -1), pose, body.v_template[None].expand(B, -1, -1).contiguous(), body.shapedirs,
                  body.posedirs, body.J_regressor, body.parents, body.lbs_weights, return_affine_mat=True)
    A = A.clone()
    A[:, :, :3, 3] += transl.unsqueeze(dim=1)            # submodules/smplx/body_models.py:380-383
    np.savez_compressed(os.path.join(OUT, "smpl_A.npz"), pose=pose.numpy(), transl=transl.numpy(), A=A.numpy(),
                        rest_joints=body.rest_joints().numpy(), body_seed=0)


def _pop_case(name, inp, S, B, seed, hsize=128, c_geom=64, pose=False):
    torch.manual_seed(0)
    net = POP_no_unet(c_geom=c_geom, geom_layer_type="conv", nf=32, hsize=hsize, up_mode="upconv", use_dropout=False, uv_feat_dim=2)
    p = seeded_pop_params(seed, c_geom, hsize)
    missing = net.load_state_dict(p, strict=False)
    assert not missing.unexpected_keys
    assert all("running" in k or "num_batches" in k for k in missing.missing_keys), missing.missing_keys
    net.train()                                          # the reference scripts never call .eval() (SURVEY §3.2)
    g = torch.Generator().manual_seed(seed + 1)
    geo = (torch.randn(1, c_geom, inp, inp, generator=g) * 0.01).requires_grad_(True)
    uv = getIdxMap_torch(torch.rand(3, S, S))            # utils/general_utils.py:188
    # stage 2 (model/avatar_model.py:401-405): a per-frame pose feature map is added to the geometry features
    pf = (torch.randn(B, c_geom, inp, inp, generator=g) * 0.05).requires_grad_(True) if pose else None
    res, sc, shs = net.forward(pose_featmap=pf, geom_featmap=geo.expand(B, -1, -1, -1).contiguous(),
                               uv_loc=uv[None].expand(B, -1, -1).contiguous())
    gr, gs, gc = (torch.randn(res.shape, generator=g), torch.randn(sc.shape, generator=g), torch.randn(shs.shape, generator=g))
    loss = (res * gr).sum() + (sc * gs).sum() + (shs * gc).sum()
    loss.backward()
    grads = {k: v.grad.numpy() for k, v in net.named_parameters()}
    keep = ["decoder.conv1.weight", "decoder.conv1.bias", "decoder.bn1.weight", "decoder.bn1.bias", "decoder.conv5.weight",
            "decoder.bn5.weight", "decoder.conv8.weight", "decoder.conv8.bias", "decoder.conv8N.weight", "decoder.conv7SH.weight",
            "decoder.bn7SH.bias", "decoder.conv6N.bias", "geom_proc_layers.conv1.weight", "geom_proc_layers.conv3.weight"]
    out = dict(res=res.detach().numpy(), scales=sc.detach().numpy(), shs=shs.detach().numpy(), uv=uv.numpy(),
               geo_grad_sub=geo.grad.numpy()[:, ::4, ::max(1, inp // 8), ::max(1, inp // 8)].copy(),
               geo_grad_norm=float(geo.grad.norm()), bn1_running_mean=net.decoder.bn1.running_mean.numpy(),
               bn1_running_var=net.decoder.bn1.running_var.numpy(), inp=inp, S=S, B=B, seed=seed, hsize=hsize, c_geom=c_geom)
    if pose:
        out["pose_featmap"] = pf.detach().numpy()
        out["pose_grad"] = pf.grad.numpy()
    for k in keep:
        out["grad:" + k] = grads[k][:8, :8].copy() if k.startswith("geom_proc") else grads[k]
    out["grad_norms"] = np.array([np.linalg.norm(grads[k]) for k in sorted(grads)])
    out["grad_names"] = np.array(sorted(grads))
    np.savez_compressed(os.path.join(OUT, name), **out)


def gen_pop():
    _pop_case("pop_s32_in16.npz", inp=16, S=32, B=2, seed=5)          # resample 16 -> 32, batch-identical inputs
    _pop_case("pop_s32_in32.npz", inp=32, S=32, B=1, seed=6)          # feat_res == uv_res: resample skipped (network.py:65)
    _pop_case("pop_s48_in128.npz", inp=128, S=48, B=1, seed=7)        # the real 128^2 input map, down-sampling case
    _pop_case("pop_s32_in16_pose.npz", inp=16, S=32, B=2, seed=8, pose=True)   # stage 2: per-frame pose_featmap, BatchNorm over both frames


def gen_losses():
    g = torch.Generator().manual_seed(9)
    a = torch.rand(2, 3, 40, 52, generator=g).requires_grad_(True)
    b = torch.rand(2, 3, 40, 52, generator=g)
    l1 = l1_loss_w(a, b)
    s = ssim(a, b)
    (0.8 * l1 + 0.2 * (1 - s)).backward()
    np.savez_compressed(os.path.join(OUT, "losses.npz"), img=a.detach().numpy(), gt=b.numpy(), l1=l1.item(), ssim=s.item(),
                        grad=a.grad.numpy())


def gen_camera():
    c = np.load(os.path.join(REF, "assets/test_pose/cam_parms.npz"))
    out = {}
    for side in (1024, 512):
        K = np.array(c["intrinsic"], np.float32).reshape(3, 3).copy()
        sc = side / 1024.0
        K[0, 0] *= sc; K[1, 1] *= sc; K[0, 2] *= sc; K[1, 2] *= sc
        extr = c["extrinsic"]
        R = np.array(extr[:3, :3], np.float32).reshape(3, 3).transpose(1, 0)     # scene/dataset_mono.py:165-166
        T = np.array([extr[:3, 3]], np.float32)
        FovY, FovX = focal2fov(K[1, 1], side), focal2fov(K[0, 0], side)
        wvt = torch.tensor(getWorld2View2(R, T, np.array([0.0, 0.0, 0.0]), 1.0)).transpose(0, 1)
        # numpy-1.x semantics of the reference env: python-float / np.float32 -> float64 scalar (assignable into a tensor)
        proj = getProjectionMatrix(znear=0.01, zfar=100.0, fovX=FovX, fovY=FovY, K=K.astype(np.float64), h=side, w=side).transpose(0, 1)
        full = (wvt.unsqueeze(0).bmm(proj.unsqueeze(0))).squeeze(0)
        out[f"wvt{side}"] = wvt.numpy(); out[f"full{side}"] = full.numpy(); out[f"center{side}"] = wvt.inverse()[3, :3].numpy()
        out[f"fov{side}"] = np.array([FovX, FovY])
    np.savez_compressed(os.path.join(OUT, "camera.npz"), **out)


def gen_param_order():
    """Parameter order of the reference's `net.parameters()` (what torch.optim.Adam's state indices refer to in a reference
    checkpoint, model/avatar_model.py:148-155,163-176): pins gaussianavatar_b200.network.REFERENCE_PARAM_ORDER."""
    import json
    net = POP_no_unet(c_geom=64, geom_layer_type="conv", nf=64, hsize=128, up_mode="upconv", use_dropout=False, uv_feat_dim=2)
    order = [[n, list(p.shape)] for n, p in net.named_parameters()]
    with open(os.path.join(OUT, "pop_param_order.json"), "w") as f:
        json.dump(order, f, indent=0)
    print("pop_param_order.json", len(order))


def gen_unet():
    """Stage-2 pose encoder: the reference's UnetNoCond5DS (model/modules.py:185-232) in training mode on a seeded input, with
    seeded parameters (oracle.avatar_oracle.seeded_unet_params): output, input gradient and two weight gradients."""
    from model.modules import UnetNoCond5DS                # reference
    nf, cin, cout, side, B, seed = 8, 3, 8, 32, 2, 11
    net = UnetNoCond5DS(input_nc=cin, output_nc=cout, nf=nf, up_mode="upconv", use_dropout=False)
    missing, unexpected = net.load_state_dict(seeded_unet_params(seed, cin, cout, nf), strict=False)
    assert not unexpected and all("running" in k or "num_batches" in k for k in missing), (missing, unexpected)
    net.train()
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, cin, side, side, generator=g).requires_grad_(True)
    gout = torch.randn(B, cout, side, side, generator=g)
    y = net(x.clone() if False else x)
    (y * gout).sum().backward()
    grads = dict(net.named_parameters())
    np.savez_compressed(os.path.join(OUT, "unet5ds_nf8_s32.npz"), nf=nf, cin=cin, cout=cout, side=side, B=B, seed=seed,
                        y=y.detach().numpy(), dx=x.grad.numpy(), d_conv3=grads["conv3.conv.weight"].grad.numpy(),
                        d_upconv4=grads["upconv4.up.weight"].grad.numpy(), d_bias=grads["upconv5.up.bias"].grad.numpy(),
                        bn2_running_mean=net.conv2.bn.running_mean.numpy())


def gen_unet_full_size():
    """The reference's UnetNoCond5DS at the size GaussianAvatar instantiates it (input_nc=3, output_nc=64, nf=32, 128 x 128 position
    maps, model/avatar_model.py:139-146): sub-sampled output / gradients keep the fixture small."""
    from model.modules import UnetNoCond5DS                # reference
    nf, cin, cout, side, B, seed = 32, 3, 64, 128, 2, 12
    net = UnetNoCond5DS(input_nc=cin, output_nc=cout, nf=nf, up_mode="upconv", use_dropout=False)
    missing, unexpected = net.load_state_dict(seeded_unet_params(seed, cin, cout, nf), strict=False)
    assert not unexpected and all("running" in k or "num_batches" in k for k in missing), (missing, unexpected)
    net.train()
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, cin, side, side, generator=g).requires_grad_(True)
    gout = torch.randn(B, cout, side, side, generator=g)
    y = net(x)
    (y * gout).sum().backward()
    grads = dict(net.named_parameters())
    np.savez_compressed(os.path.join(OUT, "unet5ds_nf32_s128.npz"), nf=nf, cin=cin, cout=cout, side=side, B=B, seed=seed,
                        y_sub=y.detach().numpy()[:, :, ::8, ::8], y_norm=float(y.detach().norm()), dx_sub=x.grad.numpy()[:, :, ::4, ::4],
                        dx_norm=float(x.grad.norm()), d_conv3_sub=grads["conv3.conv.weight"].grad.numpy()[:16, :16],
                        d_upconv4_sub=grads["upconv4.up.weight"].grad.numpy()[:16, :16], d_bias=grads["upconv5.up.bias"].grad.numpy(),
                        grad_norms=np.array([float(grads[k].grad.norm()) for k in sorted(grads)]), grad_names=np.array(sorted(grads)),
                        bn2_running_mean=net.conv2.bn.running_mean.numpy())


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    gen_test_pose_subset()
    gen_smpl_A()
    gen_pop()
    gen_losses()
    gen_camera()
    gen_param_order()
    gen_unet()
    gen_unet_full_size()
    gen_dataset_items()
    gen_dataset_items_stage1()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
