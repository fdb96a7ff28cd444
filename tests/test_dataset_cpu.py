"""CPU: the reference's dataset folder contract (scene/dataset_mono.py) read by gaussianavatar_b200.dataset.  Pinned against the
reference's OWN dataset classes run on the same synthetic folder, through the items oracle/gen_golden.py stored from those classes:
tests/golden/dataset_items.npz (first and last item of the stage-2 datasets) and tests/golden/dataset_items_stage1.npz (every item of
the stage-1 datasets)."""
import os

import numpy as np
import torch

from dataset_fixture import write_synthetic_dataset

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dataset_items.npz")
GOLD_STAGE1 = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dataset_items_stage1.npz")
FIELDS = ("original_image", "world_view_transform", "projection_matrix", "full_proj_transform", "camera_center")


def _item_arrays(item):
    out = {k: np.asarray(item[k], dtype=np.float64) for k in FIELDS if k in item}
    out["scalars"] = np.array([item["FovX"], item["FovY"], item["width"], item["height"], item["pose_idx"]], dtype=np.float64)
    for k in ("pose_data", "transl_data", "inp_pos_map"):
        if k in item:
            out[k] = np.asarray(item[k], dtype=np.float64)
    return out


def _ours(tmp_path, stage2=False):
    """no_mask=1: the reference's masked branch (dataset_mono.py:214 hands PIL an int8 array) does not run under this image's Pillow, so
    the comparison against the reference's classes covers images / cameras / poses / position maps; the mask arithmetic is pinned
    against its two-line formula in test_mask_compositing_formula."""
    from gaussianavatar_b200 import dataset as ds
    mp = write_synthetic_dataset(str(tmp_path), stage2=stage2)
    mp.no_mask = 1
    return mp, dict(train=ds.MonoDataset_train(mp), test=ds.MonoDataset_test(mp), novel_pose=ds.MonoDataset_novel_pose(mp))


def test_items_match_golden_from_reference_classes(tmp_path):
    mp, sets = _ours(tmp_path, stage2=True)
    gold = np.load(GOLD)
    for name, dset in sets.items():
        assert len(dset) == int(gold[f"{name}/len"])
        for i in (0, len(dset) - 1):
            for k, v in _item_arrays(dset[i]).items():
                np.testing.assert_allclose(v, gold[f"{name}/{i}/{k}"], rtol=0, atol=1e-7, err_msg=f"{name}[{i}].{k}")


def test_items_match_reference_classes_directly(tmp_path):
    """Every item of the stage-1 datasets, field for field, against what the reference's classes returned for the same folder."""
    mp, sets = _ours(tmp_path)
    gold = np.load(GOLD_STAGE1)
    for name, dset in sets.items():
        assert len(dset) == int(gold[f"{name}/len"])
        for i in range(len(dset)):
            a = _item_arrays(dset[i])
            pfx = f"{name}/{i}/"
            assert set(a) == {k[len(pfx):] for k in gold.files if k.startswith(pfx)}
            for k in a:
                np.testing.assert_allclose(a[k], gold[pfx + k], rtol=0, atol=1e-7, err_msg=f"{name}[{i}].{k}")


def test_device_decode_is_bit_identical_to_host_compositing(tmp_path):
    from gaussianavatar_b200 import dataset as ds
    mp = write_synthetic_dataset(str(tmp_path))
    host, raw = ds.MonoDataset_train(mp), ds.MonoDataset_train(mp, device_decode=True)
    imgs = torch.stack([raw[i]["image_u8"] for i in range(3)]); masks = torch.stack([raw[i]["mask_u8"] for i in range(3)])
    out = ds.composite_on_device(imgs, masks)            # runs on whatever device the tensors live on
    for i in range(3):
        assert torch.equal(out[i], host[i]["original_image"])


def test_mask_compositing_formula(tmp_path):
    """dataset_mono.py:207-217: mask < 128 -> 0, >= 128 -> 1; colour = image * mask + (1 - mask) * 255; then / 255 and clamp."""
    from PIL import Image
    from gaussianavatar_b200 import dataset as ds
    mp = write_synthetic_dataset(str(tmp_path))
    d = ds.MonoDataset_train(mp)
    for i in range(len(d)):
        name = d.name_list[i][1]
        img = np.array(Image.open(os.path.join(d.data_folder, "images", name + ".png")))
        mask = np.array(Image.open(os.path.join(d.data_folder, "masks", name + ".png")))[..., None].copy()
        mask[mask < 128] = 0
        mask[mask >= 128] = 1
        ref = torch.from_numpy((img * mask + (1 - mask) * 255).astype(np.uint8)) / 255.0
        assert torch.equal(d[i]["original_image"], ref.permute(2, 0, 1).clamp(0.0, 1.0))
    assert (d[0]["original_image"] == 1.0).any() and (d[0]["original_image"] < 1.0).any()


def test_novel_view_orbit_keeps_the_camera_distance(tmp_path):
    from gaussianavatar_b200 import dataset as ds
    mp = write_synthetic_dataset(str(tmp_path))
    nv = ds.MonoDataset_novel_view(mp)
    nv.update_smpl(1, 8, pelvis_pos=np.array([0.0, -0.2, 0.0]))
    assert len(nv) == 8
    c0 = nv[0]["camera_center"].double().numpy()
    for i in range(8):
        it = nv[i]
        d = np.linalg.norm(it["camera_center"].double().numpy() - nv.Th)
        assert abs(d - np.linalg.norm(c0 - nv.Th)) < 1e-4
        assert it["pose_idx"] == 1 and it["pose_data"].shape == (72,)
    assert np.allclose(nv[0]["world_view_transform"].numpy(), ds.camera_item(nv.intrinsic, nv.extr_npy, 64, 64)["world_view_transform"].numpy(), atol=1e-6)
