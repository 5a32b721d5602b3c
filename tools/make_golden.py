"""Generate tests/golden/*.npz by running the REAL reference code (loaded by path, oracle/refload.py).

Only runs where /root/reference exists.  The fixtures pin the oracle restatements on machines without the
reference (tests/test_oracle_golden.py).  Inputs are seeded; outputs are the reference's own return values.
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from megapose6d_b200 import procedural  # noqa: E402
from oracle import refload, resnet_ref  # noqa: E402
from tests import helpers  # noqa: E402

OUT = ROOT / "tests" / "golden"


def lib3d_inputs():
    g = torch.Generator().manual_seed(123)
    n = 6
    TCO = torch.from_numpy(procedural.random_poses(n, 42)).float()
    K = torch.from_numpy(procedural.example_camera()).float().unsqueeze(0).repeat(n, 1, 1)
    pts = torch.randn(n, 256, 3, generator=g) * 0.05
    p9 = torch.randn(n, 9, generator=g)
    p9[:, 8] = 1 + 0.1 * p9[:, 8]
    bb = torch.tensor([[384.0, 234, 522, 455]]).repeat(n, 1) + 5 * torch.randn(n, 4, generator=g)
    Tn = TCO + 0.01 * torch.randn(n, 4, 4, generator=g)
    return dict(TCO=TCO, K=K, pts=pts, p9=p9, bb=bb, Tn=Tn)


def main():
    ref = refload.load()
    OUT.mkdir(parents=True, exist_ok=True)
    i = lib3d_inputs()
    uv = ref.camera_geometry.project_points_robust(i["pts"], i["K"], i["TCO"])
    boxes = ref.camera_geometry.boxes_from_uv(uv)
    Kc = ref.camera_geometry.get_K_crop_resize(i["K"].clone(), boxes, (480, 640), (240, 320))
    R6 = ref.rotations.compute_rotation_matrix_from_ortho6d(i["p9"][:, :6])
    tCR = i["TCO"][:, :3, 3] + 0.01
    upd = ref.cosypose_ops.pose_update_with_reference_point(i["TCO"], Kc, i["p9"][:, 6:], R6, tCR)
    init = ref.cosypose_ops.TCO_init_from_boxes_autodepth_with_R(i["bb"], i["pts"], i["K"], R6)
    center = ref.camera_geometry.project_points_robust(torch.zeros(6, 1, 3), i["K"], i["TCO"])
    dboxes = ref.cropping.deepim_boxes(center, boxes, boxes, lamb=1.4, im_size=(480, 640))
    np.savez(OUT / "lib3d.npz", **{k: v.numpy() for k, v in i.items()}, uv=uv.numpy(), boxes=boxes.numpy(), K_crop=Kc.numpy(),
             R6=R6.numpy(), normT=ref.transform_ops.normalize_T(i["Tn"]).numpy(), update=upd.numpy(), init=init.numpy(),
             deepim_boxes=dboxes.numpy(), sample_ids=np.random.RandomState(0).choice(5002, 2000, replace=False)[:64])

    # crop (roi_align incl. depth masking) on a small synthetic RGB-D frame
    rng = np.random.RandomState(7)
    img = torch.from_numpy(rng.rand(1, 4, 60, 80).astype(np.float32))
    img[:, 3, ::5, ::3] = 0
    b5 = torch.tensor([[0, 10.3, 5.2, 60.7, 44.1], [0, -6.0, -4.0, 30.0, 20.0], [0, 50.0, 30.0, 95.0, 70.0]])
    crops = ref.cropping.crop_images(img, b5, output_size=(12, 16), sampling_ratio=4)
    np.savez(OUT / "crop.npz", img=img.numpy(), boxes5=b5.numpy(), crops=crops.numpy())

    # backbone + head on a small input (coarse 9 channels / refiner 27 channels)
    for name, cfg in (("coarse", helpers.COARSE_CFG), ("refiner", helpers.REFINER_CFG)):
        sd = helpers.make_state_dict(cfg, seed=11)
        c = helpers.n_inputs(cfg)
        net = ref.torchvision_resnet.resnet34(num_classes=512, n_input_channels=c)
        net.load_state_dict({k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")})
        net.eval()
        x = torch.rand(2, c, 64, 96, generator=torch.Generator().manual_seed(3))
        head = resnet_ref.head_name(sd)
        with torch.no_grad():
            y = torch.nn.functional.linear(net(x), sd[head + ".weight"], sd[head + ".bias"])
        np.savez(OUT / f"resnet_{name}.npz", y=y.numpy())
    pipeline_fixture(ref)
    print("wrote", sorted(p.name for p in OUT.glob("*.npz")))


def pipeline_fixture(ref):
    """The reference's own PoseEstimator.run_inference_pipeline on tests/helpers.pipeline_scenario() (fp32, CPU).  Only the
    renderer is not the reference's: Panda3D is absent, the C rasteriser of oracle/raster_ref.c stands in (SURVEY 8c)."""
    from tests.test_oracle_vs_reference import _reference_predictor

    sc = helpers.pipeline_scenario()
    meshes = helpers.ref_meshes_from_dataset(sc["ds"])
    coarse = _reference_predictor(ref, helpers.COARSE_CFG, sc["sd_coarse"], meshes)
    refiner = _reference_predictor(ref, helpers.REFINER_CFG, sc["sd_refiner"], meshes)
    coarse.cfg = refiner.cfg = None
    with refload.cpu_cuda_patch():
        est = ref.pose_estimator.PoseEstimator(refiner_model=refiner, coarse_model=coarse, bsz_objects=2, bsz_images=64,
                                               SO3_grid_size=sc["grid"])
        detections = ref.tensor_collection.PandasTensorCollection(sc["det_df"].copy(), bboxes=sc["bboxes"])
        obs = ref.types.ObservationTensor(sc["images"], sc["K"])
        final, extra = est.run_inference_pipeline(obs, detections=detections, n_refiner_iterations=sc["n_refiner_iterations"],
                                                  n_pose_hypotheses=sc["n_pose_hypotheses"])
    c = extra["coarse"]["preds"]
    f = extra["coarse_filter"]["preds"].infos
    n_det = len(sc["labels"])
    assert c.infos["bbox_id"].tolist() == sorted(c.infos["bbox_id"].tolist()), "rows are detection-major"
    kept = np.stack([np.sort(f[f["bbox_id"] == d]["hypothesis_id"].values) for d in range(n_det)])
    scored = extra["scoring"]["preds"]
    np.savez(OUT / "pipeline.npz", coarse_poses=c.poses.numpy(), coarse_logit=c.infos["coarse_logit"].values.astype(np.float32),
             coarse_hypothesis=c.infos["hypothesis_id"].values.astype(np.int64), kept_hypotheses=kept.astype(np.int64),
             scored_label=np.array(scored.infos["label"].tolist(), dtype="U"), scored_hypothesis=scored.infos["hypothesis_id"].values.astype(np.int64),
             scored_pose_logit=scored.infos["pose_logit"].values.astype(np.float32), scored_poses=scored.poses.numpy(),
             final_label=np.array(final.infos["label"].tolist(), dtype="U"), final_hypothesis=final.infos["hypothesis_id"].values.astype(np.int64),
             final_poses=final.poses.numpy(), final_pose_logit=final.infos["pose_logit"].values.astype(np.float32))


def fullsize_fixture(ref, name: str):
    """The reference's own PoseEstimator.run_inference_pipeline (fp32, CPU, C rasteriser standing in for Panda3D) on one of
    the full-size scenarios of workloads/scenes.py (BASELINE configs[1..3]) -> tests/golden/<name>.npz: every coarse logit,
    the survivors, the refiner's pose after every iteration, the scoring logits and the final poses."""
    import os
    import time

    from tests.test_oracle_vs_reference import _reference_predictor
    from workloads import scenes, weights

    sc = scenes.FULLSIZE[name]()
    meshes = helpers.ref_meshes_from_dataset(sc["ds"])
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    rgb = sc["images"][:, :3].contiguous()
    coarse = _reference_predictor(ref, weights.COARSE_CFG, sc["sd_coarse"], meshes, sc["render_size"], threads)
    refiner = _reference_predictor(ref, sc["cfg_refiner"], sc["sd_refiner"], meshes, sc["render_size"], threads)
    coarse.cfg = refiner.cfg = None
    t0 = time.time()
    with refload.cpu_cuda_patch():
        est = ref.pose_estimator.PoseEstimator(refiner_model=refiner, coarse_model=coarse, bsz_objects=8, bsz_images=128,
                                               SO3_grid_size=sc["grid"])
        detections = ref.tensor_collection.PandasTensorCollection(sc["det_df"].copy(), bboxes=sc["bboxes"])
        obs = ref.types.ObservationTensor(sc["images"], sc["K"])
        if sc["cfg_refiner"]["input_depth"]:
            # the zoo pairs an RGB coarse model with the RGB-D refiner (utils/load_model.py:18-26); the reference's coarse
            # model slices the RGB channels itself (models/pose_rigid.py:660-664 via input_rgb_dims)
            pass
        final, extra = est.run_inference_pipeline(obs, detections=detections, n_refiner_iterations=sc["n_refiner_iterations"],
                                                  n_pose_hypotheses=sc["n_pose_hypotheses"], keep_all_refiner_outputs=False)
    c = extra["coarse"]["preds"]
    f = extra["coarse_filter"]["preds"]
    n_det = len(sc["labels"])
    assert c.infos["bbox_id"].tolist() == sorted(c.infos["bbox_id"].tolist()), "rows are detection-major"
    preds = extra["refiner_all_hypotheses"]["preds"]
    iters = np.stack([preds[f"iteration={n + 1}"].poses.numpy() for n in range(sc["n_refiner_iterations"])])
    scored = extra["scoring"]["preds"]
    np.savez_compressed(
        OUT / f"{name}.npz", coarse_logit=c.infos["coarse_logit"].values.astype(np.float32),
        coarse_bbox_id=c.infos["bbox_id"].values.astype(np.int32), coarse_hypothesis=c.infos["hypothesis_id"].values.astype(np.int32),
        kept_bbox_id=f.infos["bbox_id"].values.astype(np.int32), kept_hypothesis=f.infos["hypothesis_id"].values.astype(np.int32),
        kept_poses=f.poses.numpy(), refiner_poses=iters,
        scored_label=np.array(scored.infos["label"].tolist(), dtype="U"), scored_hypothesis=scored.infos["hypothesis_id"].values.astype(np.int32),
        scored_pose_logit=scored.infos["pose_logit"].values.astype(np.float32),
        final_label=np.array(final.infos["label"].tolist(), dtype="U"), final_hypothesis=final.infos["hypothesis_id"].values.astype(np.int32),
        final_poses=final.poses.numpy(), final_pose_logit=final.infos["pose_logit"].values.astype(np.float32),
        grid=sc["grid"], n_refiner_iterations=sc["n_refiner_iterations"], render_size=np.asarray(sc["render_size"]),
        seconds_on_host=time.time() - t0, host_threads=threads)
    print(f"{name}: {n_det} detections x {sc['grid']} hypotheses, {time.time() - t0:.1f} s on {threads} threads", flush=True)


REFERENCE_TEST_MODULES = ("test_oracle_vs_reference", "test_product_vs_reference", "test_prediction_runner", "test_detector")


def reference_test_fixtures(ref, modules=REFERENCE_TEST_MODULES):
    """tests/golden/<module without test_>.npz: what the reference returned on the inputs of each module's comparisons
    with the reference (computed by the module's own `reference_outputs(ref)`)."""
    import importlib

    for name in modules:
        arrays = importlib.import_module(f"tests.{name}").reference_outputs(ref)
        path = OUT / f"{name[len('test_'):]}.npz"
        np.savez_compressed(path, **arrays)
        print(f"{path.name}: {len(arrays)} arrays, {path.stat().st_size} bytes", flush=True)


if __name__ == "__main__":
    if sys.argv[1:2] == ["tests"]:  # python tools/make_golden.py tests [test_module ...]
        reference_test_fixtures(refload.load(), sys.argv[2:] or REFERENCE_TEST_MODULES)
    elif len(sys.argv) > 1:  # python tools/make_golden.py fullsize_rgb fullsize_rgb_224 ...
        _ref = refload.load()
        for _name in sys.argv[1:]:
            fullsize_fixture(_ref, _name)
    else:
        main()
