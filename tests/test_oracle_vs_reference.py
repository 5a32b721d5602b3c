"""The oracle restatements must reproduce the REAL reference code.

The reference's outputs on the seeded inputs below are stored in tests/golden/oracle_vs_reference.npz:
`reference_outputs(ref)` computes them from the reference loaded by path (oracle/refload.py) when
tools/make_golden.py regenerates the fixture; the tests compare the oracle with the stored values everywhere.
"""
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import lib3d_ref as L
from oracle import pipeline_ref, resnet_ref
from tests import helpers

GOLDEN = Path(__file__).resolve().parent / "golden" / "oracle_vs_reference.npz"
PREDICTOR_CFGS = dict(coarse=helpers.COARSE_CFG, refiner=helpers.REFINER_CFG, refiner_rgbd=helpers.REFINER_RGBD_CFG)


@pytest.fixture(scope="module")
def want():
    return np.load(GOLDEN)


def _t(a):
    return torch.from_numpy(np.asarray(a))


def _rand_pose(n, seed):
    from megapose6d_b200.procedural import random_poses

    return torch.from_numpy(random_poses(n, seed)).float()


def _lib3d_case():
    g = torch.Generator().manual_seed(0)
    n = 7
    c = dict(TCO=_rand_pose(n, 1), K=torch.from_numpy(helpers.procedural.example_camera()).float().unsqueeze(0).repeat(n, 1, 1))
    c["pts"] = torch.randn(n, 300, 3, generator=g) * 0.05
    c["p9"] = torch.randn(n, 9, generator=g)
    c["Tn"] = c["TCO"] + 0.01 * torch.randn(n, 4, 4, generator=g)
    c["bb"] = torch.tensor([[384.0, 234, 522, 455]]).repeat(n, 1) + torch.arange(n).view(-1, 1)
    c["R"] = L.compute_rotation_matrix_from_ortho6d(torch.randn(n, 6, generator=g))
    c["uv"] = L.project_points_robust(c["pts"], c["K"], c["TCO"])
    c["boxes"] = L.boxes_from_uv(c["uv"])
    c["K_crop"] = L.get_K_crop_resize(c["K"], c["boxes"], (240, 320))
    c["dR"] = L.compute_rotation_matrix_from_ortho6d(c["p9"][:, :6])
    c["tCR"] = c["TCO"][:, :3, 3] + 0.01
    return c


def test_lib3d_functions_match(want):
    c = _lib3d_case()
    TCO, K, pts, p9 = c["TCO"], c["K"], c["pts"], c["p9"]
    assert torch.equal(c["uv"], _t(want["lib3d/uv"]))
    assert torch.equal(c["boxes"], _t(want["lib3d/boxes"]))
    assert torch.equal(c["K_crop"], _t(want["lib3d/K_crop"]))
    assert torch.equal(c["dR"], _t(want["lib3d/R6"]))
    assert torch.equal(L.normalize_T(c["Tn"]), _t(want["lib3d/normT"]))
    assert torch.equal(L.invert_transform_matrices(TCO), _t(want["lib3d/inv"]))
    assert torch.equal(L.pose_update_with_reference_point(TCO, c["K_crop"], p9[:, 6:], c["dR"], c["tCR"]), _t(want["lib3d/update"]))
    assert torch.equal(L.TCO_init_from_boxes_autodepth_with_R(c["bb"], pts, K, c["R"]), _t(want["lib3d/init"]))


def _crops_case():
    ds, images, K = helpers.make_scene(1, seed=3, with_depth=True)
    n = 3
    TCO = _rand_pose(n, 5)
    Kn = K.repeat(n, 1, 1)
    pts = torch.from_numpy(ds[0].mesh.vertices[:2000]).float().unsqueeze(0).repeat(n, 1, 1)
    obs = L.boxes_from_uv(L.project_points_robust(pts, Kn, TCO))
    return dict(imgs=images.repeat(n, 1, 1, 1), obs=obs, Kn=Kn, TCO=TCO, pts=pts)


def test_crops_match(want):
    c = _crops_case()
    b1, c1 = L.deepim_crops_robust(c["imgs"], c["obs"], c["Kn"], c["TCO"], c["TCO"][:, :3, 3], c["pts"], (240, 320))
    assert torch.equal(b1, _t(want["crops/boxes"]))
    helpers.check_sample(want, "crops/crops", c1, atol=0)


def test_sample_and_pad(want):
    pts = torch.arange(5002 * 3, dtype=torch.float32).view(1, 5002, 3)
    ids = L.sample_point_ids(5002, 2000)
    assert torch.equal(pts[:, ids], pts[:, _t(want["sample_ids"]).long()])


def test_so3_asset_matches_reference_file(want):
    from megapose6d_b200.so3 import load_SO3_grid

    for n in (72, 576, 4608):
        grid = load_SO3_grid(n)
        assert grid.shape == (n, 3, 3) and torch.equal(grid[_t(want[f"so3/{n}/rows"]).long()], _t(want[f"so3/{n}/R"]))
        assert np.isclose(grid.double().sum().item(), want[f"so3/{n}/sum"], rtol=0, atol=1e-9)


def _resnet_input(cfg):
    return torch.rand(2, helpers.n_inputs(cfg), 64, 96, generator=torch.Generator().manual_seed(2))


def test_resnet_restatement_matches_reference_module(want):
    for name, cfg in (("coarse", helpers.COARSE_CFG), ("refiner", helpers.REFINER_CFG)):
        sd = helpers.make_state_dict(cfg, seed=1)
        with torch.no_grad():
            got = resnet_ref.forward(sd, _resnet_input(cfg))
        assert torch.allclose(got, _t(want[f"resnet/{name}"]), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("backbone_str,cls", [("resnet34", "WideResNet34"), ("resnet18", "WideResNet18")])
def test_wide_resnet_restatement_matches_reference_module(want, backbone_str, cls):
    """models/wide_resnet.py:59-126 (pre-activation blocks, bare 1x1 downsample, no fc) + the spatial mean of
    PosePredictor.net_forward (models/pose_rigid.py:323-328) + head."""
    sd = resnet_ref.init_state_dict_wide(9, "views_logits_head", 2, seed=5, backbone_str=backbone_str)
    x = torch.rand(2, 9, 64, 96, generator=torch.Generator().manual_seed(2))
    w = _t(want[f"wide/{cls}"])
    with torch.no_grad():
        got = resnet_ref.forward_wide(sd, x)
        emu = resnet_ref.forward_wide_act16_emulated(sd, x)
        bound = resnet_ref.act16_forward_error_bound(sd, x)
    assert torch.allclose(got, w, rtol=1e-5, atol=1e-5)
    assert ((emu - w).abs() <= bound).all()
    from workloads import weights
    sd_w = weights.init_state_dict_wide(9, "views_logits_head", 2, seed=5, backbone_str=backbone_str)
    assert all(torch.equal(sd[k], sd_w[k]) for k in sd)  # the workload generator and the oracle agree on the layout


class _MeshDbAdapter:
    """mesh_db.select(labels).{points, sample_points} as the reference's PosePredictor expects."""

    def __init__(self, meshes, ref):
        self.m, self.ref = meshes, ref

    def select(self, labels):
        pts = self.m.select_points(labels)
        ref = self.ref

        class _Sel:
            points = pts

            @staticmethod
            def sample_points(n, deterministic=False):
                return ref.mesh_ops.sample_points(pts, n, deterministic=deterministic)

        return _Sel()


def _reference_predictor(ref, cfg, sd, meshes, render_size=(240, 320), n_threads=None):
    class Renderer(ref.Panda3dBatchRenderer):
        def __init__(self, inner):
            self.inner = inner

        def render(self, labels, TCO, K, light_datas, resolution, render_depth=False, render_mask=False,
                   render_normals=False):
            d = self.inner.render(labels, TCO, K, None, resolution, render_depth, render_mask, render_normals)
            return type("Out", (), d)

    c = helpers.n_inputs(cfg)
    backbone = ref.torchvision_resnet.resnet34(num_classes=512, n_input_channels=c)
    backbone.n_features = 512
    model = ref.pose_rigid.PosePredictor(
        backbone=backbone, renderer=Renderer(pipeline_ref.RefRenderer(meshes, **({} if n_threads is None else dict(n_threads=n_threads)))),
        mesh_db=_MeshDbAdapter(meshes, ref), render_size=tuple(render_size), n_rendered_views=cfg["n_rendered_views"], multiview_type=cfg["multiview_type"],
        render_normals=True, render_depth=cfg["render_depth"], input_depth=cfg["input_depth"],
        predict_rendered_views_logits=cfg["predict_rendered_views_logits"], remove_TCO_rendering=False,
        predict_pose_update=cfg["predict_pose_update"], depth_normalization_type=cfg["depth_normalization_type"])
    model.load_state_dict(sd)
    return model.eval()


def _predictor_case(cfg_name):
    cfg = PREDICTOR_CFGS[cfg_name]
    ds, images, K = helpers.make_scene(2, seed=4, with_depth=cfg["input_depth"])
    meshes = helpers.ref_meshes_from_dataset(ds)
    return dict(cfg=cfg, meshes=meshes, sd=helpers.make_state_dict(cfg, seed=3), labels=[ds[0].label, ds[1].label],
                TCO=_rand_pose(2, 8), imgs=images.repeat(2, 1, 1, 1), Kn=K.repeat(2, 1, 1))


@pytest.mark.parametrize("cfg_name", ["coarse", "refiner", "refiner_rgbd"])
def test_pose_predictor_matches_reference(want, cfg_name):
    c = _predictor_case(cfg_name)
    cfg, p = c["cfg"], f"predictor/{cfg_name}"
    oracle = pipeline_ref.RefPosePredictor(c["sd"], cfg, c["meshes"], pipeline_ref.RefRenderer(c["meshes"]))
    with torch.no_grad():
        if cfg["predict_pose_update"]:
            # one iteration at a time, each from the reference's own input pose (the refiner loop carries nothing else
            # from one iteration to the next), so that no iteration inherits the previous one's network rounding
            TCO_in = c["TCO"]
            for it in ("iteration=1", "iteration=2"):
                g = oracle.forward(c["imgs"], c["Kn"], c["labels"], TCO_in, n_iterations=1)["iteration=1"]
                q = f"{p}/{it}"
                w_TCO = _t(want[f"{q}/TCO_output"])
                # the pose update on the reference's own network output: fp32 geometry, exact to rounding
                T = L.normalize_T(TCO_in)
                upd = L.update_pose(T, _t(want[f"{q}/K_crop"]), _t(want[f"{q}/network_output"]), T[..., :3, -1])
                assert torch.allclose(upd, w_TCO, rtol=1e-5, atol=1e-6)
                # end to end the pose carries the network output's tolerance: the host's fp32 convolutions round
                # differently from one CPU architecture to another
                assert torch.allclose(g["TCO_output"], w_TCO, rtol=1e-4, atol=1e-5)
                TCO_in = w_TCO
                w_K = _t(want[f"{q}/K_crop"])
                assert torch.equal(g["K_crop"], w_K) or torch.allclose(g["K_crop"], w_K, rtol=1e-6, atol=1e-4)
                assert torch.allclose(g["KV_crop"], _t(want[f"{q}/KV_crop"]), rtol=1e-6, atol=1e-4)
                helpers.check_sample(want, f"{q}/renders", g["renders"], atol=1e-6)
                helpers.check_sample(want, f"{q}/images_crop", g["images_crop"], atol=1e-6)
                assert torch.allclose(g["network_output"], _t(want[f"{q}/network_output"]), rtol=1e-4, atol=1e-5)
        else:
            got = oracle.forward_coarse(c["imgs"], c["Kn"], c["labels"], c["TCO"])
            helpers.check_sample(want, f"{p}/renders", got["renders"], atol=1e-6)
            helpers.check_sample(want, f"{p}/images_crop", got["images_crop"], atol=1e-6)
            assert torch.allclose(got["logits"], _t(want[f"{p}/logits"]), rtol=1e-4, atol=1e-5)


def _pipeline_case():
    ds, images, K = helpers.make_scene(2, seed=6)
    meshes = helpers.ref_meshes_from_dataset(ds)
    sd_c, sd_r = helpers.make_state_dict(helpers.COARSE_CFG, 5), helpers.make_state_dict(helpers.REFINER_CFG, 6)
    labels = [o.label for o in ds.list_objects]
    TCO_gt = _rand_pose(2, 11)
    TCO_gt[:, 2, 3] = torch.tensor([0.55, 0.7])
    bboxes = torch.stack([helpers.detection_for_pose(K[0], TCO_gt[i], torch.from_numpy(ds[i].mesh.vertices).float())
                          for i in range(2)])
    det_df = pd.DataFrame(dict(label=labels, batch_im_id=0, instance_id=np.arange(2)))
    return dict(images=images, K=K, meshes=meshes, sd_c=sd_c, sd_r=sd_r, det_df=det_df, bboxes=bboxes)


def test_pose_estimator_pipeline_matches_reference(want):
    """The reference's own PoseEstimator.run_inference_pipeline vs the oracle pipeline (72-rotation grid)."""
    c = _pipeline_case()
    meshes = c["meshes"]
    oc = pipeline_ref.RefPosePredictor(c["sd_c"], helpers.COARSE_CFG, meshes, pipeline_ref.RefRenderer(meshes))
    orf = pipeline_ref.RefPosePredictor(c["sd_r"], helpers.REFINER_CFG, meshes, pipeline_ref.RefRenderer(meshes))
    oest = pipeline_ref.RefPoseEstimator(oc, orf, bsz_images=64, bsz_objects=2, SO3_grid_size=72)
    got = oest.run_inference_pipeline(c["images"], c["K"], c["det_df"].copy(), c["bboxes"], n_refiner_iterations=2,
                                      n_pose_hypotheses=2)
    assert np.allclose(got["coarse_df"]["coarse_logit"].values, want["pipeline/coarse_logit"], rtol=1e-4, atol=1e-5)
    assert torch.allclose(got["coarse_poses"], _t(want["pipeline/coarse_poses"]), rtol=1e-5, atol=1e-6)
    assert sorted(got["final_df"]["hypothesis_id"].tolist()) == sorted(want["pipeline/final_hypothesis"].tolist())
    order_w = np.argsort(want["pipeline/final_label"])
    order_g = np.argsort(got["final_df"]["label"].values)
    assert torch.allclose(got["final_poses"][order_g], _t(want["pipeline/final_poses"])[order_w], rtol=1e-4, atol=1e-5)


def reference_outputs(ref) -> dict:
    """What the reference returns on the inputs of the tests above (tools/make_golden.py -> GOLDEN)."""
    from oracle import refload

    out = {}
    c = _lib3d_case()
    cg, co = ref.camera_geometry, ref.cosypose_ops
    out["lib3d/uv"] = cg.project_points_robust(c["pts"], c["K"], c["TCO"])
    out["lib3d/boxes"] = cg.boxes_from_uv(c["uv"])
    out["lib3d/K_crop"] = cg.get_K_crop_resize(c["K"].clone(), c["boxes"], (480, 640), (240, 320))
    out["lib3d/R6"] = ref.rotations.compute_rotation_matrix_from_ortho6d(c["p9"][:, :6])
    out["lib3d/normT"] = ref.transform_ops.normalize_T(c["Tn"])
    out["lib3d/inv"] = ref.transform_ops.invert_transform_matrices(c["TCO"])
    out["lib3d/update"] = co.pose_update_with_reference_point(c["TCO"], c["K_crop"], c["p9"][:, 6:], c["dR"], c["tCR"])
    out["lib3d/init"] = co.TCO_init_from_boxes_autodepth_with_R(c["bb"], c["pts"], c["K"], c["R"])

    c = _crops_case()
    boxes, crops = ref.cropping.deepim_crops_robust(images=c["imgs"], obs_boxes=c["obs"], K=c["Kn"], TCO_pred=c["TCO"],
                                                    tCR_in=c["TCO"][:, :3, 3], O_vertices=c["pts"], output_size=(240, 320),
                                                    lamb=1.4)
    out["crops/boxes"] = boxes
    helpers.record_sample(out, "crops/crops", crops)

    pts = torch.arange(5002 * 3, dtype=torch.float32).view(1, 5002, 3)
    out["sample_ids"] = (ref.mesh_ops.sample_points(pts, 2000, deterministic=True)[0, :, 0] / 3).int()
    for n in (72, 576, 4608):  # parsed from the reference's own data_<n>.qua; every row of the smallest grid, a sample of the others
        text = (refload.REF_ROOT / "data" / f"data_{n}.qua").read_text()
        grid = L.unitquat_to_rotmat(torch.tensor([[float(v) for v in line.split()] for line in text.splitlines() if line.strip()]))
        rows = np.arange(n) if n == 72 else np.sort(np.random.RandomState(n).choice(n, 256, replace=False))
        out[f"so3/{n}/rows"], out[f"so3/{n}/R"], out[f"so3/{n}/sum"] = rows, grid[rows], grid.double().sum().item()

    for name, cfg in (("coarse", helpers.COARSE_CFG), ("refiner", helpers.REFINER_CFG)):
        sd = helpers.make_state_dict(cfg, seed=1)
        net = ref.torchvision_resnet.resnet34(num_classes=512, n_input_channels=helpers.n_inputs(cfg))
        net.load_state_dict({k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")})
        net.eval()
        head = resnet_ref.head_name(sd)
        with torch.no_grad():
            out[f"resnet/{name}"] = torch.nn.functional.linear(net(_resnet_input(cfg)), sd[head + ".weight"], sd[head + ".bias"])
    for backbone_str, cls in (("resnet34", "WideResNet34"), ("resnet18", "WideResNet18")):
        sd = resnet_ref.init_state_dict_wide(9, "views_logits_head", 2, seed=5, backbone_str=backbone_str)
        net = getattr(ref.wide_resnet, cls)(n_inputs=9)
        net.load_state_dict({k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")})
        net.eval()
        x = torch.rand(2, 9, 64, 96, generator=torch.Generator().manual_seed(2))
        with torch.no_grad():
            out[f"wide/{cls}"] = torch.nn.functional.linear(net(x).flatten(2).mean(dim=-1), sd["views_logits_head.weight"],
                                                            sd["views_logits_head.bias"])

    for cfg_name in PREDICTOR_CFGS:
        c = _predictor_case(cfg_name)
        cfg, p = c["cfg"], f"predictor/{cfg_name}"
        model = _reference_predictor(ref, cfg, c["sd"], c["meshes"])
        with torch.no_grad():
            if cfg["predict_pose_update"]:
                w = model(images=c["imgs"], K=c["Kn"], labels=c["labels"], TCO=c["TCO"], n_iterations=2)
                for it in ("iteration=1", "iteration=2"):
                    q = f"{p}/{it}"
                    out[f"{q}/TCO_output"], out[f"{q}/K_crop"], out[f"{q}/KV_crop"] = w[it].TCO_output, w[it].K_crop, w[it].KV_crop
                    out[f"{q}/network_output"] = w[it].network_outputs["pose"]
                    helpers.record_sample(out, f"{q}/renders", w[it].renders)
                    helpers.record_sample(out, f"{q}/images_crop", w[it].images_crop)
            else:
                w = model.forward_coarse(images=c["imgs"], K=c["Kn"], labels=c["labels"], TCO_input=c["TCO"],
                                         return_debug_data=True)
                out[f"{p}/logits"] = w["logits"]
                helpers.record_sample(out, f"{p}/renders", w["renders"])
                helpers.record_sample(out, f"{p}/images_crop", w["images_crop"])

    c = _pipeline_case()
    coarse = _reference_predictor(ref, helpers.COARSE_CFG, c["sd_c"], c["meshes"])
    refiner = _reference_predictor(ref, helpers.REFINER_CFG, c["sd_r"], c["meshes"])
    coarse.cfg = refiner.cfg = None
    with refload.cpu_cuda_patch():
        est = ref.pose_estimator.PoseEstimator(refiner_model=refiner, coarse_model=coarse, bsz_objects=2, bsz_images=64,
                                               SO3_grid_size=72)
        detections = ref.tensor_collection.PandasTensorCollection(c["det_df"].copy(), bboxes=c["bboxes"])
        final, extra = est.run_inference_pipeline(ref.types.ObservationTensor(c["images"], c["K"]), detections=detections,
                                                  n_refiner_iterations=2, n_pose_hypotheses=2)
    coarse_preds = extra["coarse"]["preds"]
    out["pipeline/coarse_logit"] = coarse_preds.infos["coarse_logit"].to_numpy()
    out["pipeline/coarse_poses"] = coarse_preds.poses
    out["pipeline/final_hypothesis"] = final.infos["hypothesis_id"].to_numpy()
    out["pipeline/final_label"] = np.array(final.infos["label"].tolist(), dtype="U")
    out["pipeline/final_poses"] = final.poses
    return {k: v.detach().numpy() if isinstance(v, torch.Tensor) else v for k, v in out.items()}
