"""Detector front-end (SURVEY 8 f4): the product's Detector against what the reference's own class
(src/megapose/inference/detector.py:34-142) returned when fed by the same stand-in network (tests/golden/detector.npz,
written by `reference_outputs(ref)` through tools/make_golden.py); load_detector round trip."""
import importlib.util
import sys
import types
from pathlib import Path

import numpy as np
import pytest
import torch

from megapose6d_b200 import detector as D
from megapose6d_b200.load_model import Cfg
from megapose6d_b200.types import ObservationTensor
from tests import helpers

GOLDEN = Path(__file__).resolve().parent / "golden" / "detector.npz"


class FakeMaskRCNN(torch.nn.Module):
    """torchvision-format outputs, deterministic per image: a list of dicts(boxes, labels, scores, masks[n,1,H,W])."""

    def __init__(self, counts, seed=0):
        super().__init__()
        self.config = types.SimpleNamespace(label_to_category_id={"ycbv-obj_000001": 1, "ycbv-obj_000002": 2, "ycbv-obj_000005": 3})
        self.counts, self.seed = counts, seed

    def forward(self, images):
        g = torch.Generator().manual_seed(self.seed)
        out = []
        for img, n in zip(images, self.counts):
            h, w = img.shape[-2:]
            xy = torch.rand(n, 2, generator=g) * torch.tensor([w / 2, h / 2])
            wh = torch.rand(n, 2, generator=g) * torch.tensor([w / 2, h / 2]) + 1
            out.append(dict(boxes=torch.cat([xy, xy + wh], 1), labels=torch.randint(1, 4, (n,), generator=g),
                            scores=torch.rand(n, generator=g), masks=torch.rand(n, 1, h, w, generator=g)))
        return out


def _reference_detector_cls(ref):
    from oracle import refload

    name = "megapose.inference.detector"
    if name not in sys.modules:
        sys.modules.setdefault("megapose.utils", types.ModuleType("megapose.utils")).tensor_collection = ref.tensor_collection
        spec = importlib.util.spec_from_file_location(name, refload.REF_ROOT / "inference/detector.py")
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    return sys.modules[name].Detector


def _same(a, b):
    da, db = a.infos.reset_index(drop=True), b.infos.reset_index(drop=True)
    # the pandas of this image drops the grouping columns inside the reference's groupby().apply() (add_instance_id,
    # inference/utils.py:166-169; the reference's pinned pandas keeps them): compare the columns the reference still has
    assert set(db.columns) <= set(da.columns) and {"batch_im_id", "label", "score", "instance_id"} == set(da.columns)
    assert len(da) == len(db)
    for c in db.columns:
        if c == "score":
            assert np.array_equal(da[c].to_numpy(dtype=np.float64), db[c].to_numpy(dtype=np.float64))
        else:
            assert list(da[c]) == list(db[c]), c
    assert torch.equal(a.bboxes.cpu(), b.bboxes.cpu()) and a.bboxes.dtype == b.bboxes.dtype
    ta, tb = set(a._tensors.keys()), set(b._tensors.keys())
    assert ta == tb
    if "masks" in ta:
        assert torch.equal(a.masks.cpu(), b.masks.cpu())


COUNTS = [(3, 0, 5), (1,), (4, 4)]
KWS = [dict(), dict(detection_th=0.4), dict(output_masks=True, mask_th=0.6),
       dict(one_instance_per_class=True, detection_th=0.1, output_masks=True)]


def _detector_inputs(counts):
    return torch.rand(len(counts), 3, 24, 32), torch.eye(3).repeat(len(counts), 1, 1)


def _rgb():
    return (np.random.RandomState(0).rand(24, 32, 3) * 255).astype(np.uint8)


@pytest.fixture(scope="module")
def want():
    return np.load(GOLDEN)


@pytest.mark.parametrize("counts", COUNTS)
@pytest.mark.parametrize("kw", KWS)
def test_detector_matches_reference_class(want, counts, kw):
    images, K = _detector_inputs(counts)
    mine = D.Detector(FakeMaskRCNN(counts))
    got = mine.get_detections(ObservationTensor(images, K), **kw)
    _same(got, helpers.restore_collection(want, f"{COUNTS.index(counts)}/{KWS.index(kw)}"))
    assert helpers.tensor_digest(mine.image_tensor_from_numpy(_rgb())) == str(want["image_tensor"])


def reference_outputs(ref) -> dict:
    """What the reference's Detector returns on the inputs of test_detector_matches_reference_class (tools/make_golden.py)."""
    from oracle import refload

    RefDetector = _reference_detector_cls(ref)
    out = {}
    for i, counts in enumerate(COUNTS):
        for j, kw in enumerate(KWS):
            images, K = _detector_inputs(counts)
            with refload.cpu_cuda_patch():
                a = RefDetector(FakeMaskRCNN(counts)).get_detections(ref.types.ObservationTensor(images, K), **kw)
            helpers.record_collection(out, f"{i}/{j}", a)
    out["image_tensor"] = np.array(helpers.tensor_digest(RefDetector(FakeMaskRCNN((1,))).image_tensor_from_numpy(_rgb())))
    return out


def test_detector_without_detections():
    det = D.Detector(FakeMaskRCNN((0, 0)))
    out = det(ObservationTensor(torch.rand(2, 3, 24, 32), torch.eye(3).repeat(2, 1, 1)), output_masks=True, detection_th=0.5)
    assert len(out) == 0 and out.bboxes.shape == (0, 4) and out.masks.shape == (0, 24, 32)
    assert {"score", "label", "batch_im_id", "instance_id"} <= set(out.infos.columns)


def test_load_detector_round_trip(tmp_path):
    pytest.importorskip("torchvision")
    import yaml

    cfg = Cfg(input_resize=(48, 64), backbone_str="resnet50-fpn", anchor_sizes=[[32], [64], [128], [256], [512]],
              train_ds_names=[["ycbv.pbr", 1]], label_to_category_id={"obj_000001": 1, "obj_000002": 2})
    model = D.create_model_detector(cfg, n_classes=len(cfg.label_to_category_id))  # as inference/utils.py:62
    run = tmp_path / "detector-test"
    run.mkdir()
    (run / "config.yaml").write_text(yaml.safe_dump(dict(cfg)))
    torch.save({"state_dict": model.state_dict()}, run / "checkpoint.pth.tar")
    det = D.load_detector("detector-test", models_root=tmp_path, device="cpu")
    assert det.category_id_to_label == {1: "ycbv-obj_000001", 2: "ycbv-obj_000002"}
    out = det(ObservationTensor(torch.rand(1, 3, 48, 64), torch.eye(3)[None]), output_masks=True)
    assert out.bboxes.shape[1] == 4 and "instance_id" in out.infos.columns
    sd = det.model.state_dict()
    assert all(torch.equal(v, sd[k]) for k, v in model.state_dict().items())


class _BoxModel(torch.nn.Module):
    """Stand-in network that 'detects' given boxes (torchvision output format) -- the Mask R-CNN itself is a library model."""

    def __init__(self, labels, bboxes):
        super().__init__()
        self.config = types.SimpleNamespace(label_to_category_id={l: i + 1 for i, l in enumerate(labels)})
        self.bboxes = bboxes

    def forward(self, images):
        n = len(self.bboxes)
        h, w = images[0].shape[-2:]
        return [dict(boxes=self.bboxes.to(images[0].device), labels=torch.arange(1, n + 1, device=images[0].device),
                     scores=torch.linspace(0.9, 0.8, n, device=images[0].device),
                     masks=torch.ones(n, 1, h, w, device=images[0].device))]


@pytest.mark.gpu
def test_pipeline_with_run_detector_equals_passing_the_detections(tmp_path):
    import pandas as pd

    from megapose6d_b200 import load_model, procedural
    from megapose6d_b200.tensor_collection import PandasTensorCollection
    from tests import helpers

    ds, images, K = helpers.make_scene(2, seed=6)
    load_model.write_run(tmp_path, "coarse-rgb-906902141", helpers.make_state_dict(helpers.COARSE_CFG, 5))
    load_model.write_run(tmp_path, "refiner-rgb-653307694", helpers.make_state_dict(helpers.REFINER_CFG, 6))
    est = load_model.load_named_model("megapose-1.0-RGB", ds, models_root=tmp_path)
    est.load_SO3_grid(72)
    labels = [o.label for o in ds.list_objects]
    TCO_gt = torch.from_numpy(procedural.random_poses(2, 11)).float()
    TCO_gt[:, 2, 3] = torch.tensor([0.55, 0.7])
    bboxes = torch.stack([helpers.detection_for_pose(K[0], TCO_gt[i], torch.from_numpy(ds[i].mesh.vertices).float()) for i in range(2)])
    obs = ObservationTensor(images[:, :3].contiguous(), K.clone()).cuda()
    est.detector_model = D.Detector(_BoxModel(labels, bboxes))
    a, extra = est.run_inference_pipeline(obs, run_detector=True, n_refiner_iterations=2)
    det = PandasTensorCollection(pd.DataFrame(dict(label=labels, batch_im_id=0, score=[0.9, 0.8])), bboxes=bboxes.cuda())
    b, _ = est.run_inference_pipeline(obs, detections=det, n_refiner_iterations=2)
    assert list(a.infos["label"]) == list(b.infos["label"]) and torch.equal(a.poses, b.poses)
    assert np.array_equal(a.infos["pose_score"].to_numpy(), b.infos["pose_score"].to_numpy())
