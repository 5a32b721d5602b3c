"""Host-side containers and helpers of the product against the REAL reference classes.

What the reference's classes return on the inputs below is stored in tests/golden/product_vs_reference.npz
(`reference_outputs(ref)`, run by tools/make_golden.py with the reference loaded by path); the tests hold the product to it."""
import json
import pickle
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
import torch

from megapose6d_b200 import pose_estimator as mine_pe
from megapose6d_b200 import tensor_collection as mine_tc
from megapose6d_b200.types import ObservationTensor as MineObs
from tests import helpers

GOLDEN = Path(__file__).resolve().parent / "golden" / "product_vs_reference.npz"


@pytest.fixture(scope="module")
def want():
    return np.load(GOLDEN)


def _frame(n, seed):
    rs = np.random.RandomState(seed)
    return pd.DataFrame(dict(label=[f"obj_{k}" for k in rs.randint(0, 3, n)], batch_im_id=rs.randint(0, 2, n),
                             score=rs.rand(n)), index=rs.permutation(n) + 10)


def _same(a, b):
    assert len(a) == len(b)
    pd.testing.assert_frame_equal(a.infos, b.infos)
    assert list(a.tensors.keys()) == list(b.tensors.keys())
    for k in a.tensors:
        assert torch.equal(a.tensors[k], b.tensors[k]), k


def _collection_steps(tc):
    """The same sequence of operations on a PandasTensorCollection of module `tc` (the reference's or ours): yields
    (name, collection) after each step."""
    n = 9
    g = torch.Generator().manual_seed(0)
    poses, boxes = torch.randn(n, 4, 4, generator=g), torch.randn(n, 4, generator=g)
    a = tc.PandasTensorCollection(infos=_frame(n, 1), poses=poses.clone(), bboxes=boxes.clone())
    yield "new", a                                        # index reset to 0..n-1 on construction
    for k, ids in enumerate(([2, 0, 5], torch.tensor([1, 1, 8]), np.array([3, 4]), [0])):
        yield f"getitem{k}", a[ids]
    extra = pd.DataFrame(dict(label=["obj_0", "obj_1", "obj_2"], diameter=[0.1, 0.2, 0.3]))
    yield "merge_df", a.merge_df(extra, on="label")
    yield "concatenate", tc.concatenate([a[[0, 1]], a[[5]]])
    yield "clone", a.clone()
    a.register_tensor("extra", torch.arange(n))
    a.poses = a.poses * 2
    yield "registered", a
    a.delete_tensor("extra")
    yield "pickled", pickle.loads(pickle.dumps(a))
    yield "double", a.double()


def test_pandas_tensor_collection_behaves_like_the_reference(want):
    for name, b in _collection_steps(mine_tc):
        _same(helpers.restore_collection(want, f"tc/{name}"), b)
        if name == "new":
            assert b.device == torch.device(str(want["tc/device"]))
            with pytest.raises(AttributeError):
                _ = b.not_a_tensor
    assert len(mine_tc.concatenate([])) == int(want["tc/empty_len"]) == 0


def _observation_inputs():
    rs = np.random.RandomState(3)
    rgb = rs.randint(0, 255, size=(12, 16, 3), dtype=np.uint8)
    depth = rs.rand(12, 16).astype(np.float32)
    K = np.array([[500.0, 0, 8], [0, 510, 6], [0, 0, 1]])
    rgb_b = torch.from_numpy(rs.randint(0, 255, size=(2, 3, 12, 16), dtype=np.uint8))
    dep_b = torch.from_numpy(rs.rand(2, 1, 12, 16).astype(np.float32))
    return rgb, depth, K, rgb_b, dep_b, torch.from_numpy(np.stack([K, K])).float()


def test_observation_tensor_behaves_like_the_reference(want):
    rgb, depth, K, rgb_b, dep_b, Kb = _observation_inputs()
    for name, d in (("rgb", None), ("rgbd", depth)):
        b = MineObs.from_numpy(rgb, d, K)
        assert torch.equal(b.images, torch.from_numpy(want[f"obs/{name}/images"])) and torch.equal(b.K, torch.from_numpy(want[f"obs/{name}/K"]))
        assert (b.batch_size, b.channel_dim, b.is_valid()) == tuple(want[f"obs/{name}/{k}"].item() for k in ("batch_size", "channel_dim", "is_valid"))
        if d is not None:
            assert torch.equal(b.depth, torch.from_numpy(want[f"obs/{name}/depth"]))
    b = MineObs.from_torch_batched(rgb_b, dep_b, Kb)
    assert torch.equal(b.images, torch.from_numpy(want["obs/batched/images"])) and torch.equal(b.K, torch.from_numpy(want["obs/batched/K"]))
    assert b.channel_dim == want["obs/batched/channel_dim"].item() == 4
    # [B,H,W] depth: the reference drops the result of `depth.unsqueeze(1)` (inference/types.py:224-229) and raises; the
    # product accepts it as documented there
    assert want["obs/bhw_depth_raises"].item()
    assert torch.equal(MineObs.from_torch_batched(rgb_b, dep_b[:, 0], Kb).images, b.images)


FILTERS = (dict(labels=["obj_0", "obj_2"]), dict(one_instance_per_class=True), dict(labels=["obj_1"], one_instance_per_class=True))


def test_instance_ids_and_detection_filter_match_the_reference(want):
    for seed in range(4):
        n = 11
        boxes = torch.randn(n, 4, generator=torch.Generator().manual_seed(seed))
        b = mine_pe.add_instance_id(mine_tc.PandasTensorCollection(infos=_frame(n, seed), bboxes=boxes.clone()))
        assert b.infos["instance_id"].tolist() == want[f"ids/{seed}/instance_id"].tolist()
        # an existing column is left alone
        assert mine_pe.add_instance_id(b).infos["instance_id"].tolist() == want[f"ids/{seed}/instance_id"].tolist()
        for k, kwargs in enumerate(FILTERS):
            fb = mine_pe.filter_detections(b, **kwargs)
            assert fb.infos["label"].tolist() == want[f"ids/{seed}/filter{k}/label"].tolist()
            assert fb.infos["score"].tolist() == want[f"ids/{seed}/filter{k}/score"].tolist()
            assert torch.equal(fb.bboxes, torch.from_numpy(want[f"ids/{seed}/filter{k}/bboxes"]))


class _AttrDict(dict):
    """OmegaConf-like config for the reference function: attribute access, `in`, `del`, hasattr."""
    __getattr__ = lambda self, k: self[k] if k in self else (_ for _ in ()).throw(AttributeError(k))  # noqa: E731
    __setattr__ = dict.__setitem__
    __delattr__ = dict.__delitem__


def _config_cases():
    from megapose6d_b200 import load_model

    return [
        dict(load_model.ZOO_CONFIGS["coarse-rgb-906902141"]),
        dict(load_model.ZOO_CONFIGS["refiner-rgbd-288182519"]),
        dict(input_strategy="input=obs+one_render", multiview_type="TCO", backbone_str="vanilla_resnet34"),
        dict(multiview_type="front_3views", n_views=4, backbone_str="vanilla_resnet34"),
        dict(multiview_type="front_5views", n_rendered_views=6, render_normals=True, depth_augmentation=True,
             depth_normalization_type="tCR_scale_clamp_center"),
    ]


CONFIG_KEYS = ("is_coarse_compat", "n_rendered_views", "multiview_type", "predict_rendered_views_logits", "remove_TCO_rendering",
               "predict_pose_update", "render_normals", "render_depth", "input_depth", "renderer", "depth_normalization_type")


def test_check_update_config_matches_the_reference(want):
    """training/pose_models_cfg.py:36-87 of the reference (check_update_config, stored results) against
    load_model.check_update_config on legacy and current run configurations."""
    from megapose6d_b200 import load_model

    for case, w in zip(_config_cases(), json.loads(str(want["config/results"]))):
        got = load_model.check_update_config(load_model.Cfg(dict(case)))
        for key in CONFIG_KEYS:
            if key in w:
                assert got[key] == w[key], (case, key, got[key], w[key])
        assert "n_views" not in got


def reference_outputs(ref) -> dict:
    """What the reference's classes return on the inputs of the tests above (tools/make_golden.py -> GOLDEN)."""
    import logging
    import re

    from oracle import refload

    out = {}
    for name, a in _collection_steps(ref.tensor_collection):
        helpers.record_collection(out, f"tc/{name}", a)
        if name == "new":
            out["tc/device"] = np.array(str(a.device))
    out["tc/empty_len"] = np.array(len(ref.tensor_collection.concatenate([])))

    RObs = ref.types.ObservationTensor
    rgb, depth, K, rgb_b, dep_b, Kb = _observation_inputs()
    for name, d in (("rgb", None), ("rgbd", depth)):
        a = RObs.from_numpy(rgb, d, K)
        rec = dict(images=a.images, K=a.K, batch_size=a.batch_size, channel_dim=a.channel_dim, is_valid=a.is_valid())
        if d is not None:
            rec["depth"] = a.depth
        out.update({f"obs/{name}/{k}": np.asarray(v) for k, v in rec.items()})
    a = RObs.from_torch_batched(rgb_b, dep_b, Kb)
    out.update({"obs/batched/images": a.images.numpy(), "obs/batched/K": a.K.numpy(), "obs/batched/channel_dim": np.asarray(a.channel_dim)})
    try:
        RObs.from_torch_batched(rgb_b, dep_b[:, 0], Kb)
        out["obs/bhw_depth_raises"] = np.asarray(False)
    except RuntimeError:
        out["obs/bhw_depth_raises"] = np.asarray(True)

    R, U = ref.tensor_collection, ref.inference_utils
    for seed in range(4):
        n = 11
        boxes = torch.randn(n, 4, generator=torch.Generator().manual_seed(seed))
        a = U.add_instance_id(R.PandasTensorCollection(infos=_frame(n, seed), bboxes=boxes.clone()))
        out[f"ids/{seed}/instance_id"] = a.infos["instance_id"].to_numpy()
        # (with this pandas the reference's groupby().apply() drops the grouping columns from `a.infos`; the product keeps
        # them, as the reference did with the pandas it was written for) -> give the reference filter the complete frame
        infos = _frame(n, seed).reset_index(drop=True)
        infos["instance_id"] = out[f"ids/{seed}/instance_id"]
        a = R.PandasTensorCollection(infos=infos, bboxes=boxes.clone())
        for k, kwargs in enumerate(FILTERS):
            fa = U.filter_detections(a, **kwargs)
            out[f"ids/{seed}/filter{k}/label"] = np.array(fa.infos["label"].tolist(), dtype="U")
            out[f"ids/{seed}/filter{k}/score"] = fa.infos["score"].to_numpy()
            out[f"ids/{seed}/filter{k}/bboxes"] = fa.bboxes.numpy()

    src = (refload.REF_ROOT / "training/pose_models_cfg.py").read_text()
    body = src[src.index("def check_update_config"):src.index("def create_model_pose")]
    body = re.sub(r"\(cfg: TrainingConfig\) -> TrainingConfig", "(cfg)", body)
    ns = dict(logger=logging.getLogger("ref"))
    exec(compile(body, "pose_models_cfg.py", "exec"), ns)
    results = []
    for case in _config_cases():
        w = ns["check_update_config"](_AttrDict(case))
        results.append({k: w[k] for k in CONFIG_KEYS if k in w})
    out["config/results"] = np.array(json.dumps(results))
    return out
