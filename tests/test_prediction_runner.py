"""Frame-level caller (megapose6d_b200/prediction_runner.py): host logic on the CPU with a stand-in estimator, what the
REAL reference caller returned on the same frames as the checker (tests/golden/prediction_runner.npz, written by
`reference_outputs(ref)` through tools/make_golden.py), and a world_size-2 gloo run of the frame sharding.

The stand-in estimator is a deterministic function of the observation and the detections; it works with the reference's
collections and with ours, so the reference's `PredictionRunner` and ours can be driven by the same object."""
import importlib.util
import json
import os
import pickle
import socket
import sys
import types
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from megapose6d_b200 import prediction_runner as pr
from megapose6d_b200.example import CameraData, ObjectData
from megapose6d_b200.types import InferenceConfig
from tests import helpers


# ------------------------------------------------------------------------------------------------------ fixtures
def make_observations(n_frames=5, h=24, w=32, seed=0, with_init=False):
    rs = np.random.RandomState(seed)
    out = []
    for f in range(n_frames):
        n_obj = 1 + f % 3
        objs = []
        for k in range(n_obj):
            x1, y1 = rs.uniform(0, w / 2), rs.uniform(0, h / 2)
            T = np.eye(4)
            T[:3, 3] = rs.uniform(-0.1, 0.1, 3) + [0, 0, 0.8]
            objs.append(ObjectData(label=f"obj_{(f + k) % 4 + 1:06d}", TWO=T, unique_id=k,
                                   bbox_modal=np.array([x1, y1, x1 + rs.uniform(4, w / 2), y1 + rs.uniform(4, h / 2)]),
                                   visib_fract=float(np.round(rs.uniform(0.5, 1), 3)),
                                   TWO_init=(T @ _shift(0.01 * (k + 1))) if with_init else None))
        TWC = np.eye(4)
        TWC[:3, 3] = rs.uniform(-0.05, 0.05, 3)
        cam = CameraData(K=np.array([[30.0, 0, w / 2], [0, 31.0, h / 2], [0, 0, 1]]), resolution=(h, w), TWC=TWC,
                         TWC_init=TWC if with_init else None)
        out.append(pr.SceneObservation(rgb=rs.randint(0, 256, (h, w, 3)).astype(np.uint8),
                                       depth=rs.uniform(0.3, 1.5, (h, w)).astype(np.float32),
                                       infos=pr.ObservationInfos(scene_id=f // 2 + 1, view_id=f * 7 + 3),
                                       object_datas=objs, camera_data=cam))
    return out


def _shift(dx):
    T = np.eye(4)
    T[0, 3] = dx
    return T


class StandInEstimator:
    """`run_inference_pipeline` with the estimator's signature and return structure; poses are a function of the image, K
    and the boxes, so that a wrong frame / detection pairing or a dropped row shows."""
    sharder = None

    def __init__(self):
        self.calls = []

    def run_inference_pipeline(self, observation, detections=None, run_detector=None, n_refiner_iterations=5,
                               n_pose_hypotheses=1, keep_all_refiner_outputs=False, detection_filter_kwargs=None,
                               run_depth_refiner=False, bsz_images=None, bsz_objects=None, cuda_timer=False,
                               coarse_estimates=None):
        src = detections if coarse_estimates is None else coarse_estimates
        cls = src.__class__
        self.calls.append((tuple(observation.images.shape), len(src), bsz_images, bsz_objects))
        n = len(src)
        infos = src.infos[["label", "batch_im_id"]].copy()
        infos["instance_id"] = infos.groupby(["batch_im_id", "label"]).cumcount().values
        infos["hypothesis_id"] = 0
        key = src.bboxes if "bboxes" in src.tensors else src.poses[:, :3, 3]
        sig = key.double().sum(dim=1) + float(observation.images.double().mean()) + float(observation.K.double().sum())
        infos["pose_score"] = torch.sigmoid(sig / 100).numpy()
        infos["pose_logit"] = (sig / 100).numpy()
        poses = torch.eye(4).repeat(n, 1, 1)
        poses[:, 0, 3] = (sig / 1000).float()
        poses[:, 2, 3] = 0.5 + float(n_refiner_iterations) / 10 + 0.01 * n_pose_hypotheses
        final = cls(infos=infos.copy(), poses=poses.clone())
        refined = cls(infos=infos.copy(), poses=poses.clone() * 1.0)
        coarse_infos = pd.concat([infos.assign(hypothesis_id=h, coarse_logit=float(h)) for h in range(2)]).reset_index(drop=True)
        coarse = cls(infos=coarse_infos, poses=poses.repeat(2, 1, 1))
        extra = dict(coarse=dict(preds=coarse), refiner=dict(preds=refined), time=0.0)
        if run_depth_refiner:
            extra["depth_refiner"] = dict(preds=cls(infos=infos.copy(), poses=poses.clone()))
        return final, extra


CFG = InferenceConfig(detection_type="gt", n_refiner_iterations=3, n_pose_hypotheses=2, bsz_images=64, bsz_objects=4)


def _same_collection(a, b, drop=("time",)):
    ia = a.infos.drop(columns=[c for c in drop if c in a.infos])
    ib = b.infos.drop(columns=[c for c in drop if c in b.infos])
    pd.testing.assert_frame_equal(ia, ib, check_dtype=False)
    assert sorted(a.tensors) == sorted(b.tensors)
    for k in a.tensors:
        assert torch.equal(a.tensors[k], b.tensors[k]), k


# ------------------------------------------------------------------------------------------- the reference's caller
GOLDEN = Path(__file__).resolve().parent / "golden" / "prediction_runner.npz"
SAMPLER_CASES = [(n, world, shuffle, rank) for n in (1, 2, 7, 50, 1000) for world in (1, 2, 3, 8) for shuffle in (True, False)
                 for rank in range(world)]
COLLATE_LABELS = (None, ["obj_000001", "obj_000002", "obj_000003"])
RUNNER_MODES = ("gt", "external", "depth_refiner")


@pytest.fixture(scope="module")
def want():
    return np.load(GOLDEN)


def _runner_cfg(mode):
    return InferenceConfig(**{**CFG.__dict__, **dict(coarse_estimation_type="external" if mode == "external" else "SO3_grid",
                                                     run_depth_refiner=(mode == "depth_refiner"))})


def test_sampler_matches_the_reference(want):
    state = np.random.get_state()[1].copy()
    ends = np.cumsum(want["sampler/lengths"])
    for k, (n, world, shuffle, rank) in enumerate(SAMPLER_CASES):
        b = pr.DistributedSceneSampler(range(n), world, rank, shuffle=shuffle)
        w = want["sampler/indices"][ends[k] - want["sampler/lengths"][k]:ends[k]]
        assert list(b) == w.tolist() and len(b) == len(w)
    assert np.array_equal(state, np.random.get_state()[1])


@pytest.mark.parametrize("with_init", [False, True])
def test_collate_matches_the_reference(want, with_init):
    obs = make_observations(3, with_init=with_init)
    for n_labels, labels in enumerate(COLLATE_LABELS):
        p = f"collate/{with_init}/{n_labels}"
        b = pr.SceneObservation.collate_fn(obs, labels)
        assert sorted(b) == sorted(str(k) for k in want[f"{p}/keys"])
        assert helpers.tensor_digest(b["rgb"]) == str(want[f"{p}/rgb"]) and helpers.tensor_digest(b["depth"]) == str(want[f"{p}/depth"])
        assert json.loads(str(want[f"{p}/im_infos"])) == b["im_infos"]
        assert torch.equal(torch.from_numpy(want[f"{p}/K"]), b["cameras"].K)
        for k in ("gt_detections", "gt_data", "initial_data"):
            if f"{p}/{k}/tensors" not in want:
                assert b[k] is None
            else:
                _same_collection(helpers.restore_collection(want, f"{p}/{k}"), b[k])
                assert b[k].poses.dtype == torch.float32


@pytest.mark.parametrize("mode", RUNNER_MODES)
def test_runner_matches_the_reference_runner(want, mode):
    """Same frames, same stand-in estimator, the reference's PredictionRunner against ours: per-key predictions equal (but
    for our extra `time` column), same frame order, the first frame run twice (warm-up) by both."""
    obs = make_observations(5, with_init=(mode == "external"))
    runner = pr.PredictionRunner(pr.ListSceneDataset(obs, load_depth=True), _runner_cfg(mode), device="cpu")
    est_b = StandInEstimator()
    got = runner.get_predictions(est_b)
    p = f"runner/{mode}"
    assert json.loads(json.dumps([list(c) for c in est_b.calls])) == json.loads(str(want[f"{p}/calls"])) and len(est_b.calls) == len(obs) + 1
    assert set(got) == {str(k) for k in want[f"{p}/keys"]}
    for k in got:
        _same_collection(helpers.restore_collection(want, f"{p}/{k}"), got[k])
        assert "time" in got[k].infos
    assert [(t["scene_id"], t["view_id"]) for t in runner.frame_times] == \
        [(obs[i].infos.scene_id, obs[i].infos.view_id) for i in runner.sampler]


def test_bop_csv_matches_the_toolkit_writer(tmp_path, want):
    """Byte-for-byte against the BOP toolkit's `inout.save_bop_results` as vendored by the reference."""
    pr.save_bop_results(tmp_path / "mine.csv", pr.predictions_to_bop(_predictions(7)))
    assert (tmp_path / "mine.csv").read_bytes() == want["bop_csv"].tobytes()


def _reference_caller(ref):
    """The reference's samplers.py, scene_dataset.py and prediction_runner.py, loaded by path on top of oracle/refload.py.
    Stubbed (absent packages): webdataset, pinocchio's Transform (a numpy 4x4 holder: the runner only reads `.matrix`),
    megapose.utils.random (its two pure-Python helpers are exec'ed from the source), DataLoader workers (n_workers=0)."""
    from oracle import refload

    ns = ref
    ref_root = refload.REF_ROOT
    sys.modules.setdefault("webdataset", types.ModuleType("webdataset"))

    src = (ref_root / "utils/random.py").read_text().splitlines()
    a = next(i for i, l in enumerate(src) if l.startswith("def make_seed"))
    b = next(i for i, l in enumerate(src) if l.startswith("def get_unique_seed"))
    m = types.ModuleType("megapose.utils.random")
    import contextlib

    m.__dict__.update(contextlib=contextlib, np=np)
    exec(compile("\n".join(src[a:b]), str(ref_root / "utils/random.py"), "exec"), m.__dict__)
    sys.modules[m.__name__] = m

    class Transform:
        def __init__(self, matrix):
            self._m = np.asarray(matrix, dtype=np.float64)

        @property
        def matrix(self):
            return self._m

    m = types.ModuleType("megapose.lib3d.transform")
    m.Transform = Transform
    sys.modules[m.__name__] = m
    m = types.ModuleType("megapose.utils.types")
    m.Resolution = tuple
    sys.modules[m.__name__] = m
    d = sys.modules["megapose.utils.distributed"]
    d.get_tmp_dir = lambda: None

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, ref_root / rel)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    stub_scene = sys.modules.get("megapose.datasets.scene_dataset")
    out = types.SimpleNamespace(ns=ns, Transform=Transform)
    out.samplers = load("megapose.datasets.samplers", "datasets/samplers.py")
    out.scene_dataset = load("megapose.datasets.scene_dataset", "datasets/scene_dataset.py")
    sys.modules["megapose"].inference = sys.modules["megapose.inference"]
    sys.modules.setdefault("megapose.evaluation", types.ModuleType("megapose.evaluation"))
    out.prediction_runner = load("megapose.evaluation.prediction_runner", "evaluation/prediction_runner.py")
    if stub_scene is not None:
        out.scene_dataset.Resolution = getattr(stub_scene, "Resolution", tuple)
    return out


def _to_reference_observation(ref_caller, obs):
    S, T = ref_caller.scene_dataset, ref_caller.Transform
    objs = [S.ObjectData(label=o.label, TWO=T(o.TWO), unique_id=o.unique_id, bbox_modal=o.bbox_modal, visib_fract=o.visib_fract,
                         TWO_init=None if o.TWO_init is None else T(o.TWO_init)) for o in obs.object_datas]
    cam = S.CameraData(K=obs.camera_data.K, resolution=obs.camera_data.resolution, TWC=T(obs.camera_data.TWC),
                       TWC_init=None if obs.camera_data.TWC_init is None else T(obs.camera_data.TWC_init))
    return S.SceneObservation(rgb=obs.rgb, depth=obs.depth, infos=S.ObservationInfos(obs.infos.scene_id, obs.infos.view_id),
                              object_datas=objs, camera_data=cam)


def reference_outputs(ref) -> dict:
    """What the reference's caller returns on the inputs of the tests above (tools/make_golden.py -> GOLDEN)."""
    from oracle import refload

    R = _reference_caller(ref)
    out = {}
    state = np.random.get_state()[1].copy()
    lists = []
    for n, world, shuffle, rank in SAMPLER_CASES:
        a = R.samplers.DistributedSceneSampler(range(n), world, rank, shuffle=shuffle)
        assert len(a) == len(list(a))
        lists.append(list(a))
    out["sampler/lengths"] = np.array([len(x) for x in lists], dtype=np.int32)
    out["sampler/indices"] = np.concatenate([np.asarray(x, dtype=np.int32) for x in lists])
    assert np.array_equal(state, np.random.get_state()[1])

    for with_init in (False, True):
        obs = make_observations(3, with_init=with_init)
        for n_labels, labels in enumerate(COLLATE_LABELS):
            p = f"collate/{with_init}/{n_labels}"
            a = R.scene_dataset.SceneObservation.collate_fn([_to_reference_observation(R, o) for o in obs], labels)
            out[f"{p}/keys"] = np.array(sorted(a), dtype="U")
            out[f"{p}/rgb"], out[f"{p}/depth"] = np.array(helpers.tensor_digest(a["rgb"])), np.array(helpers.tensor_digest(a["depth"]))
            out[f"{p}/K"] = a["cameras"].K.numpy()
            out[f"{p}/im_infos"] = np.array(json.dumps(a["im_infos"]))
            for k in ("gt_detections", "gt_data", "initial_data"):
                if a[k] is not None:
                    helpers.record_collection(out, f"{p}/{k}", a[k])

    # device moves of the reference (hard-coded .cuda()) -> identity on the host
    TC, Obs = R.ns.tensor_collection.TensorCollection, R.ns.types.ObservationTensor
    U = sys.modules["megapose.inference.utils"]
    saved = (TC.cuda, Obs.cuda, U.add_instance_id)
    TC.cuda, Obs.cuda = (lambda self: self), (lambda self, *a: self)
    try:
        for mode in RUNNER_MODES:
            obs = make_observations(5, with_init=(mode == "external"))

            class RefDataset(R.scene_dataset.SceneDataset):
                def __init__(self):
                    super().__init__(pd.DataFrame(dict(scene_id=[o.infos.scene_id for o in obs],
                                                       view_id=[o.infos.view_id for o in obs])), load_depth=True)

                def _load_scene_observation(self, infos):
                    o = next(o for o in obs if (o.infos.scene_id, o.infos.view_id) == (infos.scene_id, infos.view_id))
                    return _to_reference_observation(R, o)

            U.add_instance_id = saved[2]
            if mode == "external":
                # the reference helper relies on groupby().apply() keeping the grouping columns (true for the pandas it pins,
                # not for the one used here, see tests/test_product_vs_reference.py): put them back after its own call
                def add_instance_id(inputs, original=saved[2]):
                    before = inputs.infos[["batch_im_id", "label"]].copy()
                    res = original(inputs)
                    for c in before:
                        if c not in res.infos:
                            res.infos[c] = before[c]
                    return res

                U.add_instance_id = add_instance_id
            runner = R.prediction_runner.PredictionRunner(RefDataset(), R.ns.types.InferenceConfig(**_runner_cfg(mode).__dict__),
                                                          batch_size=1, n_workers=0)
            est = StandInEstimator()
            preds = runner.get_predictions(est)
            out[f"runner/{mode}/calls"] = np.array(json.dumps([list(c) for c in est.calls]))
            out[f"runner/{mode}/keys"] = np.array(sorted(preds), dtype="U")
            for k, v in preds.items():
                helpers.record_collection(out, f"runner/{mode}/{k}", v)
    finally:
        TC.cuda, Obs.cuda, U.add_instance_id = saved

    for name in ("imageio", "png"):
        sys.modules.setdefault(name, types.ModuleType(name))
    pkg = types.ModuleType("bop_toolkit_lib")
    pkg.__path__ = []
    pkg.misc = types.ModuleType("bop_toolkit_lib.misc")
    sys.modules.setdefault("bop_toolkit_lib", pkg)
    sys.modules.setdefault("bop_toolkit_lib.misc", pkg.misc)
    spec = importlib.util.spec_from_file_location(
        "bop_toolkit_lib_inout_ref", refload.REF_ROOT.parents[1] / "deps/bop_toolkit_challenge/bop_toolkit_lib/inout.py")
    inout = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(inout)
    import tempfile

    with tempfile.TemporaryDirectory() as tmp:
        inout.save_bop_results(str(Path(tmp) / "ref.csv"), pr.predictions_to_bop(_predictions(7)))
        out["bop_csv"] = np.frombuffer((Path(tmp) / "ref.csv").read_bytes(), dtype=np.uint8)
    return out


# ------------------------------------------------------------------------------------------ no reference needed
def _predictions(n, seed=0):
    from megapose6d_b200.tensor_collection import PandasTensorCollection

    g = torch.Generator().manual_seed(seed)
    poses = torch.eye(4).repeat(n, 1, 1)
    poses[:, :3, :3] = torch.linalg.qr(torch.randn(n, 3, 3, generator=g))[0]
    poses[:, :3, 3] = torch.randn(n, 3, generator=g)
    infos = pd.DataFrame(dict(label=[f"obj_{k % 21 + 1:06d}" for k in range(n)], scene_id=48 + np.arange(n) // 3,
                              view_id=np.arange(n) * 5, pose_score=np.linspace(0.1, 0.9, n), score=1.0,
                              time=np.linspace(0.01, 0.02, n)))
    return PandasTensorCollection(infos=infos, poses=poses)


def test_bop_csv_round_trip(tmp_path):
    preds = _predictions(6)
    results = pr.format_results({"refiner/final": preds})
    torch.save(results, tmp_path / "results.pth.tar")
    out = pr.convert_results_to_bop(tmp_path / "results.pth.tar", tmp_path / "csv" / "out.csv", "refiner/final")
    text = out.read_text()
    assert text.splitlines()[0] == "scene_id,im_id,obj_id,score,R,t,time" and not text.endswith("\n")
    back = pr.load_bop_results(out)
    assert len(back) == 6
    for n, r in enumerate(back):
        row = preds.infos.iloc[n]
        assert (r["scene_id"], r["im_id"], r["obj_id"]) == (row.scene_id, row.view_id, n % 21 + 1)
        assert r["score"] == pytest.approx(row.pose_score) and r["time"] == pytest.approx(row.time)
        assert np.allclose(r["R"], preds.poses[n, :3, :3].numpy(), atol=1e-7)
        assert np.allclose(r["t"][:, 0], preds.poses[n, :3, 3].numpy() * 1e3, rtol=1e-6)      # metres -> millimetres
    by_score = pr.predictions_to_bop(preds, use_pose_score=False)
    assert all(r["score"] == 1.0 for r in by_score)
    with pytest.raises(ValueError):
        (tmp_path / "bad.csv").write_text("scene_id,im_id,obj_id,score,R,t,time\n1,2,3\n")
        pr.load_bop_results(tmp_path / "bad.csv")


def test_sampler_partitions_the_frames():
    state = np.random.get_state()[1].copy()
    for n in (0, 1, 5, 64, 1001):
        for world in (1, 2, 4, 8):
            parts = [list(pr.DistributedSceneSampler(range(n), world, r)) for r in range(world)]
            assert sorted(sum(parts, [])) == list(range(n))
            assert max(map(len, parts)) - min(map(len, parts)) <= 1
            unshuffled = [list(pr.DistributedSceneSampler(range(n), world, r, shuffle=False)) for r in range(world)]
            assert sum(unshuffled, []) == list(range(n))
    assert np.array_equal(state, np.random.get_state()[1])


def test_runner_single_process_and_result_files(tmp_path):
    obs = make_observations(4)
    est = StandInEstimator()
    out = pr.run_predictions(pr.ListSceneDataset(obs, load_depth=True), est, CFG, save_dir=tmp_path / "run", device="cpu")
    preds = out["results"]["predictions"]
    assert set(preds) == {"final", "refiner/iteration=3", "refiner/final", "coarse"}
    n_det = sum(len(o.object_datas) for o in obs)
    assert len(preds["final"]) == n_det and len(preds["coarse"]) == 2 * n_det
    # every prediction row is tagged with its frame and the frame's pipeline time
    frames = {(o.infos.scene_id, o.infos.view_id) for o in obs}
    assert set(zip(preds["final"].infos.scene_id, preds["final"].infos.view_id)) == frames
    assert (preds["final"].infos.time > 0).all()
    assert all(c[0] == (1, 4, 24, 32) and c[2:] == (64, 4) for c in est.calls)          # rgb + depth, batch sizes forwarded
    saved = torch.load(tmp_path / "run" / "results.pth.tar", weights_only=False)
    _same_collection(saved["predictions"]["final"], preds["final"], drop=())
    assert len(pr.load_bop_results(tmp_path / "run" / "bop_refiner_final.csv")) == n_det
    # rgb only
    est2 = StandInEstimator()
    pr.PredictionRunner(pr.ListSceneDataset(obs, load_depth=False), CFG, device="cpu").get_predictions(est2)
    assert all(c[0] == (1, 3, 24, 32) for c in est2.calls)


def test_runner_rejects_bad_configurations():
    obs = make_observations(1)
    ds = pr.ListSceneDataset(obs)
    with pytest.raises(ValueError):
        pr.PredictionRunner(ds, InferenceConfig(detection_type="oracle"), device="cpu").get_predictions(StandInEstimator())
    with pytest.raises(AssertionError):
        pr.PredictionRunner(ds, InferenceConfig(detection_type="gt", coarse_estimation_type="external"),
                            device="cpu").get_predictions(StandInEstimator())
    with pytest.raises(AssertionError):
        pr.PredictionRunner(ds, CFG, batch_size=2, device="cpu")
    with pytest.raises(AssertionError):
        pr.ListSceneDataset(obs + obs)


def test_example_dir_dataset(tmp_path):
    from PIL import Image
    import json

    obs = make_observations(2)
    dirs = []
    for n, o in enumerate(obs):
        d = tmp_path / f"frame{n}"
        (d / "inputs").mkdir(parents=True)
        Image.fromarray(o.rgb).save(d / "image_rgb.png")
        Image.fromarray(np.round(o.depth * 1000).astype(np.uint16)).save(d / "image_depth.png")
        (d / "camera_data.json").write_text(o.camera_data.to_json())
        (d / "inputs" / "object_data.json").write_text(json.dumps([x.to_json() for x in o.object_datas]))
        dirs.append(d)
    ds = pr.ExampleDirSceneDataset(dirs, load_depth=True)
    assert len(ds) == 2
    for n, o in enumerate(obs):
        got = ds[n]
        assert np.array_equal(got.rgb, o.rgb) and np.allclose(got.depth, o.depth, atol=5.1e-4)
        assert (got.infos.scene_id, got.infos.view_id) == (n, 0)
        assert np.allclose(got.camera_data.K, o.camera_data.K) and np.allclose(got.camera_data.TWC, o.camera_data.TWC)
        assert [x.label for x in got.object_datas] == [x.label for x in o.object_datas]
        for x, y in zip(got.object_datas, o.object_datas):
            assert np.allclose(x.bbox_modal, y.bbox_modal) and np.allclose(x.TWO, y.TWO) and x.visib_fract == y.visib_fract
    batch = pr.SceneObservation.collate_fn([ds[0]])
    assert batch["rgb"].shape == (1, 3, 24, 32) and batch["depth"].shape == (1, 1, 24, 32)


# ------------------------------------------------------------------------------------------------- two ranks, gloo
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, n_frames, save_dir, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        obs = make_observations(n_frames)
        est = StandInEstimator()
        out = pr.run_predictions(pr.ListSceneDataset(obs, load_depth=True), est, CFG, save_dir=save_dir, device="cpu")
        preds = out["results"]["predictions"]
        # plain pickle: tensors by value (the queue's own reducer would pass shared-memory handles of a process that exits)
        q.put(pickle.dumps((rank, {k: (v.infos, {n: t for n, t in v.tensors.items()}) for k, v in preds.items()},
                            [(t["scene_id"], t["view_id"]) for t in out["frame_times"]], out["save_dir"] is not None)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n_frames", [5, 1])
def test_frames_sharded_over_two_ranks(tmp_path, n_frames):
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_frames, tmp_path / "run", q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((pickle.loads(q.get(timeout=180)) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
    obs = make_observations(n_frames)
    # each rank ran its own frames ...
    for rank, _, frames, saved in res:
        want = [(obs[i].infos.scene_id, obs[i].infos.view_id) for i in pr.DistributedSceneSampler(obs, world, rank)]
        assert frames == want and saved == (rank == 0)
    # ... every rank holds the same gathered predictions: rank 0's rows first, then rank 1's ...
    for k in res[0][1]:
        pd.testing.assert_frame_equal(res[0][1][k][0].drop(columns="time"), res[1][1][k][0].drop(columns="time"))
        for n in res[0][1][k][1]:
            assert torch.equal(res[0][1][k][1][n], res[1][1][k][1][n])
    # ... and they are the single-process predictions of the same frames, reordered
    order = [i for r in range(world) for i in pr.DistributedSceneSampler(obs, world, r)]
    single = pr.PredictionRunner(pr.ListSceneDataset([obs[i] for i in order], load_depth=True), CFG, device="cpu")
    single.sampler.local_indices = list(range(len(order)))
    want = single.get_predictions(StandInEstimator())
    from megapose6d_b200.tensor_collection import PandasTensorCollection

    for k, v in want.items():
        got = PandasTensorCollection(infos=res[0][1][k][0], **res[0][1][k][1])
        _same_collection(v, got)
    assert (tmp_path / "run" / "results.pth.tar").exists()


# --------------------------------------------------------------------------------------------- real estimator (GPU)
@pytest.mark.gpu
def test_runner_with_the_real_estimator(tmp_path):
    """Three frames through the runner == three direct pipeline calls (the fused pipeline is deterministic for equal
    inputs), with the look-ahead copies on the side stream in play."""
    from megapose6d_b200 import load_model, procedural
    from megapose6d_b200.example import make_detections_from_object_data
    from megapose6d_b200.types import ObservationTensor
    from tests import helpers

    ds, _, _ = helpers.make_scene(2, seed=6)
    load_model.write_run(tmp_path, "coarse-rgb-906902141", helpers.make_state_dict(helpers.COARSE_CFG, 5))
    load_model.write_run(tmp_path, "refiner-rgb-653307694", helpers.make_state_dict(helpers.REFINER_CFG, 6))
    est = load_model.load_named_model("megapose-1.0-RGB", ds, models_root=tmp_path).cuda()
    K = procedural.example_camera()
    rs = np.random.RandomState(0)
    frames = []
    for f in range(3):
        objs = [ObjectData(label=ds[k].label, bbox_modal=np.array([200.0 + 40 * k + 10 * f, 150, 330 + 40 * k + 10 * f, 290]))
                for k in range(1 + f % 2)]
        frames.append(pr.SceneObservation(rgb=rs.randint(0, 256, (480, 640, 3)).astype(np.uint8), depth=None,
                                          infos=pr.ObservationInfos(scene_id=1, view_id=f), object_datas=objs,
                                          camera_data=CameraData(K=K, resolution=(480, 640))))
    cfg = InferenceConfig(detection_type="gt", n_refiner_iterations=2, n_pose_hypotheses=1, bsz_images=576, bsz_objects=16)
    runner = pr.PredictionRunner(pr.ListSceneDataset(frames), cfg)
    preds = runner.get_predictions(est)
    assert len(preds["final"]) == sum(len(f.object_datas) for f in frames) and torch.isfinite(preds["final"].poses).all()
    rows = 0
    for i in runner.sampler:
        f = frames[i]
        # same conversion as the runner's (and the reference runner's, evaluation/prediction_runner.py:104-112): uint8 ->
        # float32 / 255 ON THE DEVICE -- torch's CUDA division by a scalar multiplies by the reciprocal, one ulp away from
        # the host's true division on a third of the 256 levels
        obs = ObservationTensor.from_torch_batched(torch.from_numpy(f.rgb).permute(2, 0, 1).unsqueeze(0).cuda(), None,
                                                   torch.as_tensor(K).unsqueeze(0).cuda())
        det = make_detections_from_object_data(f.object_datas).cuda()
        want, _ = est.run_inference_pipeline(obs, detections=det, n_refiner_iterations=2, n_pose_hypotheses=1,
                                             bsz_images=576, bsz_objects=16)
        got = preds["final"][list(range(rows, rows + len(want)))]
        rows += len(want)
        assert got.infos["view_id"].tolist() == [f.infos.view_id] * len(want)
        assert got.infos["label"].tolist() == want.infos["label"].tolist()
        assert torch.allclose(got.poses.cpu(), want.poses.cpu(), atol=1e-6)
