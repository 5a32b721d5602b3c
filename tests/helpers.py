"""Shared builders for the tests: the synthetic workloads (re-exported from workloads/), oracle objects, reference
adapters and the checker of the reference's pipeline fixtures."""
from __future__ import annotations

import numpy as np
import torch

from megapose6d_b200 import procedural
from oracle import pipeline_ref, resnet_ref  # noqa: F401
from workloads.scenes import (FULLSIZE, bench_scene, detection_for_pose, make_scene, pipeline_scenario,  # noqa: F401
                              rgbd_scene, ycbv_scene)
from workloads.weights import (COARSE_CFG, REFINER_CFG, REFINER_RGBD_CFG, calibration_batch, make_state_dict,  # noqa: F401
                               n_inputs)

_calibration_batch = calibration_batch


def ref_meshes_from_dataset(ds) -> pipeline_ref.RefMeshes:
    labels, v, n, c, f, uv, tex, mod = [], [], [], [], [], [], [], []
    for obj in ds.list_objects:
        m = obj.mesh.with_defaults()
        labels.append(obj.label)
        v.append(np.asarray(m.vertices, np.float64) * obj.scale)
        n.append(m.vertex_normals)
        c.append(np.clip(m.vertex_colors, 0, 1))
        f.append(m.faces)
        uv.append(m.uv)
        tex.append(m.texture)
        mod.append(1 if m.texture_modulate else 0)
    return pipeline_ref.RefMeshes(labels, v, n, c, f, uv, tex, mod)


def check_pipeline_against_golden(golden, coarse_poses, coarse_logits, kept_hypotheses, exact_network: bool,
                                  final_labels=None, final_hypotheses=None, final_poses=None):
    """`golden`: tests/golden/pipeline.npz (outputs of the reference's own PoseEstimator.run_inference_pipeline).
    coarse_poses [2*72,4,4] / coarse_logits [2*72] in the reference's row order (detection-major, grid order);
    kept_hypotheses: per detection, the set of hypothesis ids that survived the coarse filter.

    Tolerances: the initial poses are fp32 geometry -> rtol 2e-5 / atol 2e-6 (the oracle reproduces the reference to
    1e-5 / 1e-6, the CUDA path the oracle to the same).  Logits: an fp32 network (`exact_network`) must reproduce them to
    rtol 1e-4 / atol 1e-5 and give the same final result; the bf16 CUDA network is checked through what the logits are
    used for -- the same survivors wherever the reference's ranking margin is well above the observed noise."""
    want_poses = torch.from_numpy(golden["coarse_poses"])
    assert torch.allclose(coarse_poses.float().cpu(), want_poses, rtol=2e-5, atol=2e-6)
    want = torch.from_numpy(golden["coarse_logit"]).float()
    got = torch.as_tensor(np.array(torch.as_tensor(coarse_logits).cpu() if torch.is_tensor(coarse_logits) else coarse_logits, dtype=np.float32))
    err = (got - want).abs()
    if exact_network:
        assert torch.allclose(got, want, rtol=1e-4, atol=1e-5), f"coarse logits: max err {err.max():.3g}"
        tol = 1e-4
    else:
        tol = 4.0 * err.median().item() + 0.05
    n_det, m = golden["kept_hypotheses"].shape[0], want.numel() // golden["kept_hypotheses"].shape[0]
    k = golden["kept_hypotheses"].shape[1]
    checked = 0
    for det in range(n_det):
        ranked = torch.sort(want[det * m:(det + 1) * m], descending=True).values
        if (ranked[k - 1] - ranked[k]).item() > 2 * tol:
            assert set(int(h) for h in kept_hypotheses[det]) == set(int(h) for h in golden["kept_hypotheses"][det]), det
            checked += 1
    if exact_network:
        assert checked == n_det, "the scenario was chosen with clear margins"
        order_w, order_g = np.argsort(golden["final_label"]), np.argsort(np.asarray(final_labels))
        assert [int(h) for h in np.asarray(final_hypotheses)[order_g]] == [int(h) for h in golden["final_hypothesis"][order_w]]
        assert torch.allclose(final_poses.float().cpu()[order_g], torch.from_numpy(golden["final_poses"])[order_w],
                              rtol=1e-4, atol=1e-5)
    return dict(max_logit_err=err.max().item(), survivors_checked=checked)


# ------------------------------------------------------------------------------------------------------------------------
# Outputs of the original project, stored under tests/golden/ (tools/make_golden.py writes them): data frames and tensor
# collections flattened into the arrays of one .npz, and read back with the index, column order and dtypes they had.
# ------------------------------------------------------------------------------------------------------------------------
def record_frame(out: dict, prefix: str, df) -> None:
    """One JSON string: column names and dtypes, index and values (Python's float repr round-trips exactly)."""
    import json

    import pandas as pd

    cols = [str(c) for c in df.columns]
    numeric = {c: pd.api.types.is_numeric_dtype(df[c]) or pd.api.types.is_bool_dtype(df[c]) for c in df.columns}
    rec = dict(columns=cols, dtypes=[str(df[c].dtype) if numeric[c] else "str" for c in df.columns],
               index=df.index.tolist(), data=[df[c].tolist() if numeric[c] else [str(v) for v in df[c]] for c in df.columns])
    out[prefix] = np.frombuffer(json.dumps(rec).encode(), dtype=np.uint8)


def restore_frame(d, prefix: str):
    import json

    import pandas as pd

    rec = json.loads(d[prefix].tobytes())
    data = {c: v if t == "str" else np.array(v, dtype=t) for c, t, v in zip(rec["columns"], rec["dtypes"], rec["data"])}
    return pd.DataFrame(data, columns=rec["columns"], index=pd.Index(np.array(rec["index"], dtype=np.int64)))


class StoredCollection:
    """A PandasTensorCollection read back from a fixture: `infos` with its original index, the tensors in their order."""

    def __init__(self, infos, tensors):
        self.infos, self._tensors = infos, tensors

    @property
    def tensors(self):
        return self._tensors

    def __len__(self):
        return len(self.infos)

    def __getattr__(self, name):
        if name.startswith("_") or name not in self._tensors:
            raise AttributeError(name)
        return self._tensors[name]


def record_collection(out: dict, prefix: str, c) -> None:
    record_frame(out, f"{prefix}/infos", c.infos)
    out[f"{prefix}/tensors"] = np.array(list(c.tensors.keys()), dtype="U")
    for k, t in c.tensors.items():
        out[f"{prefix}/t/{k}"] = t.numpy()


def restore_collection(d, prefix: str) -> StoredCollection:
    tensors = {str(k): torch.from_numpy(d[f"{prefix}/t/{k}"]) for k in d[f"{prefix}/tensors"]}
    return StoredCollection(restore_frame(d, f"{prefix}/infos"), tensors)


def record_sample(out: dict, prefix: str, t: torch.Tensor, n: int = 256, seed: int = 0) -> None:
    """A fixed sample of a large tensor: n values at seeded positions, n more among its non-zero values (renders are
    mostly background), and the float64 sum of every [H, W] plane."""
    flat = t.detach().reshape(-1)
    rs = np.random.RandomState(seed)
    nz = np.flatnonzero(flat.numpy())
    idx = np.concatenate([rs.choice(flat.numel(), min(n, flat.numel()), replace=False),
                          rs.choice(nz, min(n, len(nz)), replace=False) if len(nz) else np.zeros(0, np.int64)])
    out[f"{prefix}/idx"] = idx.astype(np.int32)
    out[f"{prefix}/val"] = flat[torch.from_numpy(idx)].numpy()
    out[f"{prefix}/plane_sum"] = t.detach().double().flatten(-2).sum(-1).numpy()
    out[f"{prefix}/shape"] = np.asarray(t.shape, dtype=np.int64)


def check_sample(d, prefix: str, t: torch.Tensor, atol: float) -> None:
    """`t` against record_sample's data: same shape, the sampled values within atol, each plane's sum within atol per
    element of the plane."""
    assert tuple(t.shape) == tuple(d[f"{prefix}/shape"]), (prefix, tuple(t.shape))
    got = t.detach().reshape(-1)[torch.from_numpy(d[f"{prefix}/idx"]).long()]
    want = torch.from_numpy(d[f"{prefix}/val"])
    if atol == 0:
        assert torch.equal(got, want), prefix
    else:
        assert torch.allclose(got, want, atol=atol, rtol=0), (prefix, (got - want).abs().max())
    hw = t.shape[-1] * t.shape[-2]
    sums = t.detach().double().flatten(-2).sum(-1)
    assert torch.allclose(sums, torch.from_numpy(d[f"{prefix}/plane_sum"]), rtol=1e-9, atol=max(atol, 1e-9) * hw), prefix


def tensor_digest(t) -> str:
    """dtype, shape and SHA-256 of the bytes: equal digests <=> torch.equal for tensors of the same dtype (no NaN)."""
    import hashlib

    a = np.ascontiguousarray(t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t))
    return f"{a.dtype}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()}"
