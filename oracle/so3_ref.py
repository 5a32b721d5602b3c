"""oracle/so3_ref.py -- SO(3) grid for the CPU oracle (TEST INFRASTRUCTURE ONLY).

Restates load_SO3_grid (src/megapose/utils/transform_utils.py:27-50) on the converted data asset
(tests/test_oracle_vs_reference.py holds the asset to the grid parsed from the reference's own text file).
"""
from __future__ import annotations

from pathlib import Path

import numpy as np
import torch

from .lib3d_ref import unitquat_to_rotmat

_ASSET = Path(__file__).resolve().parents[1] / "megapose6d_b200" / "data"


def load_quats(resolution: int) -> torch.Tensor:
    return torch.tensor(np.load(_ASSET / f"so3_grid_{resolution}.npy").tolist())


def load_SO3_grid_reference(resolution: int) -> torch.Tensor:
    return unitquat_to_rotmat(load_quats(resolution))
