"""Drop-in surface (SURVEY §8b, VERDICT r1 weak #10): (1) every `FantasyWorld.*` import the reference CLIs perform resolves against
the mirror package and yields the named objects; (2) the FULL-depth model (16 PCB + 24 IRG, heads) has exactly the reference's
state_dict schema (3132 keys) — so the released `model.pth` loads with no missing / unexpected keys (inference_wan21.py:215-220).
The reference side is pinned by goldens taken from the unmodified reference (tools/make_golden_ref_parity.py): the CLIs' import
lists, the schema digest and the pose-encoding helpers' outputs."""
import hashlib
import json
from pathlib import Path

import pytest
import torch

from _common import GOLD, gold

ROOT = Path(__file__).resolve().parent.parent
FULL_SCHEMA_SHA256 = "00e3ba3a81647252f5a9ccac297d6bf44b332c554164914219d7942132082606"   # reference, 16 PCB + 24 IRG, heads: 3132 keys
FULL_SCHEMA_KEYS = 3132


def _mirror_full_schema():
    from fwb200.synth import CAMERA_CFG, VGGT_CFG, WAN21_I2V_14B
    from FantasyWorld.fusion.model_wan21 import FantasyWorldFusionModel
    with torch.device("meta"):
        m = FantasyWorldFusionModel(start_index=16, use_gradient_checkpointing=False, cross_attention_list=list(range(24)), dit_path=None,
                                    vggt_cfg=dict(VGGT_CFG), camera_control=True, camera_cfg=dict(CAMERA_CFG), dit_config=dict(WAN21_I2V_14B))
    return {k: list(v.shape) for k, v in m.state_dict().items()}


def test_full_depth_state_dict_schema_is_the_reference_one():
    ours = _mirror_full_schema()
    assert len(ours) == FULL_SCHEMA_KEYS
    assert hashlib.sha256(json.dumps(sorted(ours.items())).encode()).hexdigest() == FULL_SCHEMA_SHA256
    # the surgery leaves Identity behind exactly where the reference does (model_wan21.py:74-75)
    assert not any(k.startswith(("pipe.dit.blocks.16.", "pipe.dit.blocks.39.", "vggt.aggregator.global_blocks.")) for k in ours)


@pytest.mark.parametrize("cli", ["inference_wan21.py", "inference_wan22.py"])
def test_reference_cli_import_block_resolves_against_the_mirror(cli):
    checked = 0
    for module, names in json.loads((GOLD / "reference_cli_imports.json").read_text())[cli]:
        if "vram_management" in module:
            continue        # CPU offload: not part of this build (everything stays resident in HBM)
        mod = __import__(module, fromlist=names)
        assert str(Path(mod.__file__).resolve()).startswith(str(ROOT / "fantasy-world_b200")), (module, mod.__file__)
        for name in names:
            assert hasattr(mod, name), f"{cli}: from {module} import {name}"
            checked += 1
    assert checked >= 2, checked


def pose_inputs():
    """Random and degenerate (180 degree) rotations, their matrices, extrinsics and intrinsics (float64)."""
    from FantasyWorld.vggt.utils.rotation import quat_to_mat
    g = torch.Generator().manual_seed(3)
    q = torch.randn(2, 37, 4, generator=g, dtype=torch.float64)
    q[0, :6] = torch.tensor([[1.0, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1], [1, 1, 0, 0], [0.6, 0, 0.8, 1e-9]], dtype=torch.float64)
    R = quat_to_mat(q)
    ext = torch.cat([R, torch.randn(2, 37, 3, 1, generator=g, dtype=torch.float64)], dim=-1)
    K = torch.zeros(2, 37, 3, 3, dtype=torch.float64)
    K[..., 0, 0], K[..., 1, 1], K[..., 0, 2], K[..., 1, 2], K[..., 2, 2] = 500.0, 450.0, 416.0, 240.0, 1.0
    return q, R, ext, K


def test_pose_encoding_helpers_match_reference():
    """FantasyWorld.vggt.utils.{pose_enc, rotation} (imported by both reference CLIs): the mirror against the reference's own
    functions (golden pose_enc_ref.pt) on random and degenerate (180 degree) rotations, plus the encode -> decode round trip."""
    from FantasyWorld.vggt.utils import pose_enc as mine
    from FantasyWorld.vggt.utils.rotation import mat_to_quat, quat_to_mat
    q, R, ext, K = pose_inputs()
    assert torch.allclose(R @ R.transpose(-1, -2), torch.eye(3, dtype=torch.float64).expand_as(R), atol=1e-12)
    q2 = mat_to_quat(R)
    assert (q2[..., 3] >= 0).all() and torch.allclose(quat_to_mat(q2), R, atol=1e-9)
    enc = mine.extri_intri_to_pose_encoding(ext, K, (480, 832))
    assert enc.shape == (2, 37, 9) and enc.dtype == torch.float32
    e2, k2 = mine.pose_encoding_to_extri_intri(enc.double(), (480, 832))
    assert torch.allclose(e2, ext, atol=1e-5) and torch.allclose(k2, K, atol=1e-3)
    ref = gold("pose_enc_ref.pt")
    assert torch.allclose(q2, ref["mat_to_quat"], atol=1e-12)
    assert torch.allclose(R, ref["quat_to_mat"], atol=1e-12)
    assert torch.equal(enc, ref["encoding"])
    me, mk = mine.pose_encoding_to_extri_intri(enc, (480, 832))
    assert torch.equal(me, ref["extri"]) and torch.equal(mk, ref["intri"])
