"""The reference runner (oracle/ref_runner.py: the UNMODIFIED reference in its own process) against the oracle on the CPU.

This pins the plumbing the GPU parity goldens rely on: the runner builds the reference with the per-key synthetic weights and
the seeded block inputs of fwb_synth, and must therefore reproduce what the oracle computes from the same state_dict and
inputs (fp32, tolerance = summation order).  The runner's output is the golden ref_runner_blocks_cpu.pt
(tools/make_golden_ref_parity.py); the staging recipe that puts the reference next to the runner is checked on a scratch tree."""
import json
import sys
from pathlib import Path

import torch

from _common import gold, rel_err, synth_state_dict

ROOT = Path(__file__).resolve().parent.parent


def test_staged_reference_is_unmodified(tmp_path, monkeypatch):
    sys.path.insert(0, str(ROOT))
    from oracle import make_ref
    if (make_ref.DST / "MANIFEST.json").exists():
        assert make_ref.verify()
    src, dst = tmp_path / "src", tmp_path / "dst"
    (src / "FantasyWorld" / "fusion").mkdir(parents=True)
    (src / "FantasyWorld" / "fusion" / "block.py").write_bytes(b"x = 1\n")
    (src / "inference_wan21.py").write_bytes(b"import FantasyWorld\n")
    monkeypatch.setattr(make_ref, "SRC", src)
    monkeypatch.setattr(make_ref, "DST", dst)
    assert make_ref.stage() == dst and make_ref.verify()
    assert (dst / "FantasyWorld" / "fusion" / "block.py").read_bytes() == b"x = 1\n"
    assert sorted(json.loads((dst / "MANIFEST.json").read_text())["files"]) == ["FantasyWorld/fusion/block.py", "inference_wan21.py"]
    (dst / "inference_wan21.py").write_bytes(b"import FantasyWorld  # edited\n")
    assert not make_ref.verify()
    monkeypatch.setattr(make_ref, "SRC", tmp_path / "absent")
    assert make_ref.stage() == dst            # no source: the copy already staged is used as is


def test_runner_blocks_match_oracle_fp32():
    from fwb_synth import synth_block_inputs
    from oracle import fw_oracle as O
    f, h, w, text_len = 1, 4, 4, 64
    ref = gold("ref_runner_blocks_cpu.pt")
    assert ref["report"]["grid"] == [f, h, w]
    assert ref["report"]["modes"]["fp32"]["dit_attention_backend"] == "F.scaled_dot_product_attention"
    sd = {k: v.to(torch.bfloat16).float() for k, v in synth_state_dict().items()}      # the fp32 mode runs on bf16-valued weights
    inp = synth_block_inputs(f, h, w, text_len)
    tab, tab_d, tab_a = O.rope_table_3d(128, f, h, w), O.rope_table_3d(96, f, h, w), O.rope_table_3d_with_extra(96, f, h, w, 5)
    _, pos = O.aggregator_input(sd, "vggt.aggregator", torch.zeros(1, f, h, w, 1024))
    pcb = O.dit_block(sd, "pipe.dit.blocks.0", inp["x_dit"], inp["context"], inp["t_mod"], tab, inp["plucker"])
    frame = O.vggt_block(sd, "vggt.aggregator.frame_blocks.0", inp["x_agg"], pos, inp["e0"])
    xd, xa, _ = O.irg_block(sd, "IRGBlock.0", inp["x_dit"], inp["x_agg"], inp["context"], inp["t_mod"], tab, tab_d, tab_a, pos, inp["e0"],
                            inp["plucker"])
    assert rel_err(ref["pcb"], pcb) < 2e-4, rel_err(ref["pcb"], pcb)
    assert rel_err(ref["frame"], frame) < 2e-4, rel_err(ref["frame"], frame)
    assert rel_err(ref["irg_x"], xd) < 2e-4, rel_err(ref["irg_x"], xd)
    assert rel_err(ref["irg_tokens"].reshape(xa.shape), xa) < 2e-4, rel_err(ref["irg_tokens"].reshape(xa.shape), xa)
