"""Shared helpers for the tests: synthetic state_dict from the committed schema, golden loading."""
from __future__ import annotations

import functools
import json
from pathlib import Path

import torch

GOLD = Path(__file__).resolve().parent / "golden"


def gold(name):
    """A golden file; "parts" names further files whose tensors complete its "taps" (kept apart so no file exceeds 1 MB)."""
    g = torch.load(GOLD / name, map_location="cpu", weights_only=False)
    for part in g.pop("parts", []) if isinstance(g, dict) else []:
        g.setdefault("taps", {}).update(torch.load(GOLD / part, map_location="cpu", weights_only=False))
    return g


def sample_index(numel, n=8192):
    """Flat indices of a fixed sample of n elements out of numel (all of them when numel <= n): a multiplicative hash by a
    prime, so the same positions are chosen on every machine and torch version."""
    if numel <= n:
        return torch.arange(numel)
    return (torch.arange(n, dtype=torch.int64) * 2654435761 + 40503) % numel


def take_sample(t, n=8192):
    """The elements of `t` at sample_index(t.numel(), n), dtype kept."""
    return t.detach().reshape(-1)[sample_index(t.numel(), n).to(t.device)].cpu()


@functools.lru_cache(maxsize=1)
def schema():
    return json.loads((GOLD / "schema_reduced.json").read_text())


@functools.lru_cache(maxsize=1)
def synth_state_dict():
    """fp32 CPU state_dict with the reference's key schema (reduced depth: 1 PCB + 1 IRG), values from the per-key
    seeded generator — identical to what tools/make_golden.py loaded into the reference."""
    from fwb_synth import synth_tensor
    return {k: synth_tensor(k, shape, seed=0, device="cpu") for k, shape in schema().items()}


def subset(sd, prefixes):
    return {k: v for k, v in sd.items() if any(k.startswith(p) for p in prefixes)}


def rel_err(a, b):
    a, b = a.float(), b.float()
    return float((a - b).norm() / (b.norm() + 1e-12))


def max_err(a, b):
    return float((a.float() - b.float()).abs().max())


def assert_close_frac(out, ref, rtol, atol, loose_atol, max_bad_frac=2e-4):
    """assert_close that tolerates a tiny fraction of elements (bf16 round-to-nearest ties that fall the other way because
    fp32 sums were accumulated in a different order) at a looser absolute bound."""
    out, ref = out.float(), ref.float()
    diff = (out - ref).abs()
    bad = diff > (atol + rtol * ref.abs())
    frac = float(bad.float().mean())
    assert frac <= max_bad_frac, f"{frac:.2e} of elements outside rtol={rtol} atol={atol}"
    assert float(diff.max()) <= loose_atol, f"max abs diff {float(diff.max()):.3e} > {loose_atol}"
