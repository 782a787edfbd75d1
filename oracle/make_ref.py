"""oracle/make_ref.py — recipe that stages the UNMODIFIED reference next to the oracle so that it can travel to the GPU box.

    python oracle/make_ref.py            # /root/reference -> oracle/_ref/   (run by __graft_entry__.build() in the build container)

TEST INFRASTRUCTURE ONLY.  The reference (Fantasy-AMAP/fantasy-world) is pure Python: there is nothing to compile, and it
has no setup.py / pyproject.toml, so `pip install --target baseline/_ref` does not apply.  What the parity contract needs
(SURVEY §8c, VERDICT r1 item 1) is the reference's own modules running on the same B200 under
`torch.autocast("cuda", bf16)` as the bf16 parity target and as the GPU baseline.  `/root/reference` does not exist on
the GPU box, but `oracle/_ref/` (git-ignored, NOT gpurun-ignored, exactly like a compiled oracle/_ref/*.so) ships with
every `gpurun` snapshot.  This script copies the reference's Python sources byte for byte — no edits — into
`oracle/_ref/`, and writes a manifest (sha256 per file + the reference commit) so that a parity run can state exactly
what it compared against.  Nothing under `oracle/_ref/` is ever committed and nothing in the product path reads it: only
tools/ref_shim.py (used by oracle/ref_runner.py — i.e. tests/ and bench.py's reference legs — and by the golden generators) puts it on sys.path.
"""
from __future__ import annotations

import hashlib
import json
import shutil
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
SRC = Path("/root/reference")
DST = HERE / "_ref"
TOP_LEVEL = ("inference_wan21.py", "inference_wan22.py", "utils.py")   # CLI boundary files (import-block test)


def stage(force: bool = False) -> Path | None:
    """Copy FantasyWorld/**/*.py (+ the CLI files) from /root/reference to oracle/_ref.  Returns the destination, or None
    when the reference is absent (GPU box: the already-staged copy, if any, is used as is)."""
    try:
        present = SRC.is_dir()
    except OSError:             # e.g. the reference sits in a directory this user may not enter
        present = False
    if not present:
        return DST if (DST / "MANIFEST.json").exists() else None
    files = sorted(p for p in (SRC / "FantasyWorld").rglob("*.py"))
    files += [SRC / n for n in TOP_LEVEL if (SRC / n).exists()]
    manifest = {"source": str(SRC), "files": {}}
    sub = SRC / ".SUBMODULES.json"
    if sub.exists():
        try:
            manifest["commit"] = json.loads(sub.read_text()).get("commit")
        except Exception:
            pass
    for p in files:
        rel = p.relative_to(SRC)
        data = p.read_bytes()
        manifest["files"][str(rel)] = hashlib.sha256(data).hexdigest()
        out = DST / rel
        if force or not out.exists() or out.read_bytes() != data:
            out.parent.mkdir(parents=True, exist_ok=True)
            out.write_bytes(data)
    # drop files that no longer exist in the source
    for p in list(DST.rglob("*.py")):
        if str(p.relative_to(DST)) not in manifest["files"]:
            p.unlink()
    (DST / "MANIFEST.json").write_text(json.dumps(manifest, indent=1, sort_keys=True))
    return DST


def verify() -> bool:
    """True when every staged file still has the sha256 recorded at staging time (i.e. the staged reference is unmodified)."""
    mf = DST / "MANIFEST.json"
    if not mf.exists():
        return False
    files = json.loads(mf.read_text())["files"]
    return all((DST / rel).exists() and hashlib.sha256((DST / rel).read_bytes()).hexdigest() == h for rel, h in files.items())


if __name__ == "__main__":
    if "--clean" in sys.argv and DST.exists():
        shutil.rmtree(DST)
    d = stage(force="--force" in sys.argv)
    print(d, "verified" if d and verify() else "ABSENT")
