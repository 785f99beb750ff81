"""TEST INFRASTRUCTURE — recipe that installs the UNMODIFIED reference (s3prl) into oracle/_ref.

    python oracle/build_ref.py [--force]

The reference is the s3prl repository checked out beside this one (../reference), or wherever S3PRL_REFERENCE points.
Without a readable checkout the recipe is a no-op and an install made earlier stays in use. oracle/_ref/ is
git-ignored (no reference source ever enters the history); a copy of the tree that includes it lets
`bench.py --impl reference` time the reference's own `s3prl.upstream.hubert.expert.UpstreamExpert` +
`s3prl.upstream.interfaces.Featurizer` on the host cores (cpu_baseline.kind = "reference"),
`python -m s3prl_b200.run_downstream` import the reference's Runner (config 5), and the tests that drive it run.

s3prl is pure Python, so the install is a copy of what its wheel packages (the Python files, version.txt and the yaml
configs), plus the vocabularies of the one downstream recipe the launcher uses (downstream/ctc/vocab), which the wheel
does not package. No pip is needed.
"""
from __future__ import annotations

import os
import shutil
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
REFERENCE = Path(os.environ.get("S3PRL_REFERENCE") or ROOT.parent / "reference")
TARGET = ROOT / "oracle" / "_ref"


def exists(path: Path) -> bool:
    """Path.exists() that answers False for a path the current user may not look into."""
    try:
        return path.exists()
    except OSError:
        return False


def is_current() -> bool:
    return exists(TARGET / "s3prl" / "upstream" / "hubert" / "expert.py") and exists(
        TARGET / "s3prl" / "downstream" / "ctc" / "librispeech.yaml"
    )


def _not_packaged(directory: str, names: list) -> list:
    """copytree filter: skip what the s3prl wheel leaves out (data and result directories, caches, non-config files)."""
    def packaged(name: str) -> bool:
        if (Path(directory) / name).is_dir():
            return name not in ("data", "result", "__pycache__")
        return name.endswith((".py", ".yaml")) or name == "version.txt"

    return [n for n in names if not packaged(n)]


def build(force: bool = False) -> Path | None:
    if not exists(REFERENCE / "s3prl" / "upstream" / "hubert" / "expert.py"):
        return TARGET if is_current() else None
    if is_current() and not force:
        return TARGET
    if TARGET.exists():
        shutil.rmtree(TARGET)
    shutil.copytree(REFERENCE / "s3prl", TARGET / "s3prl", ignore=_not_packaged)
    vocab = REFERENCE / "s3prl" / "downstream" / "ctc" / "vocab"
    if vocab.exists():
        shutil.copytree(vocab, TARGET / "s3prl" / "downstream" / "ctc" / "vocab", dirs_exist_ok=True)
    return TARGET


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
