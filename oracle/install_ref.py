"""Put the UNMODIFIED original CoLearn project under ``oracle/_ref`` (git-ignored) for ``bench.py --impl reference``.

The original is a flat tree of scripts without ``setup.py`` / ``pyproject.toml``, so pip cannot install it.  Its modules
are meant to be run from the checkout, so the "install" is a byte-identical copy of the Python sources + the example
dataset + the allow-list, with a ``SHA256SUMS`` manifest that ``verify()`` re-checks before every reference-arm run.
Nothing here imports the product package.

The source is a checkout of the original project: ``--src``, else the ``COLEARN_REFERENCE_SRC`` environment variable,
else ``DEFAULT_SRC`` when a readable checkout is there.  ``__graft_entry__.build()`` runs :func:`install` whenever
:func:`source` finds one, so the reference arm and its tests have the original wherever it is available at build time.

    python oracle/install_ref.py --src <checkout of the original project>
"""
from __future__ import annotations

import hashlib
import os
import shutil
import sys
from typing import Dict, Optional

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
SRC_ENV = "COLEARN_REFERENCE_SRC"
DEFAULT_SRC = "/root/reference"     # default location of a checkout of the original project
FILES = ["federated_coordinator.py", "client_federated.py", "remote_worker.py", "datasets.py", "event_parser.py", "settings.py",
         "README.md", "device_filtering/filtering_file.txt", "device_filtering/file_upgrader.py",
         "dataset_example/UNSW_2018_IoT_Botnet_Final_10_best_Training_1_1.csv"]


def _sha(path: str) -> str:
    h = hashlib.sha256()
    with open(path, "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def source() -> Optional[str]:
    """The checkout named by ``COLEARN_REFERENCE_SRC``, else ``DEFAULT_SRC`` if a readable checkout is there, else None."""
    if os.environ.get(SRC_ENV):
        return os.environ[SRC_ENV]
    return DEFAULT_SRC if os.access(os.path.join(DEFAULT_SRC, "federated_coordinator.py"), os.R_OK) else None


def install(src: str, dest: str = DEST) -> Dict[str, str]:
    sums = {}
    for rel in FILES:
        s, d = os.path.join(src, rel), os.path.join(dest, rel)
        if not os.path.exists(s):
            continue
        os.makedirs(os.path.dirname(d), exist_ok=True)
        shutil.copyfile(s, d)
        sums[rel] = _sha(d)
        assert sums[rel] == _sha(s)
    with open(os.path.join(dest, "SHA256SUMS"), "w") as f:
        for rel, h in sorted(sums.items()):
            f.write(f"{h}  {rel}\n")
    return sums


def verify(dest: str = DEST) -> Dict[str, str]:
    """Re-hash the installed files against the manifest written at install time; returns {file: sha256}."""
    manifest = os.path.join(dest, "SHA256SUMS")
    if not os.path.exists(manifest):
        raise FileNotFoundError(f"{manifest} missing: run `python oracle/install_ref.py --src <checkout of the original project>`")
    sums = {}
    with open(manifest) as f:
        for line in f:
            h, rel = line.strip().split("  ", 1)
            if _sha(os.path.join(dest, rel)) != h:
                raise RuntimeError(f"oracle/_ref/{rel} differs from the installed reference file")
            sums[rel] = h
    return sums


if __name__ == "__main__":
    src = sys.argv[sys.argv.index("--src") + 1] if "--src" in sys.argv else source()
    if not src:
        sys.exit(f"no checkout of the original project at {DEFAULT_SRC}: python oracle/install_ref.py --src <checkout> (or set {SRC_ENV})")
    for rel, h in sorted(install(src).items()):
        print(h, rel)
