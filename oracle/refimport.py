"""Import the UNMODIFIED reference (chzhang18/RAG ``src/``) -- TEST / BASELINE INFRASTRUCTURE ONLY.

The reference is a tree of plain Python files without a package or a setup.py; ``tools/install_ref.sh``
(run by ``__graft_entry__.build()``) copies it to the git-ignored ``oracle/_ref/src``, inside the repository tree, so
that it goes wherever the built tree goes.  This helper reads the reference from there only: it puts that directory
on ``sys.path`` and imports the modules the hot path lives in.  Nothing under ``rag_b200/`` imports this file; users
are ``tests/``, ``__graft_entry__.smoke()`` and bench.py's reference / cpu_baseline legs.

On a machine without a CUDA driver the reference's head cannot run as written (``rag_model.py:26`` builds its
``arange`` on ``torch.cuda.current_device()``); ``cpu_patch=True`` applies the one monkeypatch that makes the
unmodified code run on CPU (SURVEY.md section 8c).  On the GPU box the reference runs unmodified.
"""
from __future__ import annotations

import hashlib
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = os.path.join(ROOT, "oracle", "_ref")
SRC = os.path.join(BASE, "src")


def ref_src() -> str | None:
    return SRC if os.path.isdir(os.path.join(SRC, "models")) else None


def available() -> bool:
    return ref_src() is not None


def verify_manifest() -> int:
    """Check oracle/_ref against the sha256 manifest written at install time; returns #files checked."""
    n = 0
    with open(os.path.join(BASE, "MANIFEST.sha256")) as f:
        for line in f:
            digest, rel = line.split()
            with open(os.path.join(SRC, rel), "rb") as g:
                if hashlib.sha256(g.read()).hexdigest() != digest:
                    raise RuntimeError(f"oracle/_ref/src/{rel} differs from the installed reference")
            n += 1
    return n


def import_reference(cpu_patch: bool = False) -> types.SimpleNamespace:
    """Returns a namespace with the reference modules: rag_model, mdenas_basicmodel, operations_3d,
    genotypes_2d, utils, metrics.  Raises RuntimeError when the reference is not installed."""
    src = ref_src()
    if src is None:
        raise RuntimeError("the reference is not installed: run tools/install_ref.sh (RAG_REFERENCE = a checkout of it)")
    if src not in sys.path:
        sys.path.insert(0, src)
    if cpu_patch:
        import torch

        if not torch.cuda.is_available():
            torch.cuda.current_device = lambda: "cpu"  # rag_model.py:26 (permanent: there is no CUDA device to name)
    import automl.genotypes_2d as genotypes_2d
    import automl.mdenas_basicmodel as mdenas_basicmodel
    import automl.operations_3d as operations_3d
    import models.rag_model as rag_model
    import utils as ref_utils
    import utilstool.metrics as metrics

    if not hasattr(ref_utils, "get_model"):
        raise RuntimeError(f"'utils' resolved to {ref_utils.__file__}, not the reference's src/utils.py")
    return types.SimpleNamespace(src=src, rag_model=rag_model, mdenas_basicmodel=mdenas_basicmodel,
                                 operations_3d=operations_3d, genotypes_2d=genotypes_2d, utils=ref_utils, metrics=metrics)


class on_cpu:
    """Context manager for running the unmodified reference head on CPU tensors on a machine that HAS a CUDA device:
    rag_model.py:26 builds its ``arange`` on ``torch.cuda.current_device()``, so for the duration of the block that
    function answers 'cpu' (the one monkeypatch of SURVEY.md section 8c); restored on exit."""

    def __enter__(self):
        import torch

        self._orig = torch.cuda.current_device
        torch.cuda.current_device = lambda: "cpu"
        return self

    def __exit__(self, *exc):
        import torch

        torch.cuda.current_device = self._orig
        return False


def make_genotype(ref, seed: int = 0):
    """A Genotype of the shape ``BasicNetwork.genotype()`` returns (mdenas_basicmodel.py:110-133): per cell, for
    each of the 3 steps the two chosen input edges and an op index in {0: skip_connect, 1: conv_3x3}."""
    import numpy as np

    rng = np.random.RandomState(seed)

    def gene():
        rows, start, n = [], 0, 2
        for _ in range(3):
            edges = rng.choice(np.arange(start, start + n), size=2, replace=False)
            for e in sorted(edges):
                rows.append([int(e), int(rng.randint(0, 2))])
            start += n
            n += 1
        return np.array(rows)

    return ref.genotypes_2d.Genotype(normal=gene(), normal_concat=None, reduce=gene(), reduce_concat=None)
