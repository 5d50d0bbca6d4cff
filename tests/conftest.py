import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class GoldenArchives(dict):
    """The arrays of several .npz archives as one mapping, in archive order; ``files`` lists the keys like ``np.load``'s."""

    @property
    def files(self):
        return list(self)


@pytest.fixture(scope="session")
def golden():
    """Vectors produced by the unmodified reference (tests/golden/make_golden.py), split over
    reference_vectors_<n>.npz so that no file exceeds 1 MB."""
    paths = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "reference_vectors_*.npz")),
                   key=lambda p: int(p.rsplit("_", 1)[1][:-4]))
    assert paths, "tests/golden/reference_vectors_*.npz not found"
    out = GoldenArchives()
    for path in paths:
        with np.load(path) as z:
            out.update((k, z[k]) for k in z.files)
    return out


@pytest.fixture(scope="session")
def pl_graph(golden):
    """The 60 x 90 power-law graph of the golden file as dense ids + oracle CSR."""
    from oracle import hgr_oracle as O

    u, i = golden["pl_dense_u"], golden["pl_dense_i"]
    n_users, n_items = len(golden["pl_id2user"]), len(golden["pl_id2item"])
    csr = O.build_norm_adj(u, i, n_users, n_items)
    return dict(u=u, i=i, n_users=n_users, n_items=n_items, csr=csr)


def rowwise_rel_err(a, b):
    """max over ROWS of  max_j |a_ij - b_ij| / max_j |b_ij| : every embedding row (last-dimension vector) is judged against
    its OWN magnitude, so a row of small embeddings cannot hide behind the largest entry of the table (VERDICT r1).  A
    reference row that is exactly zero (an empty segment, an isolated node) must be reproduced exactly.  Scalars and 1-D
    arrays count as one row."""
    import torch

    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    a, b = a.astype(np.float64), b.astype(np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    if b.size == 0:
        return 0.0
    a2, b2 = (a.reshape(1, -1), b.reshape(1, -1)) if b.ndim < 2 else (a.reshape(-1, b.shape[-1]), b.reshape(-1, b.shape[-1]))
    diff = np.abs(a2 - b2).max(axis=1)
    scale = np.abs(b2).max(axis=1)
    err = np.where(scale > 0, diff / np.where(scale > 0, scale, 1.0), np.where(diff > 0, np.inf, 0.0))
    return float(err.max())


def global_rel_err(a, b):
    """max |a - b| / max |b| over the whole tensor.  Used for GRADIENTS of the losses only: a gradient row is a sum of
    per-triple (per-pair) terms that largely cancel, so its own magnitude says nothing about the rounding error of the terms
    that produced it; the scale of the terms is the scale of the largest rows."""
    import torch

    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    return float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max() / max(np.abs(b).max(), 1e-30))
