"""`hypergraph_diffusion_for_recommendation_b200.install()`: the reference's own modules import this package at every seam
(SURVEY.md section 8b).  Runs without a GPU: everything up to the first kernel call must work, and that call must fail loudly
(there is no CPU path).  Each case runs in a fresh interpreter so the swapped `sys.modules` entries do not leak into other tests."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# a checkout of the reference project (HD_SELFRec), the same variable the generators under tests/golden/ read
REF = os.environ.get("HGR_REFERENCE", "")
STUB = os.path.join(ROOT, "tests", "refstub")


def run(code, cwd=None):
    env = dict(os.environ, PYTHONPATH=ROOT, PYTHONDONTWRITEBYTECODE="1")
    p = subprocess.run([sys.executable, "-c", textwrap.dedent(code)], capture_output=True, text=True, env=env, cwd=cwd, timeout=600)
    assert p.returncode == 0, p.stdout[-3000:] + "\n" + p.stderr[-3000:]
    return p.stdout


SEAM_CHECK = """
    import hypergraph_diffusion_for_recommendation_b200 as hgr
    from hypergraph_diffusion_for_recommendation_b200 import data, encoders, evaluation, loss_torch, sampler, _lib
    mods = hgr.install(ROOT_OF_TREE)
    import model.graph.LightGCN as M
    import base.graph_recommender as G
    import util.loss_torch as L
    import util.sampler as S
    assert M.TorchGraphInterface is encoders.TorchGraphInterface          # seam 2
    assert M.bpr_loss is loss_torch.bpr_loss and M.l2_reg_loss is loss_torch.l2_reg_loss   # seam 4
    assert M.next_batch_pairwise is sampler.next_batch_pairwise           # 8f-1
    assert G.Interaction is data.Interaction                             # seam 1
    assert G.FileIO.load_data_set is data.FileIO.load_data_set
    assert G.GraphRecommender.test.__module__.endswith("b200.install")    # seam 5
    assert G.ranking_evaluation is evaluation.ranking_evaluation
    assert L.contrastLoss is loss_torch.contrastLoss and L.InfoNCE is loss_torch.InfoNCE
"""


def test_seams_resolve_on_the_stand_in_tree_and_the_first_kernel_call_fails_without_a_gpu(tmp_path):
    out = run(SEAM_CHECK.replace("ROOT_OF_TREE", repr(STUB)) + """
    import torch
    assert L.only_in_the_tree(1) == 2           # not provided by the package: falls through to the tree's own module
    assert hasattr(G.FileIO, "write_file")
    train = [[u, 100 + (u * 7 + k) % 40, 1.0] for u in range(30) for k in range(5)]
    test = [[u, 100 + (u * 11 + 3) % 40, 1.0] for u in range(30)]
    if torch.cuda.is_available():
        print("cuda present: constructor not expected to fail")
    else:
        try:
            M.LightGCN(None, train, test, item_ranking="10,20", batch_size=64)
            raise SystemExit("constructing the model without a GPU should have raised")
        except _lib.HgrError as e:
            assert "GPU" in str(e) or "CUDA" in str(e), str(e)
            print("raised:", e)
    """)
    assert "raised:" in out or "cuda present" in out


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs HGR_REFERENCE: a checkout of the unmodified reference project")
def test_the_reference_lightgcn_imports_this_package_at_every_seam(tmp_path):
    """The UNMODIFIED reference: `model/graph/LightGCN.py`, `base/graph_recommender.py`, `util/conf.py` from the HGR_REFERENCE checkout;
    conf/LightGCN.conf as shipped; train / test files in the reference's text format."""
    d = tmp_path / "dataset" / "lastfm"
    d.mkdir(parents=True)
    lines = ["user\titem"] + ["%d\t%d" % (u, 1000 + (u * 7 + k) % 50) for u in range(40) for k in range(6)]
    (d / "train.txt").write_text("\n".join(lines) + "\n")
    (d / "test.txt").write_text("\n".join(["user\titem"] + ["%d\t%d" % (u, 1000 + (u * 11 + 3) % 50) for u in range(40)]) + "\n")
    (d / "lastfm.kg").write_text("head\trelation\ttail\n0\t0\t1\n")
    os.symlink(os.path.join(REF, "conf"), tmp_path / "conf")
    out = run(SEAM_CHECK.replace("ROOT_OF_TREE", repr(REF)) + """
    import torch
    from util.conf import ModelConf
    assert callable(L.kl_divergence)                                     # reference-only helper still importable
    assert hasattr(G.FileIO, "load_kg_data") and hasattr(S, "next_batch_pointwise")
    conf = ModelConf("./conf/LightGCN.conf")
    conf.config["dataset"] = "lastfm"
    train = G.FileIO.load_data_set("./dataset/lastfm/train.txt", conf["model.type"])
    test = G.FileIO.load_data_set("./dataset/lastfm/test.txt", conf["model.type"])
    assert type(train).__name__ == "InteractionList" and len(train) == 240
    kw = dict(experiment="full", item_ranking="10,20", batch_size=64, lrate=0.001, lr_decay=0.9, weight_decay=5e-6, reg=0.1, p=0.3,
              drop_rate=0.2, n_layers=2, temp=0.2, cl_rate=1e-5, max_epoch=1, early_stopping_steps=5)
    if torch.cuda.is_available():
        print("cuda present: constructor not expected to fail")
    else:
        try:
            M.LightGCN(conf, train, test, None, **kw)
            raise SystemExit("constructing the reference model without a GPU should have raised")
        except _lib.HgrError as e:
            print("raised:", e)
    """, cwd=str(tmp_path))
    assert "raised:" in out or "cuda present" in out
