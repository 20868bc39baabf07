"""The reference's UNMODIFIED learning/main.py driven on top of superpoint_graph_b200 (VERDICT r1 #8):
compat/run_main.py installs the drop-in mirrors, resolves the packages the image lacks (igraph, h5py,
torchnet, transforms3d) to the stand-ins under compat/, and runpy-executes main.py from the reference
as compiled into oracle/_ref/ by build() (oracle/build_ref.py) on a synthetic S3DIS-layout dataset written by
compat/make_fixture.py.  The repository does not carry the reference's sources: without oracle/_ref both runs skip.

CPU box: `--cuda 0` must get through argument parsing, dataset reading, graph sub-sampling, collate
(`ecc.GraphConvInfo` = ours), model construction (ours) and die at the first forward with the explicit
"CUDA only" error — there is no CPU fallback.  GPU box: one full epoch + test + multi-sample final
evaluation runs for real."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "compat"))


def _have_reference():
    sys.path.insert(0, ROOT)
    from oracle import build_ref
    return build_ref.available()


def _run(tmp_path, cuda, extra=()):
    import make_fixture
    root = str(tmp_path / "s3dis")
    make_fixture.make(root, rooms_per_area=2, n_sp=60, seed=1)
    cmd = [sys.executable, os.path.join(ROOT, "compat", "run_main.py"), "--", "--dataset", "s3dis", "--S3DIS_PATH", root,
           "--cvfold", "5", "--epochs", "1", "--test_nth_epoch", "1", "--test_multisamp_n", "2", "--cuda", str(cuda),
           "--odir", os.path.join(root, "out"), "--nworkers", "0", "--use_pyg", "0", "--batch_size", "2",
           # S3DIS.md:27-30 (model for 13 classes; the script's defaults are Semantic3D's f_8)
           "--model_config", "gru_10_1_1_1_0,f_13", "--ptn_nfeat_stn", "14", "--pc_attribs", "xyzrgbelpsvXYZ"] + list(extra)
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=str(tmp_path))
    return root, out


def test_compat_igraph_semantics():
    import igraph
    G = igraph.Graph(n=5, edges=[[0, 1], [1, 2], [3, 4], [4, 0], [2, 1]], directed=True,
                     edge_attrs={"f": [10, 11, 12, 13, 14]}, vertex_attrs={"v": list(range(5)), "s": [5, 50, 7, 70, 9]})
    assert G.indegree(G.vs, loops=True) == [1, 2, 1, 0, 1]
    S = G.subgraph([4, 0, 1])  # renumbered in increasing order of the old ids: 0->0, 1->1, 4->2
    assert S.vcount() == 3 and S.vs["v"] == [0, 1, 4] and S.get_edgelist() == [(0, 1), (2, 0)] and S.es["f"] == [10, 13]
    P = G.permute_vertices([2, 0, 1, 4, 3])  # vertex i becomes perm[i]
    assert P.vs["v"] == [1, 2, 0, 4, 3] and P.get_edgelist()[0] == (2, 0) and P.es["f"] == G.es["f"]
    assert sorted(G.neighborhood([3], 2)[0]) == [0, 3, 4] and G.neighborhood([3], 1)[0][0] == 3
    sub = G.es[[4, 0]]
    assert sub.get_attribute_values("f") == [14, 10] and G.vs[3]["s"] == 70


@pytest.mark.skipif(not _have_reference(), reason="needs the reference compiled into oracle/_ref (python -m oracle.build_ref)")
def test_main_py_reaches_the_first_forward_without_a_gpu(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU box: the full run is test_main_py_runs_unchanged_one_epoch")
    root, out = _run(tmp_path, cuda=0)
    assert out.returncode != 0
    assert "superpoint_graph_b200 runs on CUDA only" in out.stderr, out.stderr[-3000:]
    assert "learning/main.py" in out.stderr and "ptnCloudEmbedder.run" in out.stderr  # died inside train()
    assert "Train dataset: 10 elements - Test dataset: 2 elements" in out.stdout, out.stdout[-2000:]
    assert "GRUCellEx" in out.stdout and "PointNet" in out.stdout  # print(model): our mirrors were constructed


@pytest.mark.gpu
@pytest.mark.skipif(not _have_reference(), reason="needs the reference compiled into oracle/_ref (python -m oracle.build_ref)")
def test_main_py_runs_unchanged_one_epoch(tmp_path):
    root, out = _run(tmp_path, cuda=1)
    assert out.returncode == 0, out.stderr[-4000:]
    odir = os.path.join(root, "out")
    stats = json.load(open(os.path.join(odir, "trainlog.json")))
    assert len(stats) == 1 and np.isfinite(stats[0]["loss"]) and 0 < stats[0]["loss"] < 10
    assert 0 <= stats[0]["acc_test"] <= 100
    scores = json.load(open(os.path.join(odir, "scores_test.json")))
    assert 0 <= scores[0]["avg_iou_test"] <= 1
    import h5py  # the stand-in (or the real one): predictions of the two test rooms, 0-based classes
    with h5py.File(os.path.join(odir, "predictions_test.h5"), "r") as f:
        names = sorted(f.keys())
        assert names == ["Area_5"]
        pred = f["Area_5"]["office_1"][:]
        assert pred.shape[0] > 50 and pred.min() >= 0 and pred.max() < 13
    assert os.path.exists(os.path.join(odir, "model.pth.tar"))
    assert "[run_main] reference:" in out.stdout
