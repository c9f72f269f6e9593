"""CPU-only checks: the C-ABI library builds, loads and exports exactly what include/pcdist.h
declares; the product path fails loudly without CUDA; host-side logic (installer, sharding)."""
import importlib
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pcd = importlib.import_module("3dpointcloudattack_b200")


def header_symbols():
    src = open(os.path.join(ROOT, "include", "pcdist.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pcd_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = pcd._lib.load()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), s
    assert sorted(pcd._lib.SIGNATURES) == syms           # the ctypes table covers the header, no more no less
    out = subprocess.check_output(["nm", "-D", "--defined-only", pcd._lib.LIB_PATH], text=True)
    exported = sorted(set(re.findall(r" T (pcd_[a-z0-9_]+)", out)))
    assert exported == syms
    assert lib.pcd_version() == 203


def test_library_is_sm100a_and_uses_blackwell_instructions():
    out = subprocess.run(["cuobjdump", "-sass", pcd._lib.LIB_PATH], capture_output=True, text=True).stdout
    if not out:
        pytest.skip("cuobjdump not available")
    assert "sm_100a" in out
    for mnemonic in ("FFMA2", "FADD2", "FMUL2", "FMNMX3", "CREDUX", "UBLKCP"):
        assert mnemonic in out, mnemonic


def test_workspace_sizes_without_gpu():
    lib = pcd._lib.load()
    assert lib.pcd_nn1_workspace_bytes(32, 4096, 4096, 0) >= 32 * 4096 * (16 + 16 + 8 + 8)
    assert lib.pcd_nn1_workspace_bytes(0, 1, 1, 0) == 0
    assert lib.pcd_knn_workspace_bytes(2, 100, 100, 3, 5) > 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-box behaviour")
def test_no_cpu_fallback():
    a = torch.zeros(1, 8, 3)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.distance.chamfer(a, a)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.knn_utils.knn_points(a, a, K=2)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.pointnet2_utils.query_ball_point(0.2, 4, a, a)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.dgcnn.knn(a.transpose(1, 2), 2)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.dgcnn.get_graph_feature(a.transpose(1, 2).contiguous(), k=2, idx=torch.zeros(1, 8, 2, dtype=torch.long))
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.pointnet2_utils.farthest_point_sample(a, 4)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.curvenet_util.farthest_point_sample(a, 4)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.cw_loop.CWAttack(torch.nn.Identity(), None, None).attack(a, torch.zeros(1))
    with pytest.raises(ValueError, match="pinned"):
        pcd.graph.PipelinedLoss(lambda x, y: (x.sum(), ()), a, a)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.utility.estimate_normal(a.transpose(1, 2), 3)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.loss_utils._get_kappa_ori(a.transpose(1, 2), a.transpose(1, 2), 2)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.dist_utils.KNNDist(k=2)(a)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.taof.get_Laplace_from_pc(a.transpose(1, 2))
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.geoa3_loop.GeoA3Attack(torch.nn.Identity(), classes=3).attack(a, torch.zeros(1))


def test_clip_epilogues_have_no_cpu_fallback():
    """The fused clip / projection epilogues (functional.clip_points_, lp_clip, offset_proj, find_offset and the loop-level
    wrappers) refuse CPU tensors like every other entry of the path."""
    a = torch.zeros(1, 3, 8)
    for call in (lambda: pcd.functional.clip_points_(a, a, 0.1), lambda: pcd.functional.lp_clip(a, 0.1),
                 lambda: pcd.geoa3_loop.lp_clip(a, 0.1), lambda: pcd.cw_loop.ClipPointsLinf(0.1)(a, a),
                 lambda: pcd.cw_loop.ClipPointsL2(0.1)(a, a), lambda: pcd.cw_loop.ProjectInnerClipLinf(0.1)(a, a, a),
                 lambda: pcd.functional.offset_proj(a, a, torch.zeros(1, 8, dtype=torch.long)),
                 lambda: pcd.functional.find_offset(a, a, torch.zeros(1, 8, dtype=torch.long))):
        with pytest.raises(RuntimeError, match="CUDA only"):
            call()
    with pytest.raises(ValueError):
        pcd.functional.clip_points_(torch.zeros(1, 8, 3), torch.zeros(1, 8, 3), 0.1)      # not channel-first


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "3dpointcloudattack_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("the oracle", "").replace("CPU oracle", ""), f


def test_signatures_mirror_the_reference():
    import inspect
    assert list(inspect.signature(pcd.knn_utils.knn_points).parameters) == [
        "p1", "p2", "lengths1", "lengths2", "K", "version", "return_nn", "return_sorted"]
    assert list(inspect.signature(pcd.knn_utils.knn_gather).parameters) == ["x", "idx", "lengths"]
    assert list(inspect.signature(pcd.pointnet2_utils.query_ball_point).parameters) == ["radius", "nsample", "xyz", "new_xyz"]
    assert list(inspect.signature(pcd.dist_utils.ChamferkNNDist.__init__).parameters) == [
        "self", "chamfer_method", "knn_k", "knn_alpha", "chamfer_weight", "knn_weight"]
    assert list(inspect.signature(pcd.dist_utils.KNNDist.forward).parameters) == ["self", "pc", "weights", "batch_avg"]
    assert list(inspect.signature(pcd.dist_utils.ChamferDist.forward).parameters) == ["self", "adv_pc", "ori_pc", "weights", "batch_avg"]
    assert list(inspect.signature(pcd.dgcnn.get_graph_feature).parameters) == ["x", "k", "idx"]
    assert list(inspect.signature(pcd.utility.estimate_normal).parameters) == ["pc", "k"]
    assert list(inspect.signature(pcd.utility.estimate_perpendicular).parameters) == ["pc", "k", "sigma", "clip"]
    assert list(inspect.signature(pcd.geoa3_loop.offset_proj).parameters) == ["offset", "ori_pc", "ori_normal", "project"]
    assert list(inspect.signature(pcd.geoa3_loop.lp_clip).parameters) == ["offset", "cc_linf"]
    assert list(inspect.signature(pcd.loss_utils.displacement_loss).parameters) == ["adv_pc", "ori_pc", "k"]
    assert list(inspect.signature(pcd.loss_utils.repulsion_loss).parameters) == ["pc", "k", "h"]
    assert list(inspect.signature(pcd.taof.get_Laplace_from_pc).parameters) == ["ori_pc"]
    for fn in ("euclidean_distances", "pairwise_distances", "chamfer", "sgd_hausdorff_dis", "bid_hausdorff_dis"):
        assert callable(getattr(pcd.dis_utils_torch, fn))


# A stand-in for the reference checkout: its package layout, module names and the names install() patches or must leave
# alone, with placeholder bodies. dist_utils binds chamfer / hausdorff at import time, as dist_utils.py:6 does.
REFERENCE_STUB = {
    "utils/dis_utils_torch.py": "def chamfer(a, b): pass\ndef sgd_hausdorff_dis(a, b): pass\ndef bid_hausdorff_dis(a, b): pass\n",
    "attack/CW/CW_utils/distance.py": "class ChamferDistance: pass\nclass HausdorffDistance: pass\n"
                                      "chamfer = ChamferDistance()\nhausdorff = HausdorffDistance()\n",
    "attack/CW/CW_utils/dist_utils.py": "from attack.CW.CW_utils.distance import chamfer, hausdorff\n"
                                        "class L2Dist: pass\nclass ChamferDist: pass\nclass HausdorffDist: pass\n"
                                        "class KNNDist: pass\nclass ChamferkNNDist: pass\n",
    "attack/CW/CW_utils/clip_utils.py": "class ClipPointsL2: pass\nclass ClipPointsLinf: pass\n"
                                        "class ProjectInnerPoints: pass\nclass ProjectInnerClipLinf: pass\n",
    "attack/GeoA3/knn_utils.py": "def knn_points(p1, p2, lengths1=None, lengths2=None, K=1): pass\n"
                                 "def knn_gather(x, idx, lengths=None): pass\n",
    "attack/AOF/TAOF_attack.py": "def knn(x, k): pass\ndef get_Laplace_from_pc(ori_pc): pass\n",
    "model/dgcnn.py": "def knn(x, k): pass\ndef get_graph_feature(x, k=20, idx=None): pass\n",
    "model/pointnet2_utils.py": "def query_ball_point(radius, nsample, xyz, new_xyz): pass\n"
                                "def farthest_point_sample(xyz, npoint): pass\n",
}


def test_install_patches_reference_modules(tmp_path):
    for rel, src in REFERENCE_STUB.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(src)
    for pkg in [d for d in tmp_path.rglob("*") if d.is_dir()]:
        (pkg / "__init__.py").touch()
    sys.path.insert(0, str(tmp_path))
    try:
        rep = pcd.install.install(modules=["utils.dis_utils_torch", "attack.CW.CW_utils.distance",
                                           "attack.CW.CW_utils.dist_utils", "attack.GeoA3.knn_utils",
                                           "model.dgcnn", "model.pointnet2_utils", "attack.AOF.TAOF_attack",
                                           "attack.CW.CW_utils.clip_utils"])
        assert all(v == "patched" for v in rep.values()), rep
        import attack.CW.CW_utils.clip_utils as CU
        assert CU.ClipPointsLinf is pcd.cw_loop.ClipPointsLinf and CU.ProjectInnerClipLinf is pcd.cw_loop.ProjectInnerClipLinf
        assert hasattr(CU, "ProjectInnerPoints")
        import attack.AOF.TAOF_attack as TA
        assert TA.get_Laplace_from_pc is pcd.taof.get_Laplace_from_pc and TA.knn is pcd.dgcnn.knn
        import attack.CW.CW_utils.dist_utils as DU
        import attack.CW.CW_utils.distance as CD
        import model.dgcnn as MD
        assert CD.chamfer is pcd.distance.chamfer and DU.chamfer is pcd.distance.chamfer
        assert DU.ChamferDist is pcd.dist_utils.ChamferDist and MD.knn is pcd.dgcnn.knn
        assert hasattr(DU, "L2Dist")                       # untouched names stay the reference's
    finally:
        sys.path.remove(str(tmp_path))
        for m in [m for m in sys.modules if m.split(".")[0] in ("attack", "model", "utils")]:
            del sys.modules[m]


def test_pipelined_loss_slice_layout():
    """graph.tapered_edges: slices cover the batch exactly once, every slice is non-empty, the first one is the short one."""
    g = importlib.import_module("3dpointcloudattack_b200.graph")
    assert g.tapered_edges(32, 3) == [0, 8, 20, 32]
    assert g.tapered_edges(32, 1) == [0, 32]
    for B in (1, 2, 3, 5, 10, 32, 33, 257):
        for chunks in (1, 2, 3, 4, 8, 300):
            e = g.tapered_edges(B, chunks)
            assert e[0] == 0 and e[-1] == B and len(e) == min(chunks, B) + 1
            sizes = [b - a for a, b in zip(e[:-1], e[1:])]
            assert min(sizes) >= 1
            if B >= 4 * chunks:
                assert sizes[0] == min(sizes)
