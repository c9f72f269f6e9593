"""B200-native point-set distance path of LI-Yiquan/3DPointCloudAttack.

Hand-written sm_100a CUDA kernels behind a C ABI (include/pcdist.h, libpcdist.so), exposed
through the reference's own Python call surface:

    dis_utils_torch   <- utils/dis_utils_torch.py
    distance          <- attack/CW/CW_utils/distance.py  (+ Gen3DAdv copy)
    set_distance      <- attack/SIadv/utils/set_distance.py
    dist_utils        <- attack/CW/CW_utils/dist_utils.py (ChamferDist, HausdorffDist, KNNDist, ChamferkNNDist)
    knn_utils         <- attack/GeoA3/knn_utils.py
    loss_utils        <- attack/GeoA3/loss_utils.py (the knn_points consumers and the brute-force k-NN losses)
    utility           <- attack/GeoA3/utility.py (estimate_normal, estimate_perpendicular, ...)
    taof              <- attack/AOF/TAOF_attack.py (knn, get_Laplace_from_pc)
    dgcnn             <- model/dgcnn.py (knn, get_graph_feature)
    curvenet_util     <- model/curvenet_util.py (knn, normal_knn)
    pointnet2_utils   <- model/pointnet2_utils.py (square_distance, query_ball_point)
    defense           <- attack/SIadv/baselines/defense/drop_points/SOR.py (SORDefense; float64, no install() patch)
    metrics           <- utils/dis_utils_numpy.py (float64 Chamfer / Hausdorff for reporting; no install() patch)

`install.install()` patches these into an importable copy of the reference.  The package
directory name starts with a digit; import it with importlib or through the `pcdist` alias
module at the repository root.
"""
from . import _lib, functional  # noqa: F401
from . import (curvenet_util, cw_loop, defense, dgcnn, dis_utils_torch, dist_utils, distance, geoa3_loop, graph, install,  # noqa: F401
               knn_utils, loss_utils, metrics, pointnet2_utils, set_distance, taof, utility)

__version__ = "0.1.0"
