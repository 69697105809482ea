"""pytorch3d.ops.knn_points for K=1 (forward only), on homogeneous or ragged batches (lengths1 / lengths2: padded
queries and queries whose target cloud is empty get dist 0 and idx 0, as in PyTorch3D)."""
from collections import namedtuple

import ptk_b200

_KNN = namedtuple("KNN", "dists idx knn")


def knn_points(p1, p2, lengths1=None, lengths2=None, K=1, version=-1, return_nn=False, return_sorted=True):
    if K != 1:
        raise NotImplementedError("ptk_b200 knn_points supports K=1")
    dists, idx = ptk_b200.ops.knn1(p1, p2, lengths1, lengths2)
    return _KNN(dists=dists[..., None], idx=idx.long()[..., None], knn=None)
