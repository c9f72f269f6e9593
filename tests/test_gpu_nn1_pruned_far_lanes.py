"""The pruned NN-1 chain's point stage against the oracle: chunks in which most points have a close nearest neighbour and
a few have a far one.  The far points keep the box stage's bound loose, so the per-point bound of the other lanes is what
skips chunks there; a chunk skipped that one of them needed would change a minimum or an arg-min."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from test_gpu_nn1_pruned import B, FORMS, check, face_pair  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("lift", [0.05, 0.3])
def test_one_far_point_per_chunk(lift):
    adv, ori = face_pair(B, 4096, seed=11)
    rs = np.random.RandomState(int(lift * 100))
    for cloud, start in ((adv, 0), (ori, 16)):
        # every 32nd point of each side leaves the surface: its nearest neighbour on the other side is far, while the
        # points around it (its chunk mates after bucketing) keep close ones
        d = rs.randn(B, cloud.shape[1] // 32, 3).astype(np.float32)
        d /= np.linalg.norm(d, axis=-1, keepdims=True)
        cloud[:, start::32] += np.float32(lift) * d
    check(adv, ori, forms=FORMS)
