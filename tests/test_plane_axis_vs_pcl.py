"""The C++ statement of SACMODEL_PERPENDICULAR_PLANE / SACMODEL_PARALLEL_PLANE (tests/plane_axis_oracle.cpp) against the
REAL PCL (tests/plane_axis_pcl_ref.cpp). PCL is not installed in this repository's build image, so these tests SKIP there
and say why; with PCL >= 1.8 they pin the restatement: the inliers and coefficients
must match for at least one sum order."""
import math

import numpy as np
import pytest

import plane_axis as A
import plane_axis_oracle as PO

pytestmark = pytest.mark.skipif(not PO.pcl_available(), reason="real-PCL reference not available: " + PO.pcl_why_not())


@pytest.mark.parametrize("model,eps", [(A.PERP, math.radians(10.0)), (A.PAR, math.radians(10.0)), (A.PERP, 0.0),
                                       (A.PERP, 2.0), (A.PAR, -0.1)])
def test_axis_models_match_pcl(model, eps):
    for x in (A.wall_zone(seed=3), A.walls_only(), A.nan_zone()):
        coeff, inl = PO.pcl_plane_ransac_model(x, 0.3, 0.99, 1000, True, model, A.Z, eps)
        hits = [o for o in (0, 1, 2)
                if np.array_equal(PO.plane_ransac_model(x, 0.3, 0.99, 1000, True, 12345, o, model, A.Z, eps)["inliers"], inl)
                and PO.plane_ransac_model(x, 0.3, 0.99, 1000, True, 12345, o, model, A.Z, eps)["coeff"].tobytes()
                == np.ascontiguousarray(coeff, np.float32).tobytes()]
        assert hits, (model, eps, coeff, len(inl))
