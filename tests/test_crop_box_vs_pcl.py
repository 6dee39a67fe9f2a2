"""The C++ CropBox oracle (tests/crop_box_oracle.cpp) against the REAL pcl::CropBox (tests/crop_box_pcl_ref.cpp), on the edge
clouds and known answers of the CropBox tests. Where PCL is not installed (this repository's build image) these tests SKIP
and say why; where pkg-config finds PCL >= 1.8 the wrapper is built on first use."""
import numpy as np
import pytest

import crop_box_cases as K
import crop_box_oracle as O

pytestmark = pytest.mark.skipif(not O.pcl_available(), reason="real-PCL CropBox not available: " + O.pcl_why_not())


@pytest.mark.parametrize("name", sorted(K.BOXES))
@pytest.mark.parametrize("is_dense", [1, 0])
def test_crop_box_edge_clouds(name, is_dense):
    b = K.BOXES[name]
    x = K.edge_cloud(7 + len(name), b)
    assert np.array_equal(O.crop_box(x, bool(is_dense), b), O.pcl_crop_box(x, bool(is_dense), b)), "CropBox %s differs" % name


def test_crop_box_known_answers():
    for c in K.golden():
        assert O.pcl_crop_box(c["xyzi"], bool(c["is_dense"]), c["box"]).tolist() == c["kept"], c["name"]
