"""GPU test (-m gpu): a host path whose set-up fails part-way gives back every byte it had allocated. The handle below asks
for a raw host-path region of 6 x 2 M points x 65535 bytes (about 786 GB): that cudaMalloc fails at once and takes no memory,
after the slot workspace in front of it (about 0.9 GB) has been allocated. The test never asks for memory that exists, so it
does not crowd out other users of the GPU."""
import numpy as np
import pytest
import torch

from cloud_merger_b200 import CloudMerger, CloudMergerError, make_layout
from cloud_merger_b200._lib import CM_E_CUDA

pytestmark = pytest.mark.gpu


def test_failed_host_path_setup_leaves_no_memory_behind(gpu_ok):
    free_before, _ = torch.cuda.mem_get_info(0)
    cloud = np.zeros((1024, 4), np.float32)  # 16-byte records
    cm = CloudMerger(device=0, max_sensors=6, max_points_per_sensor=2_000_000, max_point_step=65535)
    try:
        for _ in range(8):  # every retry sets the host path up again from nothing
            with pytest.raises(CloudMergerError) as e:
                cm.submit_cloud(0, cloud, len(cloud), make_layout())
            assert e.value.code == CM_E_CUDA
    finally:
        cm.close()
    free_after, _ = torch.cuda.mem_get_info(0)
    assert free_before - free_after <= 512 << 20, "%.2f GB of device memory not given back" % ((free_before - free_after) / 1e9)
