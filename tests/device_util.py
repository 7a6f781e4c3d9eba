"""Reading libvgl's device memory from the tests (VGL_HOST_NONE batches) -- test infrastructure."""
import numpy as np
import torch


def device_plane(ptr, typestr, n):
    """a copy of n elements of a device plane, taken through its CUDA array interface"""
    if not ptr:
        return None
    dt = np.dtype(typestr)
    if n == 0:
        return np.zeros(0, dt)

    class Plane:
        __cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (ptr, False), "version": 3}
    return torch.as_tensor(Plane(), device="cuda").clone().cpu().numpy()


def device_gather(ptr, typestr, idx):
    """plane[idx] of a device plane (int64 element indices), without copying the whole plane to the host"""
    if not ptr:
        return None
    idx = np.asarray(idx, np.int64)
    if idx.size == 0:
        return np.zeros(0, np.dtype(typestr))

    class Plane:
        __cuda_array_interface__ = {"shape": (int(idx.max()) + 1,), "typestr": typestr, "data": (ptr, False), "version": 3}
    t = torch.as_tensor(Plane(), device="cuda")
    return t[torch.from_numpy(idx).cuda()].cpu().numpy()
