"""SURVEY.md §8a-5 / §8f-2 (parity-green on a B200): PillarFeatureNet (models/voxel_encoders/pillar_encoder.py:
115-210) with one PFNLayer as one launch over the `hard_voxelize` outputs."""
import numpy as np
import torch

from .._lib import check, host_floats, lib
from .._mem import ptr, require_cuda, stream


def fold_bn(bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, device):
    """BatchNorm1D(eval) as (scale, shift) device tensors, folded on the host in fp64: do this once per model."""
    s = np.asarray(bn_gamma, np.float64) / np.sqrt(np.asarray(bn_var, np.float64) + bn_eps)
    t = np.asarray(bn_beta, np.float64) - np.asarray(bn_mean, np.float64) * s
    return torch.from_numpy(s.astype(np.float32)).to(device), torch.from_numpy(t.astype(np.float32)).to(device)


def pillar_feature_net(voxels, num_points_per_voxel, coors, weight, bn_gamma, bn_beta, bn_mean, bn_var, bn_eps,
                       voxel_size, point_cloud_range, num_voxels=None, folded=None):
    """voxels [n, M, F], counts [n], coors [n, 4] (b, z, y, x) int32, weight [F + 5, C] -> [n, C] pillar features.
    folded: (scale, shift) from fold_bn - pass it to keep host->device copies out of the per-frame path (CUDA graphs)."""
    voxels = require_cuda(voxels, "voxels", torch.float32)
    npv = require_cuda(num_points_per_voxel, "num_points_per_voxel", torch.int32)
    coors = require_cuda(coors, "coors", torch.int32)
    weight = require_cuda(weight, "weight", torch.float32)
    n, m, f = voxels.shape
    c = weight.shape[1]
    if weight.shape[0] != f + 5:
        raise ValueError("weight must be [F + 5, C]")
    dev = voxels.device
    scale, shift = folded if folded is not None else fold_bn(bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, dev)
    out = torch.zeros((n, c), dtype=torch.float32, device=dev)
    nump = ptr(require_cuda(num_voxels, "num_voxels", torch.int32)) if num_voxels is not None else ptr(None)
    check(lib().p3d_pillar_feature_net(ptr(voxels), ptr(npv), ptr(coors), nump, n, m, f, c, ptr(weight), ptr(scale),
                                       ptr(shift), host_floats(voxel_size), host_floats(point_cloud_range), ptr(out),
                                       stream(dev)), "pillar_feature_net")
    return out


def pillar_feature_net_pixel_h16(voxels, num_points_per_voxel, coors, weight, bn_gamma, bn_beta, bn_mean, bn_var, bn_eps,
                                 voxel_size, point_cloud_range, batch, ny, nx, num_voxels=None, folded=None):
    """pillar_feature_net + PointPillarsScatter + nchw_to_pixel_h16 in one launch (after a zero fill of the image):
    returns (image [batch * ny * nx, 2 * C] float16 pixel fp16-pair rows, (batch, ny, nx, C)), the input of
    DenseRPNHead.forward_h16.  Values above fp16's range are saturated and set bit 0 of sparse_nn.status_tensor."""
    from .sparse_nn import status_tensor
    voxels = require_cuda(voxels, "voxels", torch.float32)
    npv = require_cuda(num_points_per_voxel, "num_points_per_voxel", torch.int32)
    coors = require_cuda(coors, "coors", torch.int32)
    weight = require_cuda(weight, "weight", torch.float32)
    n, m, f = voxels.shape
    c = weight.shape[1]
    if weight.shape[0] != f + 5:
        raise ValueError("weight must be [F + 5, C]")
    dev = voxels.device
    scale, shift = folded if folded is not None else fold_bn(bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, dev)
    batch, ny, nx = int(batch), int(ny), int(nx)
    out = torch.empty((batch * ny * nx, 2 * c), dtype=torch.float16, device=dev)
    nump = ptr(require_cuda(num_voxels, "num_voxels", torch.int32)) if num_voxels is not None else ptr(None)
    check(lib().p3d_pillar_feature_net_pixel_h16(ptr(voxels), ptr(npv), ptr(coors), nump, n, m, f, c, ptr(weight),
                                                 ptr(scale), ptr(shift), host_floats(voxel_size),
                                                 host_floats(point_cloud_range), batch, ny, nx, ptr(out),
                                                 ptr(status_tensor(dev)), stream(dev)), "pillar_feature_net_pixel_h16")
    return out, (batch, ny, nx, c)
