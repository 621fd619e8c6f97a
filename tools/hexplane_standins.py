"""PyTorch stand-ins for the reference's HexPlane field, shared by tests/test_hexplane_channels.py and
tools/time_hexplane_channels.py (so that what the profile times and what the test checks are the same modules).

  * TorchGrid: the reference's grid (oracle/field_torch.py hexplane_features: F.grid_sample on contiguous [1, C, H, W]
    planes) on copies of a b200gs.field.HexPlaneField's planes, in a chosen dtype.
  * StandInDeformation: the shape of the reference's scene/deformation.py Deformation under arguments/dynerf/default.py --
    a grid, a width-128 feature_out and five ReLU -> Linear -> ReLU -> Linear heads -- over either grid.
"""
import torch.nn as nn


class TorchGrid(nn.Module):
    def __init__(self, f, dtype):
        super().__init__()
        self.levels = len(f.grids)
        self.aabb = f.aabb.detach().to(dtype)
        self.planes = nn.ParameterList([nn.Parameter(p.detach().to(dtype).contiguous()) for p in f._planes()])
        self.feat_dim = f.feat_dim

    def forward(self, pts, t):
        from oracle import field_torch
        return field_torch.hexplane_features(pts, t, self.aabb, list(self.planes), self.levels)


class StandInDeformation(nn.Module):
    """Every head's output is returned.  Like the reference's deform_network, forward takes the [P, 63] positional
    encoding and hands the grid its first three columns (a fresh slice per call)."""
    HEADS = (("pos_deform", 3), ("scales_deform", 3), ("rotations_deform", 4), ("opacity_deform", 1), ("shs_deform", 48))

    def __init__(self, grid, W=128):
        super().__init__()
        self.grid = grid
        self.feature_out = nn.Sequential(nn.Linear(grid.feat_dim, W))
        for name, k in self.HEADS:
            setattr(self, name, nn.Sequential(nn.ReLU(), nn.Linear(W, W), nn.ReLU(), nn.Linear(W, k)))

    def forward(self, emb, t):
        hidden = self.feature_out(self.grid(emb[:, :3], t[:, :1]))
        return [getattr(self, name)(hidden) for name, _ in self.HEADS]

    def copy_mlp_from(self, other):
        for name, _ in self.HEADS + (("feature_out", 0),):
            getattr(self, name).load_state_dict(getattr(other, name).state_dict())
        return self
