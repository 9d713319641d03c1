"""CPU oracle of lattice inference (dpn_decoder_lattice) - TEST INFRASTRUCTURE ONLY.

Composed from the existing oracle pieces: the node coordinates of a regular space-time lattice (fp64, rounded once to fp32 as the
library does), sampler_oracle.trilinear for coord_data, dpn_oracle.encoding_coord / decode_generated for the six nets and
dpn_oracle.inverse_norm(with_clip=False), the de-normalisation of the reference's dense forward (interface_physics.py:533).
"""
import numpy as np
import torch

from oracle import dpn_oracle as O
from oracle import sampler_oracle as SO


def node_coords(lat, k, j, i):
    """x, y, t (float64 arrays holding fp32 values) of nodes (k, j, i) of `lat` (nx, ny, nt, x0, y0, t0, sx, sy, st)."""
    x = (lat.x0 + np.asarray(i, dtype=np.float64) * lat.sx).astype(np.float32).astype(np.float64)
    y = (lat.y0 + np.asarray(j, dtype=np.float64) * lat.sy).astype(np.float32).astype(np.float64)
    t = (lat.t0 + np.asarray(k, dtype=np.float64) * lat.st).astype(np.float32).astype(np.float64)
    return x, y, t


def node_values(coarse, W, x, y, t, dx=27000.0, dy=27000.0, lat_size=145, lon_size=257, pred_t_span=86400.0,
                cells_per_coarse=4.0, t_step=6 * 3600.0, consts=None):
    """Physical values [n, 6] (float64) of one sample at points x, y, t: coarse [Tt,Hc,Wc,6], W a dict of that sample's
    decoder tensors in dpn_oracle layout (W1 [6,256,192], ..., Wd [6,256,192], ...).  consts: the PhysicsConsts whose
    mean / std de-normalise (default: the reference config); the geometry is given by the keywords."""
    cd = torch.from_numpy(SO.trilinear(np.asarray(coarse), x, y, t, dx=dx, dy=dy, cells_per_coarse=cells_per_coarse, t_step=t_step))
    col = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float64)).reshape(-1, 1)
    pe = O.encoding_coord(col(x), col(y), col(t), dx, dy, lat_size, lon_size, pred_t_span)
    with torch.no_grad():
        return torch.cat(O.inverse_norm(O.decode_generated(pe, cd, W), with_clip=False,
                                         norm=O.OBS_NORM if consts is None else O.norm_of(consts)), 1)


def lattice_values(coarse, W, lat, **geom):
    """The whole lattice of one sample: [nt, ny, nx, 6] float64."""
    k, j, i = np.meshgrid(np.arange(lat.nt), np.arange(lat.ny), np.arange(lat.nx), indexing="ij")
    x, y, t = node_coords(lat, k.reshape(-1), j.reshape(-1), i.reshape(-1))
    return node_values(coarse, W, x, y, t, **geom).reshape(lat.nt, lat.ny, lat.nx, 6)
