"""Gaussian cube files of the electrostatic potential of a system's charges (an ESP map to colour a molecular surface
in VMD, PyMOL or ChimeraX).

The potential comes from :meth:`epnn_b200.engine.Engine.potential_points` (FP64 on the GPU).  The file follows the
Gaussian cube layout: two comment lines; the atom count and the origin; the three axis lines (point count and step);
one line per atom (Z, Z as the nuclear charge, position); then the values with x slowest and z fastest, six per line,
each ``%13.5E``, and a new line after every z row.  Distances are in bohr and values in atomic units (e/bohr), as
viewers expect.
"""
from __future__ import annotations

import numpy as np

from .engine import BOHR_ANGSTROM


def grid_around(xyz, spacing: float = 0.3, margin: float = 4.0):
    """Axis-aligned grid that covers the atoms ``xyz`` (A) plus ``margin`` A on every side, with ``spacing`` A between
    points.  Returns ``(origin (3,) float64 in A, dims (3,) int64)``."""
    if not spacing > 0 or not margin >= 0:
        raise ValueError("spacing must be positive and margin non-negative")
    x = np.asarray(xyz, np.float64).reshape(-1, 3)
    lo, hi = x.min(0) - margin, x.max(0) + margin
    dims = np.ceil((hi - lo) / spacing - 1e-9).astype(np.int64) + 1
    return lo, dims


def _plane_points(origin, spacing, dims, i0, i1):
    """Points of the x planes [i0, i1) of the grid, x slowest and z fastest, float64 (k * ny * nz, 3)."""
    ix, iy, iz = np.meshgrid(np.arange(i0, i1), np.arange(dims[1]), np.arange(dims[2]), indexing="ij")
    return np.stack([ix.ravel(), iy.ravel(), iz.ravel()], 1) * float(spacing) + np.asarray(origin, np.float64)


def _write_header(f, Z, xyz, origin, spacing, dims, comment):
    Z = np.asarray(Z).astype(np.int64).reshape(-1)
    x = np.asarray(xyz, np.float64).reshape(-1, 3) / BOHR_ANGSTROM
    o = np.asarray(origin, np.float64) / BOHR_ANGSTROM
    h = float(spacing) / BOHR_ANGSTROM
    lines = [comment.replace("\n", " "), "phi in e/bohr (atomic units), x slowest, z fastest",
             f"{len(Z):5d}{o[0]:12.6f}{o[1]:12.6f}{o[2]:12.6f}"]
    for k in range(3):
        step = [0.0, 0.0, 0.0]
        step[k] = h
        lines.append(f"{int(dims[k]):5d}{step[0]:12.6f}{step[1]:12.6f}{step[2]:12.6f}")
    lines += [f"{z:5d}{float(z):12.6f}{p[0]:12.6f}{p[1]:12.6f}{p[2]:12.6f}" for z, p in zip(Z.tolist(), x)]
    f.write("\n".join(lines) + "\n")


def _write_values(f, phi, nz):
    """phi: values in e/A of whole z rows, in file order."""
    v = np.asarray(phi, np.float64).reshape(-1) * BOHR_ANGSTROM
    row = ("%13.5E" * 6 + "\n") * (nz // 6) + ("%13.5E" * (nz % 6) + "\n" if nz % 6 else "")
    f.write((row * (v.size // nz)) % tuple(v.tolist()))


def write_cube(path, Z, xyz, origin, spacing, dims, phi, comment: str = "epnn_b200 electrostatic potential"):
    """Writes a cube file.  ``Z``: atomic numbers; ``xyz``, ``origin``, ``spacing`` in A; ``dims`` = (nx, ny, nz);
    ``phi``: nx * ny * nz values in e/A, x slowest and z fastest (any shape with that order)."""
    dims = np.asarray(dims, np.int64)
    phi = np.asarray(phi, np.float64).reshape(-1)
    if phi.size != int(np.prod(dims)):
        raise ValueError(f"phi has {phi.size} values, the grid {tuple(dims.tolist())} needs {int(np.prod(dims))}")
    with open(path, "w") as f:
        _write_header(f, Z, xyz, origin, spacing, dims, comment)
        _write_values(f, phi, int(dims[2]))


def esp_cube(path, engine, Z, xyz, q, spacing: float = 0.3, margin: float = 4.0, max_points: int = 1 << 22,
             comment: str = "epnn_b200 electrostatic potential"):
    """Writes the potential of one system's charges ``q`` (e) on the grid of :func:`grid_around` to a cube file.  The grid
    is evaluated through ``engine.potential_points`` (an :class:`~epnn_b200.engine.Engine` or a ``charge_gn.Model``) in
    slabs of whole x planes of at most ``max_points`` points (at least one plane), so host memory stays bounded for
    large grids.  Returns ``(origin, dims)``."""
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    q = np.ascontiguousarray(q, np.float64).reshape(-1)
    origin, dims = grid_around(xyz, spacing, margin)
    plane = int(dims[1] * dims[2])
    step = max(1, int(max_points) // plane)
    offs = np.array([0, len(xyz)], np.int32)
    with open(path, "w") as f:
        _write_header(f, Z, xyz, origin, spacing, dims, comment)
        for i0 in range(0, int(dims[0]), step):
            i1 = min(int(dims[0]), i0 + step)
            pts = _plane_points(origin, spacing, dims, i0, i1)
            phi = engine.potential_points(offs, xyz, q, np.array([0, len(pts)], np.int64), pts)["phi"]
            _write_values(f, phi, int(dims[2]))
    return origin, dims
