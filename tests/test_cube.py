"""Gaussian cube output (epnn_b200.cube) on the CPU: header, bohr conversion, value order and line breaks, read back with
a parser written here from the format; esp_cube's slabs with a float64 stand-in for the engine."""
import numpy as np
import pytest

from epnn_b200 import cube
from epnn_b200.engine import BOHR_ANGSTROM
from points_ref import system_ref


def parse_cube(path):
    with open(path) as f:
        lines = f.read().split("\n")
    assert lines[-1] == ""                                              # the file ends with a new line
    head = lines[2].split()
    n_atoms, origin = int(head[0]), np.array([float(v) for v in head[1:4]])
    dims, axes = [], []
    for k in range(3):
        t = lines[3 + k].split()
        dims.append(int(t[0]))
        axes.append([float(v) for v in t[1:4]])
    atoms = [lines[6 + i].split() for i in range(n_atoms)]
    body = lines[6 + n_atoms:-1]
    return dict(comments=lines[:2], origin=origin, dims=dims, axes=np.array(axes), atoms=atoms, body=body)


def values(body):
    return np.array([float(v) for line in body for v in line.split()])


def test_grid_around():
    x = np.array([[0.0, 0.0, 0.0], [1.0, 2.0, 3.0]])
    o, d = cube.grid_around(x, spacing=0.5, margin=1.0)
    assert np.allclose(o, [-1.0, -1.0, -1.0]) and d.tolist() == [7, 9, 11]       # (extent + 2 margin) / spacing + 1
    o, d = cube.grid_around(x, spacing=0.4, margin=1.0)
    assert d.tolist() == [9, 11, 14] and (o + 0.4 * (d - 1) >= x.max(0) + 1.0 - 1e-12).all()   # covers the far faces
    with pytest.raises(ValueError):
        cube.grid_around(x, spacing=0.0)


@pytest.mark.parametrize("nz", [1, 5, 6, 7, 13])
def test_write_cube_layout(tmp_path, nz):
    Z = np.array([8, 1, 1])
    xyz = np.array([[0.0, 0.0, 0.1], [0.76, 0.59, 0.0], [-0.76, 0.59, 0.0]])
    origin, spacing, dims = np.array([-2.0, -1.5, -1.0]), 0.25, (3, 4, nz)
    ix, iy, iz = np.meshgrid(*(np.arange(d) for d in dims), indexing="ij")
    phi = 1.0 + 100.0 * ix + 10.0 * iy + iz + 0.125                     # encodes its own index
    path = tmp_path / "w.cube"
    cube.write_cube(path, Z, xyz, origin, spacing, dims, phi, comment="water\nline")
    c = parse_cube(path)
    assert c["comments"][0] == "water line"
    assert np.allclose(c["origin"], origin / BOHR_ANGSTROM, atol=1e-6)
    assert c["dims"] == list(dims)
    assert np.allclose(c["axes"], np.eye(3) * spacing / BOHR_ANGSTROM, atol=1e-6)
    for a, z, x in zip(c["atoms"], Z, xyz):
        assert int(a[0]) == z and float(a[1]) == float(z)
        assert np.allclose([float(v) for v in a[2:]], x / BOHR_ANGSTROM, atol=1e-6)
    # x slowest, z fastest, 6 per line, a new line after every z row, %13.5E
    per_row = -(-nz // 6)
    assert len(c["body"]) == dims[0] * dims[1] * per_row
    for r in range(dims[0] * dims[1]):
        row = c["body"][r * per_row:(r + 1) * per_row]
        assert [len(line) for line in row] == [13 * min(6, nz - 6 * k) for k in range(per_row)]
    v = values(c["body"])
    assert np.allclose(v, phi.ravel() * BOHR_ANGSTROM, rtol=1e-5, atol=0)
    assert c["body"][0][:13] == "%13.5E" % (phi.flat[0] * BOHR_ANGSTROM)
    with pytest.raises(ValueError):
        cube.write_cube(path, Z, xyz, origin, spacing, dims, phi.ravel()[:-1])


class RefEngine:
    """Stand-in for Engine.potential_points: the float64 reference; records the size of every call."""

    def __init__(self):
        self.calls = []

    def potential_points(self, offsets, xyz, q, point_offsets, points, field=False):
        assert list(offsets) == [0, len(xyz)] and list(point_offsets) == [0, len(points)]
        self.calls.append(len(points))
        return {"phi": system_ref(xyz, q, points)["phi"]}


def test_esp_cube_slabs(tmp_path):
    rng = np.random.default_rng(4)
    xyz = rng.uniform(-1.5, 1.5, size=(6, 3)).astype(np.float32)
    q = rng.normal(scale=0.3, size=6)
    Z = np.array([6, 1, 1, 8, 7, 1])
    eng = RefEngine()
    origin, dims = cube.esp_cube(tmp_path / "a.cube", eng, Z, xyz, q, spacing=0.5, margin=2.0, max_points=2 * 9 * 9 + 5)
    plane = int(dims[1] * dims[2])
    assert max(eng.calls) <= max(plane, 2 * 9 * 9 + 5) and len(eng.calls) == -(-int(dims[0]) // max(1, (2 * 9 * 9 + 5) // plane))
    ix, iy, iz = np.meshgrid(*(np.arange(d) for d in dims), indexing="ij")
    pts = np.stack([ix.ravel(), iy.ravel(), iz.ravel()], 1) * 0.5 + origin
    want = system_ref(xyz, q, pts)["phi"] * BOHR_ANGSTROM
    got = values(parse_cube(tmp_path / "a.cube")["body"])
    assert np.allclose(got, want, rtol=1e-5, atol=1e-12)
    one = RefEngine()
    cube.esp_cube(tmp_path / "b.cube", one, Z, xyz, q, spacing=0.5, margin=2.0)
    assert one.calls == [int(np.prod(dims))]                             # the default slab holds this whole grid
    assert (tmp_path / "a.cube").read_text() == (tmp_path / "b.cube").read_text()
