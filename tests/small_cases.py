"""A seeded batch of small systems (<= 48 atoms) built from explicit coordinates at the edges of the bundle kernels.

Shared by the CPU emulation of the row-run GNN bundle kernel (tests/test_emu_bundle_run.py) and the GPU comparison of
every small-system kernel set with the float64 oracle (tests/test_gpu_small_reference.py).

Small systems are packed greedily into bundles of at most 48 atoms (whole systems, in batch order; run_chunk in
epnn_api.cu).  The batch is written as a list of intended bundles; a 48-atom system between two of them keeps them
apart.  ``small_batch`` asserts that the greedy packing gives exactly the intended bundles, and ``edge_counts`` measures
from the oracle's own neighbour sets that each edge named below really occurs:

  * maximal near list: 48 atoms in a ball of diameter < 2.99 A (47 near neighbours per row, 2 256 near slots, a full
    48-bit mask per row);
  * empty near list: atoms on a 3.5 A lattice (every column is far);
  * J = 1 with rows over several lanes: systems of 1 to 6 atoms, each alone in its bundle, npad = n and npad > n;
  * list lengths around the warp: bundles whose near list (always even: both directions) has 30, 32, 34, 64 or 66 slots
    and whose far list (dedup_far 0) has 31, 32, 33, 64 or 65 slots;
  * bundle capacity: 48 one-atom systems, one 48-atom system, 47 + 1, 24 + 24;
  * pad weights: npad = n, n + 1, 41, 255, 1 000, and bundles whose systems have different npad - n;
  * distance edges: coincident atoms (D = 0) and pairs with 2.994 A < D < 3 A (e != 0 but not near: in the GNN's
    neighbour set, not in the electron-passing one);
  * species: a system of one species only, a system holding every species of the table, the highest species index.
"""
import numpy as np

from oracle import epnn_oracle as O

BUNDLE_ATOMS = 48
LATTICE = 3.5                     # > 3 A: no two atoms of a lattice system interact
BALL = 2.9                        # diameter of a near cluster: every pair is near (is_near holds to about 2.994 A)
FAR_NOT_NEAR = (2.9945, 2.997, 2.9995)


def ball(rng, n, diameter=BALL, dmin=0.35):
    """n points in a ball of the given diameter, no two closer than dmin."""
    pts = []
    while len(pts) < n:
        p = rng.uniform(-0.5, 0.5, 3) * diameter
        if np.linalg.norm(p) <= diameter / 2 and all(np.linalg.norm(p - q) >= dmin for q in pts):
            pts.append(p)
    return np.array(pts).reshape(n, 3)


def lattice(n, spacing=LATTICE):
    side = int(np.ceil(n ** (1 / 3)))
    g = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3)
    return g[:n] * spacing


def clusters(rng, sizes):
    """Near clusters of the given sizes, 8 A apart (nothing interacts across clusters)."""
    return np.concatenate([ball(rng, k) + np.array([8.0 * c, 0.0, 0.0]) for c, k in enumerate(sizes)])


def molecule(rng, n):
    """A jittered 1.4 A lattice: near pairs, far pairs and varied degrees, like a small organic molecule."""
    return lattice(n, 1.4) + rng.normal(scale=0.1, size=(n, 3))


def small_cases(n_x, seed=0):
    """[(label, [system, ...]), ...]: intended bundles; a system is (xyz, species, Q, npad)."""
    rng = np.random.default_rng(seed)
    n_sp = n_x - 1                                                    # species of the table: 0 .. n_x - 2
    top = n_sp - 1

    def sp(n, pool=None):
        return rng.integers(0, n_sp, size=n) if pool is None else rng.choice(pool, size=n)

    def sys_(xyz, species=None, npad=None, Q=None):
        n = len(xyz)
        species = sp(n) if species is None else np.asarray(species)
        Q = float(rng.integers(-1, 2)) if Q is None else Q
        return (np.asarray(xyz, np.float64), species.astype(np.int32), Q, n if npad is None else int(npad))

    # two coincident atoms (D = 0) and three pairs at 2.994 A < D < 3 A, 5 A apart
    d1, d2, d3 = FAR_NOT_NEAR
    edge = np.array([[0, 0, 0], [0, 0, 0], [d1, 0, 0], [0, 5, 0], [d2, 5, 0], [0, 10, 0], [d3, 10, 0]], np.float64)
    bundles = [
        ("ball48", [sys_(ball(rng, 48), npad=48)]),
        ("single1", [sys_(np.zeros((1, 3)), npad=1)]),
        ("lattice48", [sys_(lattice(48), npad=49)]),
        ("pair_pad", [sys_(ball(rng, 2), npad=41)]),
        ("ball48_pad", [sys_(ball(rng, 48), npad=1000)]),
        ("cluster3", [sys_(ball(rng, 3), npad=3)]),
        ("mol48", [sys_(molecule(rng, 48), npad=48)]),
        ("cluster4_pad", [sys_(ball(rng, 4), npad=5)]),
        ("lattice48_b", [sys_(lattice(48), npad=48)]),
        ("cluster5", [sys_(ball(rng, 5), npad=5)]),
        ("ball48_b", [sys_(ball(rng, 48), species=np.full(48, top), npad=255)]),
        ("cluster6_pad", [sys_(ball(rng, 6), npad=41)]),
        ("mol48_b", [sys_(molecule(rng, 48), npad=60)]),
        # near-list lengths 30 / 32 / 34 / 64 / 66 (cluster k: k (k - 1) ordered slots); the next bundle starts with > 48 - n atoms
        ("near30", [sys_(clusters(rng, [6]), npad=6)]),
        ("mol48_c", [sys_(molecule(rng, 48), npad=48)]),
        ("near32", [sys_(clusters(rng, [5, 4]), npad=12)]),
        ("lattice48_c", [sys_(lattice(48), npad=48)]),
        ("near34", [sys_(clusters(rng, [6, 2, 2]), npad=10)]),
        ("mol48_d", [sys_(molecule(rng, 48), npad=50)]),
        ("near64", [sys_(clusters(rng, [7, 5]), npad=12), sys_(ball(rng, 2), npad=2)]),
        ("ball48_c", [sys_(ball(rng, 48), npad=48)]),
        ("near66", [sys_(clusters(rng, [8, 3, 2, 2]), npad=15)]),
        ("mol48_e", [sys_(molecule(rng, 48), npad=48)]),
        # far-list lengths (dedup_far 0: n^2 per unpadded lattice system, n^2 + n padded) 31 / 32 / 33 / 64 / 65
        ("far31", [sys_(lattice(5), npad=5), sys_(lattice(2), npad=3)]),
        ("lattice48_d", [sys_(lattice(48), npad=48)]),
        ("far32", [sys_(lattice(4), npad=4), sys_(lattice(4), npad=4)]),
        ("mol48_f", [sys_(molecule(rng, 48), npad=48)]),
        ("far33", [sys_(lattice(5), npad=5), sys_(lattice(2), npad=2), sys_(lattice(2), npad=2)]),
        ("ball48_d", [sys_(ball(rng, 48), npad=48)]),
        ("far64", [sys_(lattice(8), npad=8)]),
        ("mol48_g", [sys_(molecule(rng, 48), npad=48)]),
        ("far65", [sys_(lattice(8), npad=8), sys_(np.zeros((1, 3)), npad=1)]),
        ("lattice48_e", [sys_(lattice(48), npad=48)]),
        # bundle capacity
        ("ones48", [sys_(np.zeros((1, 3)), npad=[1, 2, 41, 255][k % 4]) for k in range(48)]),
        ("m47_1", [sys_(molecule(rng, 47), npad=47), sys_(np.zeros((1, 3)), npad=41)]),
        ("m24_24", [sys_(molecule(rng, 24), npad=25), sys_(molecule(rng, 24), npad=24)]),
        # pad weights that differ inside one bundle: npad - n = 0, 1, 41 - n, 255 - n, 1000 - n
        ("pads", [sys_(molecule(rng, 9), npad=9), sys_(ball(rng, 7), npad=8), sys_(molecule(rng, 12), npad=41),
                  sys_(lattice(6), npad=255), sys_(molecule(rng, 10), npad=1000)]),
        ("mol48_h", [sys_(molecule(rng, 48), npad=48)]),
        # distance edges: coincident atoms, pairs just inside the cutoff but not near; one species only; every species
        ("edges", [sys_(edge, npad=9), sys_(molecule(rng, 12), species=np.full(12, 0), npad=12),
                   sys_(molecule(rng, 2 * n_sp), species=np.tile(np.arange(n_sp), 2), npad=41)]),
        ("mol48_i", [sys_(molecule(rng, 48), species=sp(48, [top, 0, 1]), npad=48)]),
    ]
    return bundles


def small_batch(n_x, seed=0):
    """(offs, xyz, sp, Q, npad, labels): the packed batch of ``small_cases``; labels[b] names bundle b.  Asserts that the
    greedy bundle packing of run_chunk gives exactly the intended bundles."""
    bundles = small_cases(n_x, seed)
    systems = [s for _, b in bundles for s in b]
    offs = np.concatenate([[0], np.cumsum([len(s[0]) for s in systems])]).astype(np.int32)
    xyz = np.concatenate([s[0] for s in systems]).astype(np.float32)
    sp = np.concatenate([s[1] for s in systems]).astype(np.int32)
    Q = np.array([s[2] for s in systems], np.float32)
    npad = np.array([s[3] for s in systems], np.int32)
    assert (npad >= np.diff(offs)).all() and np.diff(offs).max() <= BUNDLE_ATOMS
    want, a = [], 0
    for _, b in bundles:
        n = sum(len(s[0]) for s in b)
        want.append((a, n))
        a += n
    assert pack_bundles(offs) == want
    return offs, xyz, sp, Q, npad, [lab for lab, _ in bundles]


def pack_bundles(offs):
    """(first atom, atom count) of every bundle: greedy runs of whole systems with <= 48 atoms (run_chunk)."""
    out, cur0, cur_n = [], 0, 0
    for s in range(len(offs) - 1):
        n = int(offs[s + 1] - offs[s])
        if cur_n and cur_n + n > BUNDLE_ATOMS:
            out.append((cur0, cur_n))
            cur_n = 0
        if not cur_n:
            cur0 = int(offs[s])
        cur_n += n
    if cur_n:
        out.append((cur0, cur_n))
    return out


def edge_counts(offs, xyz, npad):
    """Per bundle, from the oracle's descriptors: near slots (ordered is_near pairs), GNN neighbour slots (ordered e != 0
    pairs), far slots of the plain far list (non-neighbour columns incl. self + one pad slot per padded row), the largest
    degree, and over the batch the count of coincident pairs and of pairs with e != 0 that are not near."""
    out = []
    coincident = far_not_near = 0
    for b0, bn in pack_bundles(offs):
        near = nbr = far = maxdeg = 0
        for s in np.nonzero((offs[:-1] >= b0) & (offs[:-1] < b0 + bn))[0]:
            x = xyz[offs[s]:offs[s + 1]]
            n = len(x)
            e, _ = O.get_init_edges(x)
            D = O.distance_matrix(x)
            emax = e.max(-1)
            off_diag = ~np.eye(n, dtype=bool)
            is_nbr = (D < 3.0) & off_diag
            is_near = (emax > np.float32(1e-5)) & off_diag
            near += int(is_near.sum()); nbr += int(is_nbr.sum())
            far += int(n * n - is_nbr.sum()) + (n if npad[s] > n else 0)
            maxdeg = max(maxdeg, int(is_near.sum(1).max()))
            coincident += int(((D == 0) & off_diag).sum()) // 2
            far_not_near += int((is_nbr & ~is_near & (emax > 0)).sum()) // 2
        out.append(dict(near=near, nbr=nbr, far=far, maxdeg=maxdeg))
    return out, coincident, far_not_near
