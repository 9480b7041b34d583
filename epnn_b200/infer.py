"""``infer.py``-compatible command line (reference ``infer.py:37-79``).

Defaults equal the literals of the reference script (``h_dim=48, e_dim=48, layers=[32,32], T=5, n_elems=9,
./models/decay_model_weights``); ``T`` and ``n_elems`` are re-read from the checkpoint.  Like the reference it writes
``test_names.npy`` and prints per-call seconds, ``avg inference time`` and ``avg feature time``; unlike the reference
(whose ``repeats`` is undefined and whose predictions are only kept in a list) it takes ``--repeats`` and ``--out``.

    python -m epnn_b200.infer --path data/mixed/ --weights models/decay_model_weights --out preds.npy
"""
from __future__ import annotations

import argparse
import os
import time

import numpy as np

from . import charge_gn, xyzio
from .checkpoint import load_weights

model = None       # module-global like the reference (infer.py:56)


def test_step(h, e, x, q, y, mask):
    """Reference ``infer.py:32-35``: forward only (``y`` is unused)."""
    return model([h, e, x, q, mask])


def save_electrostatics(path, model, base, stems, offsets, xyz, q64):
    """``--elst``: Coulomb energy and dipole of every system, and for the dimers that carry a ``<stem>splits.npy`` the
    energy between the two monomers and the charge of the first one, from the FP64 charges of the run."""
    from .engine import COULOMB_KCAL, DEBYE_PER_E_ANGSTROM
    split = xyzio.read_splits(base, stems)
    full = model.electrostatics(offsets, xyz, q64)
    inter = model.electrostatics(offsets, xyz, q64, fragment=xyzio.fragments_from_splits(offsets, split))
    has = split >= 0
    q_first = np.full(len(stems), np.nan)
    q_first[has] = [q64[offsets[i]:offsets[i] + split[i]].sum() for i in np.nonzero(has)[0]]
    np.savez(path, names=np.array(stems), energy_kcal=full["energy"] * COULOMB_KCAL,
             inter_kcal=np.where(has, inter["energy"] * COULOMB_KCAL, np.nan), split=split, q_first_fragment=q_first,
             dipole_debye=full["dipole"] * DEBYE_PER_E_ANGSTROM)


def save_cubes(directory, model, stems, offsets, xyz, species, n_elems, q64, spacing, margin):
    """``--cube``: one Gaussian cube file of the potential of the FP64 charges per system, ``DIR/<stem>.cube``."""
    from . import cube, elements
    os.makedirs(directory, exist_ok=True)
    Z = elements.z_table(n_elems)[species]
    for i, stem in enumerate(stems):
        a0, a1 = int(offsets[i]), int(offsets[i + 1])
        cube.esp_cube(os.path.join(directory, stem + ".cube"), model, Z[a0:a1], xyz[a0:a1], q64[a0:a1], spacing, margin,
                      comment=f"{stem}: epnn_b200 electrostatic potential of the predicted charges")


def main(argv=None):
    global model
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--path", default="", help="directory with *.xyz (+ optional <stem>.npy labels); reference infer.py:42")
    ap.add_argument("--weights", default="./models/decay_model_weights", help="TF checkpoint prefix; reference infer.py:57")
    ap.add_argument("--repeats", type=int, default=1, help="timed repetitions per system (undefined upstream, infer.py:71)")
    ap.add_argument("--out", default=None, help="save predictions: (S, repeats, N, 1) float32 like protein/preds.npy")
    ap.add_argument("--npad", type=int, default=None, help="pad size N (default: largest system, charge_gn.py:340)")
    ap.add_argument("--dense", action="store_true", help="build the dense padded tensors and call the model per system "
                                                         "exactly like the reference loop (slow; default = packed fast path)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--precision", type=int, default=32, choices=[32, 64])
    ap.add_argument("--option", action="append", default=[], metavar="KEY=VALUE",
                    help="engine option (epnn_set_option), e.g. gnn_far_tensor=1, pair_tensor=1, dedup_far=0; repeatable")
    ap.add_argument("--elst", default=None, metavar="OUT.npz",
                    help="also save the electrostatics of the predicted FP64 charges (packed path only): names, energy_kcal, "
                         "inter_kcal and q_first_fragment of the two monomers of each <stem>splits.npy dimer (NaN without "
                         "one), split, dipole_debye")
    ap.add_argument("--cube", default=None, metavar="DIR",
                    help="also write DIR/<stem>.cube, the electrostatic potential of the predicted FP64 charges of every "
                         "system on a grid (Gaussian cube: bohr, e/bohr; packed path only).  At the defaults a QM9 "
                         "molecule gives about 8e4 points, about 1.1 MB (0.6 to 1.6 MB)")
    ap.add_argument("--cube-spacing", type=float, default=0.3, metavar="A", help="grid spacing of --cube in A (default 0.3)")
    ap.add_argument("--cube-margin", type=float, default=4.0, metavar="A",
                    help="space between the atoms and the faces of the --cube grid in A (default 4)")
    args = ap.parse_args(argv)
    if args.elst and args.dense:
        ap.error("--elst needs the packed path (drop --dense)")
    if args.cube and args.dense:
        ap.error("--cube needs the packed path (drop --dense)")
    if not args.cube_spacing > 0 or not args.cube_margin >= 0:
        ap.error("--cube-spacing must be positive and --cube-margin non-negative")
    options = []
    for kv in args.option:
        k, sep, v = kv.partition("=")
        if not sep:
            raise SystemExit(f"--option expects KEY=VALUE, got {kv!r}")
        options.append((k, float(v)))
    h_dim, e_dim, layers = 48, 48, [32, 32]                           # infer.py:38-40
    w = load_weights(args.weights)
    T, n_elems = w.T, w.n_x

    if args.dense:
        timeA = time.time()
        x, h, q, e, Q, y, mask, names = charge_gn.gen_padded_init_state(args.path, h_dim, e_dim, n_elems=n_elems)
        timeB = time.time()
        model = charge_gn.make_model(layers, h_dim, T, n_elems, x.shape[1], device=args.device, precision=args.precision)
        model.load_weights(args.weights)
        for k, v in options:
            model.engine.set_option(k, v)
        np.save("test_names.npy", names, allow_pickle=True)
        test_preds = []
        timeC = timeD = time.time()
        for i in range(len(x)):
            timeC = time.time()
            for _ in range(args.repeats):
                inf_1 = time.time()
                test_preds.append(test_step(h[i:i + 1], e[i:i + 1], x[i:i + 1], q[i:i + 1], y[i:i + 1], mask[i:i + 1]))
                print(time.time() - inf_1)
            timeD = time.time()
        preds = np.array(test_preds).reshape(len(x), args.repeats, x.shape[1], 1)
        sizes = mask[:, 0].sum(axis=1).astype(int)
    else:
        timeA = time.time()
        # native multi-threaded ingest (epnn_xyz_load) straight into the packed arrays of the C-ABI
        stems, offsets, xyz_all, species_all, Q_all = xyzio.read_directory_packed(args.path or ".", n_elems)
        if not stems:
            raise SystemExit(f"no .xyz files under {args.path!r}")
        names = np.array(stems)
        sizes_all = np.diff(offsets)
        timeB = time.time()
        N = args.npad or int(sizes_all.max())
        model = charge_gn.make_model(layers, h_dim, T, n_elems, N, device=args.device, precision=args.precision)
        model.load_weights(args.weights)
        for k, v in options:
            model.engine.set_option(k, v)
        np.save("test_names.npy", names, allow_pickle=True)
        runs = []
        timeC = timeD = time.time()
        q64 = None
        for _ in range(args.repeats):
            timeC = time.time()
            if args.elst or args.cube:
                q32, q64 = model.predict_packed(offsets, xyz_all, species_all, Q_all, N, want_f64=True)
                runs.append(q32)
            else:
                runs.append(model.predict_packed(offsets, xyz_all, species_all, Q_all, N))
            timeD = time.time()
            print(timeD - timeC)
        S = len(stems)
        preds = np.zeros((S, args.repeats, N, 1), np.float32)
        for r, run in enumerate(runs):
            for i in range(S):
                preds[i, r, :sizes_all[i], 0] = run[offsets[i]:offsets[i + 1]]
        sizes = sizes_all
        y = np.zeros((S, N, 1))
        base = args.path or "."
        for i, stem in enumerate(stems):                              # labels: <stem>.npy next to the xyz (charge_gn.py:311-316)
            lab = os.path.join(base, stem + ".npy")
            if os.path.exists(lab):
                yv = np.array(np.load(lab), dtype=np.float32).reshape(-1)[:sizes[i]]
                y[i, :len(yv), 0] = yv
        if args.elst:
            save_electrostatics(args.elst, model, base, stems, offsets, xyz_all, q64)
        if args.cube:
            save_cubes(args.cube, model, stems, offsets, xyz_all, species_all, n_elems, q64, args.cube_spacing,
                       args.cube_margin)

    print(f"avg inference time: {(timeD - timeC) / max(1, args.repeats)}")
    print(f"avg feature time:{(timeB - timeA)}")
    if args.out:
        np.save(args.out, preds)
    if np.any(y != 0):                                               # label-aware report like charge_gn.py:470-471
        err = [np.abs(preds[i, -1, :sizes[i], 0] - y[i, :sizes[i], 0]) for i in range(len(sizes))]
        print(f"MAE vs labels: {np.concatenate(err).mean():.5f} e over {int(sizes.sum())} atoms")
    return preds


if __name__ == "__main__":
    main()
