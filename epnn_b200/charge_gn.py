"""Drop-in facade for the reference's ``charge_gn`` module (inference surface only).

Same names, argument meaning and return layouts as the reference; the arithmetic runs in libepnn_b200.so:

* ``get_init_edges``          reference ``charge_gn.py:122-163``  -> ``epnn_init_edges`` (CUDA, float64 math)
* ``gen_padded_init_state``   reference ``charge_gn.py:292-366``  -> xyz parsing on the host, descriptors on the GPU
* ``make_model(...)``         reference ``charge_gn.py:369-391``  -> :class:`Model`; ``load_weights`` reads the TF
  tensor bundle without TensorFlow; ``model([h, e, x, q, mask])`` runs ``epnn_infer_dense`` (the literal dense graph);
  ``model.predict_systems`` / ``predict_packed`` is the fast packed path (``epnn_infer_batch``).

Out of scope (SURVEY.md section 2): the training loop, ``train_step``, the stale feature generators.
There is no CPU fallback: every call below needs the CUDA library and a GPU.
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence

import numpy as np

from . import elements, xyzio
from .checkpoint import Weights, load_weights as _load_checkpoint, save_weights as _save_checkpoint
from .engine import Engine

# reference charge_gn.py:9-28 (10-wide convention); the 9-wide table of infer.py:13-30 is elements.symbols_for(9)
atom_num_dict = dict(elements.ATOMIC_NUMBER)
elem_dict = {s: i for i, s in enumerate(elements.symbols_for(10))}

_UTIL: Optional[Engine] = None


def _util_engine() -> Engine:
    """A context with all-zero weights, used only for weight-independent entry points (descriptors)."""
    global _UTIL
    if _UTIL is None:
        from .checkpoint import MLP
        K = 2 * (9 + 49) + 48
        z = lambda *s: np.zeros(s, np.float32)
        mk = lambda out: MLP(W=[z(K, 32), z(32, 32), z(32, out)], b=[z(32), z(32), z(out)])
        w = Weights(T=1, n_x=9, h_dim=48, e_dim=48, msg=[mk(32)],
                    upd=MLP(W=[z(80, 32), z(32, 32), z(32, 48)], b=[z(32), z(32), z(48)]), pas=[mk(1)])
        _UTIL = Engine(w, device=int(os.environ.get("EPNN_DEVICE", "0")))
    return _UTIL


def get_init_edges(xyz, molecular_splits=None, num=32, cutoff=3.0, eta=2.0, _engine: Optional[Engine] = None):
    """Reference ``charge_gn.py:122-163``: returns ``(e (n,n,num) float32, C (n,n,num) float64)``.

    The CUDA kernels implement the configuration the reference always uses (``num=48, cutoff=3.0, eta=2.0``,
    ``charge_gn.py:331``); anything else is rejected loudly.  ``molecular_splits`` only feeds dead code upstream
    (``:126-146``); like the reference, a non-empty 1-D array terminates (``exit()`` at ``:145``)."""
    if molecular_splits is not None:
        ms = np.asarray(molecular_splits)
        if ms.ndim == 1 and ms.shape[0] != 0:
            print("molecular splits are not in a recognized format")
            raise SystemExit()
    if num != 48 or cutoff != 3.0 or eta != 2.0:
        raise NotImplementedError("libepnn_b200 implements get_init_edges for num=48, cutoff=3.0, eta=2.0 "
                                  "(the only configuration the reference uses, charge_gn.py:331)")
    xyz = np.ascontiguousarray(xyz, dtype=np.float32)
    e = (_engine or _util_engine()).init_edges(xyz)
    # C is returned by the reference but never consumed by the model (`this_soft_mask`, charge_gn.py:331-333)
    D = np.sqrt(((xyz.astype(np.float64)[None] - xyz.astype(np.float64)[:, None]) ** 2).sum(-1))
    C = (np.cos(np.pi * D / cutoff) + 1.0) / 2.0
    C[D >= cutoff] = 0.0
    C[D <= 0.0] = 1.0
    np.fill_diagonal(C, 0.0)
    return e, np.tile(C[..., None], (1, 1, num))


def gen_padded_init_state(path, h_dim, e_dim, n_elems: int = 10, sort: bool = False, _engine: Optional[Engine] = None):
    """Reference ``charge_gn.py:292-366``: ``(x, h, q, e, Q, y, mask, names)`` as dense float64 arrays padded to the
    largest system.  ``n_elems`` selects the feature convention (10 = charge_gn.py:9-28, the reference default;
    9 = infer.py:13-30, what ``decay_model_weights`` / ``model2_weights`` were trained with)."""
    if not path.endswith("/") and path != "":
        path = path + "/"                       # the reference concatenates path + filename (:302)
    systems = xyzio.read_directory(path or ".", sort=sort)
    if not systems:
        raise ValueError(f"no .xyz files under {path!r}")
    for s in systems:
        if s.labels is None:
            print('No labels provided, y set to 0')
    S, N = len(systems), max(s.n for s in systems)
    x = np.zeros((S, N, N, n_elems))
    h = np.zeros((S, N, N, h_dim))
    q = np.zeros((S, N, N, 1))
    e = np.zeros((S, N, N, e_dim))
    y = np.zeros((S, N, 1))
    mask = np.zeros((S, N, N))
    Q = []
    for i, s in enumerate(systems):
        n = s.n
        feats = elements.features(elements.species_index(s.symbols, n_elems), n_elems)
        x[i, :n, :n] = feats[None, :, :]                                  # x[i][j][k] = x_k  (:335,357)
        q[i, :n, :n, 0] = np.float32(np.float32(s.Q) / n)                  # :337-338
        splits_path = path + s.name + "splits.npy"                         # :305-308 (loaded, effect-free upstream)
        splits = np.load(splits_path) if os.path.exists(splits_path) else np.array([])
        e[i, :n, :n] = get_init_edges(s.xyz, splits, num=e_dim, _engine=_engine)[0]
        mask[i, :n, :n] = 1
        lab = s.labels if s.labels is not None else np.zeros(n)
        y[i, :len(lab), 0] = lab
        Q.append(np.array(s.Q, dtype=np.float32))
    return x, h, q, e, Q, y, mask, np.array([s.name for s in systems])


class Model:
    """What ``charge_gn.make_model`` returns upstream (a ``tf.keras.Model``), for inference."""

    def __init__(self, layers, h_dim, T, n_elems, natom, device: int = 0, precision: int = 32):
        if list(layers) != [32, 32] or h_dim != 48:
            raise NotImplementedError("the shipped checkpoints use layers=[32,32], h_dim=48 (infer.py:38-40)")
        self.layers, self.h_dim, self.T, self.n_elems, self.natom = list(layers), h_dim, T, n_elems, natom
        self.device, self.precision = device, precision
        self.engine: Optional[Engine] = None
        self.weights: Optional[Weights] = None

    def load_weights(self, prefix: str):
        w = _load_checkpoint(prefix)
        if w.T != self.T or w.n_x != self.n_elems:
            raise ValueError(f"checkpoint {prefix} holds a model with T={w.T}, n_elems={w.n_x}; "
                             f"make_model was called with T={self.T}, n_elems={self.n_elems}")
        if self.engine is not None:
            self.engine.close()
        self.weights = w
        self._loaded_from = prefix
        self.engine = Engine(w, device=self.device, precision=self.precision)
        return self

    def save_weights(self, prefix: str, template: Optional[str] = None):
        """``model.save_weights(prefix)`` (reference ``charge_gn.py:462``): a TF tensor-bundle checkpoint TensorFlow's own
        ``load_weights`` can restore.  The Keras object graph and the file layout come from ``template`` (default: the
        checkpoint this model was loaded from); see :func:`epnn_b200.checkpoint.save_weights`."""
        if self.weights is None:
            raise RuntimeError("nothing to save: call load_weights(prefix) first")
        _save_checkpoint(self.weights, prefix, template or self._loaded_from)
        return self

    def _need(self) -> Engine:
        if self.engine is None:
            raise RuntimeError("call load_weights(prefix) first (there is no random initialisation path: inference only)")
        return self.engine

    def __call__(self, inputs, training: bool = False):
        """``model([h, e, x, q, mask])`` -> ``(B, N, 1)`` float32, the reference call (infer.py:34)."""
        h, e, x, q, mask = inputs
        e = np.asarray(e)
        mask = np.asarray(mask)
        if mask.ndim == 4:
            mask = mask[..., 0]
        return self._need().infer_dense(h, e, x, np.asarray(q).reshape(e.shape[:3]), mask)

    predict = __call__

    def predict_packed(self, offsets, xyz, species, Q, npad=None, want_f64: bool = False):
        return self._need().infer_batch(offsets, xyz, species, Q, npad, want_f64=want_f64)

    def electrostatics(self, offsets, xyz, q, fragment=None, potential: bool = False):
        """Energy, dipole and optionally potential of given charges: :meth:`epnn_b200.engine.Engine.electrostatics`."""
        return self._need().electrostatics(offsets, xyz, q, fragment=fragment, potential=potential)

    def potential_points(self, offsets, xyz, q, point_offsets, points, field: bool = False):
        """Potential and optionally field of given charges at given points: :meth:`epnn_b200.engine.Engine.potential_points`."""
        return self._need().potential_points(offsets, xyz, q, point_offsets, points, field=field)

    def predict_systems(self, systems: Sequence[xyzio.System], npad=None) -> List[np.ndarray]:
        """Charges of parsed systems through the packed path; ``npad`` = pad size N of the reference's dense model
        (default: the largest system, as ``gen_padded_init_state`` pads, charge_gn.py:340)."""
        offsets, xyz, species, Q = xyzio.pack(systems, self.n_elems)
        if npad is None:
            npad = max(s.n for s in systems)
        out = self.predict_packed(offsets, xyz, species, Q, npad)
        return [out[offsets[i]:offsets[i + 1]] for i in range(len(systems))]


def make_model(layers, h_dim, T, n_elems, natom, device: int = 0, precision: int = 32) -> Model:
    return Model(layers, h_dim, T, n_elems, natom, device=device, precision=precision)
