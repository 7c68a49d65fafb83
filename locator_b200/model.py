"""Host-side model object: the subset of the Keras ``Sequential`` API the reference uses.

Mirrors what ``/root/reference/locator/locator.py`` calls on its model:
``fit`` (:367-376) -> object with ``.history`` dict, ``predict`` (:414,441),
``load_weights`` (:380,386), ``get_weights`` / ``set_weights`` in Keras order
``[gamma, beta, moving_mean, moving_var, W1, b1, ..., Wo1, bo1, Wo2, bo2]``.
All arithmetic happens in the CUDA library behind the C ABI (no CPU fallback).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _cabi
from ._cabi import lib, check, LocState
from .genotypes import PackedGenotypes, _as_dev, _stream, _dev


class History:
    def __init__(self):
        self.history = {"loss": [], "val_loss": [], "learning_rate": []}
        self.epoch = []


class LocatorModel:
    """BN(K) -> Dense(width, elu) x nlayers (Dropout in the middle) -> Dense(2) -> Dense(2)."""

    def __init__(self, K, width=256, nlayers=10, dropout_prop=0.25, batch_size=32, max_epochs=5000, seed=0,
                 learning_rate=1e-3, shard=None, exchange=None, l1_ctas=None):
        """shard = (k_offset, K_global): this model holds SNP columns [k_offset, k_offset + K) of a K_global-column
        model (tensor parallelism); exchange(tile) must then sum the float32 CUDA tensor `tile` in place over
        all shards on the current stream (see all_reduce_exchange)."""
        _dev()
        self.K, self.width, self.nlayers = int(K), int(width), int(nlayers)
        self.batch_size, self.max_epochs = int(batch_size), int(max_epochs)
        self.dropout_prop = float(dropout_prop)
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.learning_rate = float(learning_rate)
        h = C.c_void_p()
        check(lib.loc_model_create(C.byref(h), self.K, self.width, self.nlayers, self.batch_size, self.dropout_prop,
                                   self.max_epochs), "loc_model_create")
        self._h = h
        self.l1_ctas = None
        if l1_ctas is not None and self.impl == "tcgen05":
            # CTAs of the first-layer kernels (default: every SM)
            self.l1_ctas = int(l1_ctas)
            check(lib.loc_model_set_l1_ctas(self._h, self.l1_ctas), "loc_model_set_l1_ctas")
        self._keep = {}  # device tensors the handle points at
        self.shard = None
        if shard is not None:
            self.shard = (int(shard[0]), int(shard[1]))
            check(lib.loc_model_set_shard(self._h, self.shard[0], self.shard[1]), "loc_model_set_shard")
        self._tp = None
        if isinstance(exchange, str) and exchange == "peer":
            self.connect_peers()
        elif exchange is not None:
            self.set_exchange(exchange)
        check(lib.loc_model_init(self._h, self.seed, _stream()), "loc_model_init")
        self._wver = 0   # bumped whenever the weights may have changed (prediction memo key)
        self._memo = {}
        self.stop_training = False

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
            lib.loc_model_destroy(h)
            self._h = None
            tp = getattr(self, "_tp", None)
            if tp:
                lib.loc_tp_destroy(tp)
                self._tp = None

    def connect_peers(self, group=None):
        """Exchange through NVLink peer memory (loc_tp_*): the shards of one box map each other's tile buffers
        (cudaIpc handles travel through torch.distributed) and push / flag / sum without any library collective
        or host call per step.  One process per GPU, ranks of `group` = shards in column order."""
        import torch.distributed as dist

        rank, world = dist.get_rank(group), dist.get_world_size(group)
        tp = C.c_void_p()
        check(lib.loc_tp_create(C.byref(tp), rank, world, self.width), "loc_tp_create")
        buf = (C.c_uint8 * 64)()
        check(lib.loc_tp_handle(tp, buf), "loc_tp_handle")
        handles = [None] * world
        dist.all_gather_object(handles, bytes(buf), group=group)
        allh = b"".join(handles)
        check(lib.loc_tp_connect(tp, allh), "loc_tp_connect")
        dist.barrier(group)  # every shard has mapped every buffer before the first push
        check(lib.loc_model_set_tp(self._h, tp), "loc_model_set_tp")
        self._tp = tp

    def check_peers(self):
        if self._tp is not None and lib.loc_tp_error(self._tp) != 0:
            raise _cabi.LocatorCudaError("sharded model: a peer's tile never arrived (2 s timeout in the exchange)")

    def set_exchange(self, fn):
        """fn(tile): in-place sum of the [32 * width] float32 CUDA tensor over all shards, enqueued on the
        current stream; called once per forward pass while the kernels are being enqueued."""
        from ._cabi import EXCHANGE_FN

        tile = torch.zeros(32 * self.width, dtype=torch.float32, device="cuda")

        def hook(_ctx, _ptr, _n, _stream_ptr):
            try:
                fn(tile)
                return 0
            except Exception:  # surfaces as a LocatorCudaError of the calling entry point
                import traceback

                traceback.print_exc()
                return 1

        cb = EXCHANGE_FN(hook)
        self._keep["exchange"] = (tile, cb, fn)
        check(lib.loc_model_set_exchange(self._h, C.cast(cb, C.c_void_p), None, tile.data_ptr()), "loc_model_set_exchange")

    @property
    def impl(self):
        """First-layer kernel family: "tcgen05" or "simt" (CUDA cores)."""
        return lib.loc_model_impl(self._h).decode()

    @property
    def hidden_impl(self):
        """Hidden-stack kernel family: "tcgen05" or "simt" (CUDA cores; width-256 stacks deeper than 14 layers)."""
        return lib.loc_model_hidden_impl(self._h).decode()

    # ---- weights (Keras order) -------------------------------------------------
    def num_weights(self):
        return int(lib.loc_model_num_weights(self._h))

    def _shape(self, idx):
        K, H, L = self.K, self.width, self.nlayers
        if idx < 4:
            return (K,)
        d, isb = divmod(idx - 4, 2)
        dims = [K] + [H] * L + [2, 2]
        return (dims[d + 1],) if isb else (dims[d], dims[d + 1])

    def get_weights(self):
        out = []
        for i in range(self.num_weights()):
            n = int(lib.loc_model_weight_size(self._h, i))
            a = np.empty(n, dtype=np.float32)
            check(lib.loc_model_get_weight(self._h, i, a.ctypes.data, n, _stream()), "loc_model_get_weight")
            out.append(a.reshape(self._shape(i)))
        return out

    def set_weights(self, ws):
        self._wver += 1
        if len(ws) != self.num_weights():
            raise ValueError(f"expected {self.num_weights()} weight arrays, got {len(ws)}")
        for i, w in enumerate(ws):
            a = np.ascontiguousarray(np.asarray(w, dtype=np.float32))
            if a.shape != self._shape(i):
                raise ValueError(f"weight {i}: expected shape {self._shape(i)}, got {a.shape}")
            check(lib.loc_model_set_weight(self._h, i, a.ctypes.data, a.size, _stream()), "loc_model_set_weight")

    def get_adam(self, idx):
        n = int(lib.loc_model_weight_size(self._h, idx))
        m = np.empty(n, np.float32)
        v = np.empty(n, np.float32)
        check(lib.loc_model_get_adam(self._h, idx, m.ctypes.data, v.ctypes.data, n, _stream()), "loc_model_get_adam")
        return m.reshape(self._shape(idx)), v.reshape(self._shape(idx))

    def save_weights(self, path):
        """Weights file of this build (.npz in Keras weight order; HDF5 is not available here)."""
        ws = self.get_weights()
        with open(path, "wb") as fh:
            np.savez(fh, **{f"w{i:03d}": w for i, w in enumerate(ws)})

    def load_weights(self, path):
        with np.load(path) as z:
            self.set_weights([z[k] for k in sorted(z.files)])

    # ---- data binding ------------------------------------------------------------
    @staticmethod
    def _packed(x):
        return x if isinstance(x, PackedGenotypes) else PackedGenotypes.from_counts(x)

    def bind_train(self, x, y):
        g = self._packed(x)
        if g.K != self.K:
            raise ValueError(f"training matrix has {g.K} SNPs, model expects {self.K}")
        locs = _as_dev(np.asarray(y, dtype=np.float32), torch.float32)
        check(lib.loc_model_bind_train(self._h, g.ptr, g.n, g.row_words, locs.data_ptr()), "loc_model_bind_train")
        self._keep["train"] = (g, locs)
        return g

    def bind_val(self, x, y):
        g = self._packed(x)
        if g.K != self.K:
            raise ValueError(f"validation matrix has {g.K} SNPs, model expects {self.K}")
        locs = _as_dev(np.asarray(y, dtype=np.float32), torch.float32)
        check(lib.loc_model_bind_val(self._h, g.ptr, g.n, g.row_words, locs.data_ptr()), "loc_model_bind_val")
        self._keep["val"] = (g, locs)
        return g

    def set_dropout_masks(self, keep):
        """Test hook: keep[step, 32, width] uint8 masks ([step, batch_size, width] for batch sizes above 32) replace the
        Philox stream (None restores it)."""
        if keep is None:
            check(lib.loc_model_set_dropout_masks(self._h, None, 0), "loc_model_set_dropout_masks")
            self._keep.pop("masks", None)
            return
        keep = np.asarray(keep, dtype=np.uint8)
        rows = 32 * max(1, -(-self.batch_size // 32))  # the library indexes [step][32 * chunks of a step][width]
        assert keep.ndim == 3 and keep.shape[1] in (self.batch_size, rows) and keep.shape[2] == self.width
        if keep.shape[1] != rows:
            keep = np.concatenate([keep, np.ones((keep.shape[0], rows - keep.shape[1], self.width), np.uint8)], axis=1)
        k = _as_dev(np.ascontiguousarray(keep), torch.uint8)
        check(lib.loc_model_set_dropout_masks(self._h, k.data_ptr(), k.shape[0]), "loc_model_set_dropout_masks")
        self._keep["masks"] = k

    def set_schedule(self, lr=None, patience=100):
        check(lib.loc_model_set_schedule(self._h, float(self.learning_rate if lr is None else lr), int(patience)),
              "loc_model_set_schedule")

    # ---- training ------------------------------------------------------------------
    def state(self) -> LocState:
        st = LocState()
        check(lib.loc_model_state(self._h, C.byref(st), _stream()), "loc_model_state")
        self.check_peers()
        return st

    def train_step(self, rows):
        self._wver += 1
        r = _as_dev(np.asarray(rows, dtype=np.int32), torch.int32)
        self._keep["rows"] = r
        check(lib.loc_train_step(self._h, r.data_ptr(), int(r.numel()), _stream()), "loc_train_step")

    def debug_stage(self, stage, rows):
        self._wver += 1
        """Launch one stage (0 fwd-L1, 1 hidden, 2 bwd-L1, 3 small update) of a step on `rows`."""
        r = _as_dev(np.asarray(rows, dtype=np.int32), torch.int32)
        self._keep["rows"] = r
        check(lib.loc_debug_stage(self._h, int(stage), r.data_ptr(), int(r.numel()), _stream()), "loc_debug_stage")

    def debug_read(self, which):
        """Scratch buffers: 0 -> Z1 partial tiles [P, 32, H]; 1 -> dz [L, 32, H]; 2 -> activations [L, 32, H]."""
        n = int(lib.loc_debug_read(self._h, int(which), np.empty(1, np.float32).ctypes.data, 0, _stream()))
        if n < 0:
            raise _cabi.LocatorCudaError("loc_debug_read failed")
        a = np.empty(n, np.float32)
        lib.loc_debug_read(self._h, int(which), a.ctypes.data, n, _stream())
        return a.reshape(-1, 32, self.width)

    def train_epochs(self, perms):
        self._wver += 1
        """perms int32 [n_epochs, n_train]; enqueues the epochs (asynchronous)."""
        p = _as_dev(np.asarray(perms, dtype=np.int32), torch.int32)
        self._keep.setdefault("perms", []).append(p)
        check(lib.loc_train_epochs(self._h, p.data_ptr(), int(p.shape[0]), _stream()), "loc_train_epochs")

    def train_steps(self, perm, step0, n_steps):
        """Steps [step0, step0 + n_steps) of the epoch ordered by ``perm`` (a device int32 tensor from a previous
        call, or anything array-like of length n_train) on the production schedule; returns the device tensor
        so that a following call can continue the same epoch (loc_train_steps)."""
        self._wver += 1
        p = perm if isinstance(perm, torch.Tensor) else _as_dev(np.asarray(perm, dtype=np.int32), torch.int32)
        self._keep["span_perm"] = p
        check(lib.loc_train_steps(self._h, p.data_ptr(), int(step0), int(n_steps), _stream()), "loc_train_steps")
        return p

    def history_rows(self, n):
        a = np.zeros((max(n, 1), 3), dtype=np.float32)
        if n > 0:
            check(lib.loc_model_history(self._h, a.ctypes.data, n, _stream()), "loc_model_history")
        return a[:n]

    def fit(self, x, y, epochs=None, batch_size=None, shuffle=True, verbose=0, validation_data=None, callbacks=None,
            patience=100, shuffle_seed=None, perms=None, epochs_per_call=16):
        """Keras-style fit (locator.py:367-376): shuffled mini-batches, validation every epoch,
        checkpoint-best / early stopping / reduce-LR-on-plateau.  Returns a History.

        ``perms`` (optional [epochs, n]) fixes the batch order; otherwise each epoch draws a fresh
        permutation from ``np.random.default_rng(shuffle_seed)`` (never from numpy's legacy global
        stream, which the reference reserves for its own index draws).
        """
        if batch_size is not None and int(batch_size) != self.batch_size:
            raise ValueError("batch_size differs from the one the model was created with")
        if validation_data is None:
            raise ValueError("validation_data is required (the reference always passes it)")
        epochs = self.max_epochs if epochs is None else int(epochs)
        if epochs > self.max_epochs:
            raise ValueError("epochs exceeds max_epochs given at construction")
        g = self.bind_train(x, y)
        self.bind_val(*validation_data)
        self.set_schedule(patience=patience)
        n = g.n
        rng = np.random.default_rng(self.seed if shuffle_seed is None else shuffle_seed)
        self._keep["perms"] = []
        done = 0
        st = self.state()
        while done < epochs and not st.stopped:
            ne = min(epochs_per_call, epochs - done)
            if perms is not None:
                p = np.asarray(perms[done:done + ne], dtype=np.int32)
            elif shuffle:
                p = np.stack([rng.permutation(n) for _ in range(ne)]).astype(np.int32)
            else:
                p = np.tile(np.arange(n, dtype=np.int32), (ne, 1))
            self.train_epochs(p)
            done += ne
            st = self.state()  # synchronises the stream
            self._keep["perms"] = self._keep["perms"][-1:]
            if verbose:
                print(f"epoch {st.epoch}: loss {st.last_loss:.6f} val_loss {st.last_val_loss:.6f} lr {st.lr:g}")
            if done >= epochs:
                break
        self.stop_training = bool(st.stopped)
        h = History()
        rows = self.history_rows(st.epoch)
        h.history["loss"] = [float(v) for v in rows[:, 0]]
        h.history["val_loss"] = [float(v) for v in rows[:, 1]]
        h.history["learning_rate"] = [float(v) for v in rows[:, 2]]
        h.epoch = list(range(st.epoch))
        return h

    def _history(self, n_epochs):
        h = History()
        rows = self.history_rows(n_epochs)
        h.history["loss"] = [float(v) for v in rows[:, 0]]
        h.history["val_loss"] = [float(v) for v in rows[:, 1]]
        h.history["learning_rate"] = [float(v) for v in rows[:, 2]]
        h.epoch = list(range(n_epochs))
        return h

    def restore_best(self):
        self._wver += 1
        check(lib.loc_restore_best(self._h, _stream()), "loc_restore_best")

    def snapshot(self):
        check(lib.loc_snapshot(self._h, _stream()), "loc_snapshot")

    # ---- inference -----------------------------------------------------------------
    def predict(self, x, verbose=0):
        g = self._packed(x)
        if g.K != self.K:
            raise ValueError(f"matrix has {g.K} SNPs, model expects {self.K}")
        # the reference re-predicts the unchanged validation set for every jacknife replicate
        # (locator.py:441 inside :729-743): same weights + same device matrix -> same answer
        if g.n == 0:  # no rows (a run without NA-location samples): Keras returns an empty [0, 2] array
            return np.zeros((0, 2), dtype=np.float32)
        # memo per matrix object (a few entries: the sweep alternates a fresh clone of predgen with the one testgen)
        key = (g.version, self._wver) if isinstance(x, PackedGenotypes) else None
        hit = self._memo.get(id(g)) if key is not None else None
        if hit is not None and hit[0] == key and hit[2] is g:
            self._memo[id(g)] = self._memo.pop(id(g))  # most recently used last
            return hit[1].copy()
        out = torch.zeros((g.n, 2), dtype=torch.float32, device=_dev())
        check(lib.loc_predict(self._h, g.ptr, g.n, g.row_words, out.data_ptr(), _stream()), "loc_predict")
        res = out.cpu().numpy()
        if key is not None:
            if len(self._memo) >= 4:  # least recently used first (dicts keep insertion order)
                for k in list(self._memo)[: len(self._memo) - 3]:
                    del self._memo[k]
            self._memo[id(g)] = (key, res.copy(), g)
        return res

    def evaluate(self, x, y, verbose=0):
        g = self._packed(x)
        locs = _as_dev(np.asarray(y, dtype=np.float32), torch.float32)
        loss = C.c_float()
        check(lib.loc_eval(self._h, g.ptr, g.n, g.row_words, locs.data_ptr(), C.byref(loss), _stream()), "loc_eval")
        return float(loss.value)


MAX_GROUP = 8


def fit_group(models, xs, ys, validation_datas, epochs=None, patience=100, verbose=0, epochs_per_call=16):
    """Train up to 8 independent models (replicates) side by side on one GPU.

    Same semantics per model as ``LocatorModel.fit`` (each model keeps its own shuffle stream,
    callbacks state and history, and ends bit-identical to the same model trained alone); the steps
    are issued in lockstep through ``loc_group_train_epochs`` so the models' latency-bound hidden
    stacks share launches.  Any batch size: above 32 rows the models' batch statistics and step ends
    share one launch each, and their 32-row chunks share hidden-stack launches.  Models must have the
    same width / nlayers / batch size / number of training rows (replicates of one run do) and run one kernel
    family for the first layer and the hidden stack: all tcgen05 (width 256, nlayers up to 14) or all CUDA-core
    (other widths), i.e. ``impl == hidden_impl`` and the same for every model.  Width 256 with 15..21 layers
    (tcgen05 first layer, CUDA-core hidden stack) is refused; such models train one at a time.
    Returns the list of History objects.
    """
    G = len(models)
    if not 1 <= G <= MAX_GROUP:
        raise ValueError(f"a replicate group holds 1..{MAX_GROUP} models")
    epochs = min(m.max_epochs for m in models) if epochs is None else int(epochs)
    rngs = []
    for m, x, y, vd in zip(models, xs, ys, validation_datas):
        m.bind_train(x, y)
        m.bind_val(*vd)
        m.set_schedule(patience=patience)
        rngs.append(np.random.default_rng(m.seed))
        m._keep["perms"] = []
    n = models[0]._keep["train"][0].n
    done = 0
    states = [m.state() for m in models]
    while done < epochs:
        active = [i for i in range(G) if not states[i].stopped]
        if not active:
            break
        ne = min(epochs_per_call, epochs - done)
        perms = []
        for i in active:
            p = _as_dev(np.stack([rngs[i].permutation(n) for _ in range(ne)]).astype(np.int32), torch.int32)
            models[i]._keep["perms"] = [p]
            perms.append(p)
        handles = (C.c_void_p * len(active))(*[models[i]._h for i in active])
        pptrs = (C.c_void_p * len(active))(*[p.data_ptr() for p in perms])
        check(lib.loc_group_train_epochs(handles, len(active), pptrs, ne, _stream()), "loc_group_train_epochs")
        for i in active:
            models[i]._wver += 1
        done += ne
        for i in active:
            states[i] = models[i].state()
        if verbose:
            print(f"epoch {done}: " + " ".join(f"[{i}] val {states[i].last_val_loss:.4f}" for i in active))
    out = []
    for m, st in zip(models, states):
        m.stop_training = bool(st.stopped)
        out.append(m._history(st.epoch))
    return out


def shard_bounds(K, rank, world):
    """Columns [k0, k1) of shard `rank`: contiguous, multiples of the 64-SNP tile except the last."""
    per = -(-(-(-int(K) // 64)) // int(world)) * 64
    k0 = min(int(K), per * int(rank))
    return k0, min(int(K), k0 + per)


def all_reduce_exchange(group=None):
    """Exchange hook over torch.distributed (NCCL over NVLink on a GPU box): sum over the shards' tiles."""
    import torch.distributed as dist

    def fn(tile):
        dist.all_reduce(tile, op=dist.ReduceOp.SUM, group=group)

    return fn


def spare_cluster_l1_ctas():
    """First-layer CTA count that leaves one 16-SM cluster's worth of SMs free (experiments with concurrent
    hidden stacks; the count fixes the summation order of the layer, so use it for every model of a run)."""
    return max(1, torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count - 16)
