"""Oracle: Locator's network, loss, Adam and callbacks restated on the CPU (torch fp32).

TEST INFRASTRUCTURE -- see oracle/__init__.py.  Explicit forward/backward (no
autograd) so every formula is visible; tests cross-check it against autograd.

Follows ``/root/reference/locator/locator.py``:
  load_network   :311-327  BN(K) -> Dense(width, elu) x floor(L/2) -> Dropout(p)
                           -> Dense(width, elu) x ceil(L/2) -> Dense(2) -> Dense(2);
                           loss sqrt(sum((yhat - y)^2, -1)); optimizer "Adam"
  load_callbacks :330-362  ModelCheckpoint(best val_loss) / EarlyStopping(patience)
                           / ReduceLROnPlateau(0.5, patience//6)
  train_network  :365-394  fit(shuffle, batch_size, validation_data) + reload best
  predict_locs   :414,441  predict at batch 32

Keras defaults restated from the published Keras sources (SURVEY.md Appendix A;
TensorFlow/Keras is not installable here -> "parity unpinned" against live TF):
  BatchNormalization momentum 0.99, eps 1e-3, biased batch variance
      (tf.nn.moments), y = x*inv + (beta - mean*inv), inv = gamma*rsqrt(var+eps)
  Adam lr 1e-3, b1 0.9, b2 0.999, eps 1e-7:
      alpha = lr*sqrt(1-b2^t)/(1-b1^t); m += (g-m)(1-b1); v += (g^2-v)(1-b2);
      w -= alpha*m/(sqrt(v)+eps)
  elu alpha=1; dropout keeps with prob 1-p and scales by 1/(1-p).
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import philox_ref

F32 = torch.float32
BN_EPS = 1e-3
BN_MOM = 0.99
ADAM_B1 = 0.9
ADAM_B2 = 0.999
ADAM_EPS = 1e-7


def layer_plan(nlayers):
    """(#dense before dropout, #dense after) -- locator.py:319-323."""
    return int(np.floor(nlayers / 2)), int(np.ceil(nlayers / 2))


def init_weights(K, width=256, nlayers=10, seed=0):
    """Keras-order weight list with the device's Philox glorot init (zero biases).

    Order: [gamma, beta, moving_mean, moving_var, W1, b1, ..., W_L, b_L, Wo1, bo1, Wo2, bo2].
    Dense kernel i (0-based over all L+2 Dense layers) uses Philox stream 16+i.
    """
    ws = [np.ones(K, np.float32), np.zeros(K, np.float32), np.zeros(K, np.float32), np.ones(K, np.float32)]
    dims = [K] + [width] * nlayers + [2, 2]
    for i in range(len(dims) - 1):
        ws.append(philox_ref.glorot_uniform(dims[i], dims[i + 1], seed, 16 + i))
        ws.append(np.zeros(dims[i + 1], np.float32))
    return ws


def elu(z):
    return torch.where(z > 0, z, torch.expm1(z))


# ---- TF32 operand model (numerics="tf32") --------------------------------------------------------------
# The tcgen05 kernels feed fp32 bit patterns to kind::tf32 MMAs: the tensor core reads sign, exponent and the
# top 10 mantissa bits of each operand and accumulates in fp32.  Weights go in as stored (their low 13 bits are
# ignored: truncation); everything the kernels write into an operand tile themselves (folded-BN inputs,
# activations, dz, centred genotypes) is rounded to nearest, ties away (cvt.rna.tf32.f32) first.  TensorFlow's
# default fp32 matmul on Ampere-and-later GPUs makes the same kind of approximation.  This mode restates WHERE
# the device rounds, so that what is left between it and the device is summation order and a few
# last-place differences of rsqrt / expm1 / sqrt -- it is still test infrastructure, not a product path.
def tf32_rna(t):
    i = t.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def tf32_trunc(t):
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


class RefLocator:
    """The reference network + optimizer state, Keras semantics, fp32 on CPU."""

    def __init__(self, K, width=256, nlayers=10, dropout=0.25, weights=None, seed=0, lr=1e-3, numerics="fp32",
                 l1_parts=1):
        """numerics: "fp32" (the reference's CPU arithmetic), "tf32" (the device's operand rounding, see
        tf32_rna / tf32_trunc above) or "tf32_l1" (tcgen05 first layer, CUDA-core hidden stack -- width-256 models
        deeper than the tcgen05 stack holds: the first layer's forward and backward as in "tf32", the hidden and output
        products in fp32).  l1_parts > 1: the first layer's sum over the SNPs is taken in that many
        contiguous parts (64-SNP tiles dealt out like the device's CTAs) added in order -- a different fp32
        summation order of the same products, which is all a change of the device's CTA count does."""
        assert numerics in ("fp32", "tf32", "tf32_l1")
        self.tf32 = numerics == "tf32"  # tf32 operands in the hidden and output layers
        self.tf32_l1 = numerics in ("tf32", "tf32_l1")  # tf32 operands in the first layer, its backward as the device's
        self.l1_parts = int(l1_parts)
        if nlayers < 2:
            raise ValueError("oracle restates nlayers >= 2 (first Dense precedes Dropout)")
        self.K, self.H, self.L, self.p = K, width, nlayers, float(dropout)
        self.n_before, self.n_after = layer_plan(nlayers)
        ws = weights if weights is not None else init_weights(K, width, nlayers, seed)
        self.set_weights(ws)
        self.lr = np.float32(lr)
        self.t = 0  # optimizer iterations
        self.m = [torch.zeros_like(w) for w in self.trainable()]
        self.v = [torch.zeros_like(w) for w in self.trainable()]

    # ---- weights in Keras order ------------------------------------------
    def set_weights(self, ws):
        ws = [torch.as_tensor(np.asarray(w, dtype=np.float32)).clone() for w in ws]
        self.gamma, self.beta, self.mmean, self.mvar = ws[:4]
        rest = ws[4:]
        self.W = rest[0::2]
        self.b = rest[1::2]
        assert len(self.W) == self.L + 2

    def get_weights(self):
        out = [self.gamma, self.beta, self.mmean, self.mvar]
        for w, b in zip(self.W, self.b):
            out += [w, b]
        return [t.numpy().copy() for t in out]

    def trainable(self):
        out = [self.gamma, self.beta]
        for w, b in zip(self.W, self.b):
            out += [w, b]
        return out

    # ---- forward ----------------------------------------------------------
    def forward(self, x_u8, training, mask=None):
        """x_u8 [B,K] uint8; mask [B,H] keep-mask (bool/0-1) when training.  Returns (yhat, cache)."""
        x = torch.as_tensor(np.asarray(x_u8)).to(F32)
        c = {"x": x}
        if training:
            mean = x.mean(dim=0)
            var = ((x - mean) ** 2).mean(dim=0)  # biased (tf.nn.moments)
        else:
            mean, var = self.mmean, self.mvar
        rs = torch.rsqrt(var + BN_EPS)
        inv = rs * self.gamma
        a = x * inv + (self.beta - mean * inv)
        c.update(mean=mean, var=var, rs=rs)
        acts = [a]  # input of dense layer i
        zs = []
        op_a = tf32_rna if self.tf32 else (lambda t: t)     # operand tiles the kernels build
        op_w = tf32_trunc if self.tf32 else (lambda t: t)   # weights as stored
        for i in range(self.L):
            oa, ow = (tf32_rna, tf32_trunc) if i == 0 and self.tf32_l1 else (op_a, op_w)
            if i == 0 and self.l1_parts > 1:
                z = self._l1_in_parts(oa(acts[-1]), ow(self.W[0])) + self.b[0]
            else:
                z = oa(acts[-1]) @ ow(self.W[i]) + self.b[i]
            h = elu(z)
            zs.append(z)
            if i == self.n_before - 1:  # Dropout sits after the floor(L/2)-th Dense
                if training and self.p > 0:
                    keep = torch.as_tensor(np.asarray(mask)).to(F32)
                    h = h * keep * np.float32(1.0 / (1.0 - self.p))
                    c["keep"] = keep
            acts.append(h)
        y1 = op_a(acts[-1]) @ self.W[self.L] + self.b[self.L]  # Dense(2) runs on CUDA cores: fp32 weights
        y2 = y1 @ self.W[self.L + 1] + self.b[self.L + 1]
        c.update(acts=acts, zs=zs, y1=y1)
        return y2, c

    def _l1_in_parts(self, a, w):
        """a @ w with the K axis cut like the device cuts it (csrc/l1_tc.cu: tile_range): 64-SNP tiles, the first
        nt % P parts one tile longer than the rest."""
        nt, P = -(-self.K // 64), self.l1_parts
        q, rem = divmod(nt, P)
        z = None
        for p in range(P):
            t0 = p * q + min(p, rem)
            t1 = t0 + q + (1 if p < rem else 0)
            k0, k1 = min(self.K, 64 * t0), min(self.K, 64 * t1)
            if k1 > k0:
                part = a[:, k0:k1] @ w[k0:k1]
                z = part if z is None else z + part
        return z

    @staticmethod
    def loss_per_sample(yhat, y):
        return torch.sqrt(((yhat - y) ** 2).sum(dim=-1))

    # ---- one optimizer step ----------------------------------------------
    def gradients(self, x_u8, y, mask=None):
        """loss (python float of fp32) and grads in trainable() order, explicit backward."""
        y = torch.as_tensor(np.asarray(y, dtype=np.float32))
        yhat, c = self.forward(x_u8, True, mask)
        B = yhat.shape[0]
        d = self.loss_per_sample(yhat, y)
        loss = d.mean()
        dy2 = (yhat - y) / (d[:, None] * B)  # NaN when d == 0, as in the reference
        acts, zs = c["acts"], c["zs"]
        L = self.L
        gW = [None] * (L + 2)
        gb = [None] * (L + 2)
        gW[L + 1] = c["y1"].T @ dy2
        gb[L + 1] = dy2.sum(0)
        dy1 = dy2 @ self.W[L + 1].T
        gW[L] = acts[L].T @ dy1
        gb[L] = dy1.sum(0)
        dh = dy1 @ self.W[L].T
        dzs = [None] * L
        for i in range(L - 1, -1, -1):
            if i == self.n_before - 1 and self.p > 0:
                dh = dh * c["keep"] * np.float32(1.0 / (1.0 - self.p))
            z = zs[i]
            dz = torch.where(z > 0, dh, dh * torch.exp(z))  # EluGrad: (out+1)*g for out<0
            dzs[i] = dz
            gb[i] = dz.sum(0)
            if i == 0 and self.tf32_l1:
                break  # first layer below: the device never forms d loss / d (BN output)
            gW[i] = acts[i].T @ dz
            dh = (tf32_rna(dz) @ tf32_trunc(self.W[i]).T) if self.tf32 else (dz @ self.W[i].T)
        if self.tf32_l1:
            # first-layer backward as the device computes it (csrc/l1_tc.cu): S = (x - mean)^T dz with the centred
            # genotypes rounded to tf32 (exact for a batch of 32) and dz as hi + lo parts (fp32-accurate);
            # dW1 = inv * S + beta * c0, dgamma = rs * sum_j W1 * S, dbeta = sum_j W1 * c0, c0 = column sums of dz
            dz0 = dzs[0]
            S = tf32_rna(c["x"] - c["mean"]).T @ dz0
            c0 = dz0.sum(0)
            gW[0] = (c["rs"] * self.gamma)[:, None] * S + self.beta[:, None] * c0[None, :]
            ggamma = c["rs"] * (self.W[0] * S).sum(1)
            gbeta = self.W[0] @ c0
        else:
            # dh is now d(loss)/d(BN output)
            xn = (c["x"] - c["mean"]) * c["rs"]
            ggamma = (dh * xn).sum(0)
            gbeta = dh.sum(0)
        grads = [ggamma, gbeta]
        for w, b in zip(gW, gb):
            grads += [w, b]
        c["dzs"] = dzs  # d loss / d z_i per Dense(width) layer (tests compare dzs[0] with the device's dZ1)
        return float(loss), grads, c

    def train_step(self, x_u8, y, mask=None):
        loss, grads, c = self.gradients(x_u8, y, mask)
        # BN moving statistics (updated in the forward pass of a training step)
        self.mmean.mul_(np.float32(BN_MOM)).add_(c["mean"] * np.float32(1.0 - BN_MOM))
        self.mvar.mul_(np.float32(BN_MOM)).add_(c["var"] * np.float32(1.0 - BN_MOM))
        self.t += 1
        t = np.float32(self.t)
        b1p = np.float32(np.power(np.float32(ADAM_B1), t))
        b2p = np.float32(np.power(np.float32(ADAM_B2), t))
        alpha = np.float32(self.lr * np.sqrt(np.float32(1.0) - b2p) / (np.float32(1.0) - b1p))
        for w, g, m, v in zip(self.trainable(), grads, self.m, self.v):
            m.add_((g - m) * np.float32(1.0 - ADAM_B1))
            v.add_((g * g - v) * np.float32(1.0 - ADAM_B2))
            w.sub_((m * alpha) / (torch.sqrt(v) + np.float32(ADAM_EPS)))
        return loss

    # ---- inference ---------------------------------------------------------
    def predict(self, x_u8, batch_size=32):
        outs = []
        for s in range(0, len(x_u8), batch_size):
            yhat, _ = self.forward(x_u8[s : s + batch_size], False)
            outs.append(yhat)
        return torch.cat(outs).numpy() if outs else np.zeros((0, 2), np.float32)

    def evaluate(self, x_u8, y, batch_size=32):
        """Keras evaluate: sample-weighted mean of per-batch mean losses (fp32)."""
        y = torch.as_tensor(np.asarray(y, dtype=np.float32))
        total = np.float32(0.0)
        count = np.float32(0.0)
        for s in range(0, len(x_u8), batch_size):
            yhat, _ = self.forward(x_u8[s : s + batch_size], False)
            n = yhat.shape[0]
            bl = np.float32(self.loss_per_sample(yhat, y[s : s + n]).mean())
            total = np.float32(total + bl * np.float32(n))
            count = np.float32(count + np.float32(n))
        return float(np.float32(total / count))

    # ---- snapshot (ModelCheckpoint save_weights_only / load_weights) -------
    def snapshot(self):
        return [w.copy() for w in self.get_weights()]


class CallbackState:
    """ModelCheckpoint + EarlyStopping + ReduceLROnPlateau, in that order (locator.py:330-362)."""

    def __init__(self, patience, lr=1e-3):
        self.P = int(patience)
        self.rlr_patience = int(patience / 6)
        self.ckpt_best = math.inf
        self.es_best = math.inf
        self.es_wait = 0
        self.rlr_best = math.inf
        self.rlr_wait = 0
        self.lr = np.float32(lr)
        self.stop = False

    def on_epoch_end(self, epoch, val_loss):
        """Returns (save_checkpoint, lr_logged).  Mutates lr / stop."""
        save = bool(val_loss < self.ckpt_best)
        if save:
            self.ckpt_best = val_loss
        # EarlyStopping (min_delta 0, mode min): wait counted before the check
        self.es_wait += 1
        if val_loss < self.es_best:
            self.es_best = val_loss
            self.es_wait = 0
        elif self.es_wait >= self.P and epoch > 0:
            self.stop = True
        # ReduceLROnPlateau (factor .5, min_delta 0, cooldown 0, min_lr 0)
        lr_logged = float(self.lr)
        if val_loss < self.rlr_best:
            self.rlr_best = val_loss
            self.rlr_wait = 0
        else:
            self.rlr_wait += 1
            if self.rlr_wait >= self.rlr_patience:
                if float(self.lr) > 0.0:
                    self.lr = np.float32(max(float(self.lr) * 0.5, 0.0))
                self.rlr_wait = 0
        return save, lr_logged


def fit(model, traingen, trainlocs, valgen, vallocs, epochs, batch_size=32, patience=100,
        perms=None, masks=None, seed=0):
    """model.fit + reload-best (locator.py:367-388).

    perms[e]  : permutation of training rows for epoch e (default: numpy Generator(seed))
    masks(step, B): keep mask for global step `step`   (default: Philox, oracle/philox_ref.py)
    Returns history dict {loss, val_loss, learning_rate} (python floats of fp32 values).
    """
    n = len(traingen)
    rng = np.random.default_rng(seed)
    cb = CallbackState(patience, lr=float(model.lr))
    hist = {"loss": [], "val_loss": [], "learning_rate": []}
    best = None
    step = 0
    for e in range(epochs):
        perm = perms[e] if perms is not None else rng.permutation(n)
        total = np.float32(0.0)
        count = np.float32(0.0)
        for s in range(0, n, batch_size):
            rows = perm[s : s + batch_size]
            if masks is not None:
                mk = masks(step, len(rows))
            else:
                mk = philox_ref.dropout_keep(batch_size, model.H, model.p, seed, step)[: len(rows)]
            bl = np.float32(model.train_step(traingen[rows], trainlocs[rows], mk))
            total = np.float32(total + bl * np.float32(len(rows)))
            count = np.float32(count + np.float32(len(rows)))
            step += 1
        loss = float(np.float32(total / count))
        val = model.evaluate(valgen, vallocs, batch_size)
        save, lr_logged = cb.on_epoch_end(e, val)
        if save:
            best = model.snapshot()
        model.lr = cb.lr
        hist["loss"].append(loss)
        hist["val_loss"].append(val)
        hist["learning_rate"].append(lr_logged)
        if cb.stop:
            break
    if best is not None:
        model.set_weights(best)
    return hist
