"""Network side of the drop-in: the NNetWrapper contract (Net/NNet.py:22-101) over the bf16 tcgen05
OthelloNNet tower in liboz_b200.so.

Weights travel as ONE float32 blob in Keras ``model.get_weights()`` order for the graph of
Net/OthelloNN.py:42-52 (kernel HWIO / Dense (in,out), bias, then BN gamma, beta, moving_mean,
moving_variance after each of the six conv/dense blocks, then the two heads).
"""
from __future__ import annotations

import enum

import numpy as np

from . import engine as _engine
from ._lib import PRIOR_NET, channels_arg


class NeuralNets(enum.Enum):
    """Net/NNet.py:14-16."""
    ONN = enum.auto()
    BNN = enum.auto()


def blob_layout(board_size: int, channels: int = 512):
    """[(name, shape)] in blob order."""
    n, C = board_size, channels
    k1 = (n - 4) * (n - 4) * C
    L = []

    def bn(prefix, c):
        L.extend([(f"{prefix}.gamma", (c,)), (f"{prefix}.beta", (c,)), (f"{prefix}.mean", (c,)), (f"{prefix}.var", (c,))])

    L += [("conv1.kernel", (3, 3, 2, C)), ("conv1.bias", (C,))]
    bn("bn1", C)
    for i in (2, 3, 4):
        L += [(f"conv{i}.kernel", (3, 3, C, C)), (f"conv{i}.bias", (C,))]
        bn(f"bn{i}", C)
    L += [("fc1.kernel", (k1, 1024)), ("fc1.bias", (1024,))]
    bn("bn5", 1024)
    L += [("fc2.kernel", (1024, 512)), ("fc2.bias", (512,))]
    bn("bn6", 512)
    L += [("pi.kernel", (512, n * n)), ("pi.bias", (n * n,)), ("v.kernel", (512, 1)), ("v.bias", (1,))]
    return L


def blob_size(board_size: int, channels: int = 512) -> int:
    return int(sum(int(np.prod(s)) for _, s in blob_layout(board_size, channels)))


def unpack_blob(blob: np.ndarray, board_size: int, channels: int = 512) -> dict:
    out, off = {}, 0
    for name, shape in blob_layout(board_size, channels):
        cnt = int(np.prod(shape))
        out[name] = blob[off:off + cnt].reshape(shape)
        off += cnt
    assert off == blob.size, "blob size mismatch"
    return out


def pack_blob(weights: dict, board_size: int, channels: int = 512) -> np.ndarray:
    return np.concatenate([np.asarray(weights[name], dtype=np.float32).reshape(-1)
                           for name, _ in blob_layout(board_size, channels)])


# ---- Keras .h5 weight files (Net/NNet.py:89-96: model.save_weights(path, save_format='h5') / load_weights) -------------
# File layout written by Keras 2.4 (requirements.txt:35): root (or the 'model_weights' group of a full-model file) has the
# attribute 'layer_names' = every layer of model.layers in order; each layer group has 'weight_names' and one dataset per
# weight.  Concatenated in that order this is model.get_weights(), i.e. exactly the blob order of blob_layout().
# The HDF5 container itself is read/written by h5py (not installed in the authoring image, so the import is deferred and
# the mapping is tested against a stand-in group object, tests/test_h5_mapping_cpu.py).
KERAS_LAYER_NAMES = [("conv2d", "conv1", "bn1", "batch_normalization"), ("conv2d_1", "conv2", "bn2", "batch_normalization_1"),
                     ("conv2d_2", "conv3", "bn3", "batch_normalization_2"), ("conv2d_3", "conv4", "bn4", "batch_normalization_3"),
                     ("dense", "fc1", "bn5", "batch_normalization_4"), ("dense_1", "fc2", "bn6", "batch_normalization_5")]


def _txt(x) -> str:
    return x.decode() if isinstance(x, (bytes, np.bytes_)) else str(x)


def blob_from_h5_group(root, board_size: int, channels: int = 512) -> np.ndarray:
    """`root`: an h5py.File / Group (anything with .attrs, `in` and [] access) holding Keras layer groups."""
    g = root["model_weights"] if "model_weights" in root else root
    arrays = []
    for ln in g.attrs["layer_names"]:
        grp = g[_txt(ln)]
        for wn in grp.attrs["weight_names"]:
            arrays.append(np.asarray(grp[_txt(wn)], dtype=np.float32))
    layout = blob_layout(board_size, channels)
    if len(arrays) != len(layout):
        raise ValueError(f"checkpoint holds {len(arrays)} weight arrays, OthelloNN({board_size}x{board_size}, C={channels}) "
                         f"has {len(layout)}")
    for a, (name, shape) in zip(arrays, layout):
        if tuple(a.shape) != tuple(shape):
            raise ValueError(f"checkpoint array for {name} has shape {tuple(a.shape)}, expected {tuple(shape)}")
    return np.concatenate([a.reshape(-1) for a in arrays]).astype(np.float32)


def write_h5_group(root, blob: np.ndarray, board_size: int, channels: int = 512):
    """Fills `root` (h5py.File / Group, or a stand-in with .attrs, create_group, create_dataset) the way Keras does."""
    w = unpack_blob(np.asarray(blob, dtype=np.float32), board_size, channels)
    layers = []
    for lname, key, bnkey, bnname in KERAS_LAYER_NAMES:
        layers.append((lname, [(f"{lname}/kernel:0", w[f"{key}.kernel"]), (f"{lname}/bias:0", w[f"{key}.bias"])]))
        layers.append((bnname, [(f"{bnname}/gamma:0", w[f"{bnkey}.gamma"]), (f"{bnname}/beta:0", w[f"{bnkey}.beta"]),
                                (f"{bnname}/moving_mean:0", w[f"{bnkey}.mean"]),
                                (f"{bnname}/moving_variance:0", w[f"{bnkey}.var"])]))
    for head in ("pi", "v"):
        layers.append((head, [(f"{head}/kernel:0", w[f"{head}.kernel"]), (f"{head}/bias:0", w[f"{head}.bias"])]))
    root.attrs["layer_names"] = [ln.encode() for ln, _ in layers]
    root.attrs["backend"] = b"tensorflow"
    root.attrs["keras_version"] = b"2.4.0"
    for ln, weights in layers:
        grp = root.create_group(ln)
        grp.attrs["weight_names"] = [wn.encode() for wn, _ in weights]
        for wn, arr in weights:
            grp.create_dataset(wn, data=np.ascontiguousarray(arr, dtype=np.float32))


def _h5py():
    try:
        import h5py
        return h5py
    except ImportError as e:  # pragma: no cover - h5py is absent in the authoring image
        raise RuntimeError("Keras .h5 checkpoints need the h5py package (pip install h5py); "
                           "use a .npz path for the native format") from e


def load_keras_h5(filepath, board_size: int, channels: int = 512) -> np.ndarray:
    with _h5py().File(filepath, "r") as f:
        return blob_from_h5_group(f, board_size, channels)


def save_keras_h5(filepath, blob: np.ndarray, board_size: int, channels: int = 512):
    with _h5py().File(filepath, "w") as f:
        write_h5_group(f, blob, board_size, channels)


def init_weights(board_size: int, channels: int = 512, seed: int = 0, randomize_bn: bool = False) -> np.ndarray:
    """Keras defaults: glorot-uniform kernels, zero biases, BN gamma=1 beta=0 mean=0 var=1 (SURVEY §8c).
    randomize_bn=True perturbs BN statistics / biases so that folding is exercised by the tests."""
    rng = np.random.default_rng(seed)
    w = {}
    for name, shape in blob_layout(board_size, channels):
        kind = name.split(".")[1]
        if kind == "kernel":
            if len(shape) == 4:
                fan_in, fan_out = shape[0] * shape[1] * shape[2], shape[0] * shape[1] * shape[3]
            else:
                fan_in, fan_out = shape
            lim = np.sqrt(6.0 / (fan_in + fan_out))
            w[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)
        elif kind in ("bias", "beta", "mean"):
            w[name] = (rng.normal(0, 0.1, size=shape) if randomize_bn else np.zeros(shape)).astype(np.float32)
        elif kind == "gamma":
            w[name] = (rng.uniform(0.5, 1.5, size=shape) if randomize_bn else np.ones(shape)).astype(np.float32)
        elif kind == "var":
            w[name] = (rng.uniform(0.5, 2.0, size=shape) if randomize_bn else np.ones(shape)).astype(np.float32)
    return pack_blob(w, board_size, channels)


_SQUARE_BIT = (np.uint64(1) << (np.arange(8, dtype=np.uint64)[:, None] * np.uint64(8) + np.arange(8, dtype=np.uint64)[None, :]))


def boards_to_bits(boards) -> tuple[np.ndarray, np.ndarray]:
    """(B,N,N,2) bool/0-1 array -> (ch0 bits, ch1 bits) uint64, bit r*8+c."""
    b = np.asarray(boards).astype(bool)
    if b.ndim == 3:
        b = b[None]
    n = b.shape[1]
    w = _SQUARE_BIT[:n, :n]
    own = (b[..., 0] * w).sum(axis=(1, 2), dtype=np.uint64)
    opp = (b[..., 1] * w).sum(axis=(1, 2), dtype=np.uint64)
    return own, opp


def bits_to_board(ch0: int, ch1: int, n: int) -> np.ndarray:
    """-> (N,N,2) bool array in the reference's layout (Othello/__init__.py:22-25)."""
    words = np.array([int(ch0), int(ch1)], dtype="<u8").view(np.uint8).reshape(2, 8)     # byte r of a word = row r
    planes = np.unpackbits(words, axis=1, bitorder="little").reshape(2, 8, 8)[:, :n, :n]
    return np.ascontiguousarray(np.moveaxis(planes, 0, -1)).astype(bool)


class B200NNet:
    """NNetWrapper stand-in (Net/NNet.py:22-101) whose predict runs on the B200 tower.

    ``predict(board (N,N,2)) -> (pi (N,N) float32 probabilities, v float32)`` — Net/NNet.py:70-87.
    ``train`` is not part of the self-play hot path (SURVEY §8f rank 3) and raises.
    ``precision``: "bf16" (default) or "fp8" (conv3, conv4 and fc1 on e4m3 tcgen05 MMAs, DESIGN.md 13).  Self-play and
    the arena evaluate a net at its own precision; training stays fp32.
    """

    def __init__(self, board_size=(8, 8), num_channels_1: int = 512, network=NeuralNets.ONN, device: int = 0,
                 max_batch: int = 4096, seed: int = 0, blob: np.ndarray | None = None, precision: str = "bf16"):
        if network is not NeuralNets.ONN:
            raise TypeError("only NeuralNets.ONN is implemented on the B200 path (BNN is out of scope)")
        self.board_size_x, self.board_size_y = board_size
        assert self.board_size_x == self.board_size_y, "square boards only"
        self.action_size = self.board_size_x * self.board_size_y
        self.network_type = network
        self.channels = num_channels_1
        self.device = device
        self.max_batch = max_batch
        channels_arg(num_channels_1, precision)  # ValueError before any device work
        self.precision = precision
        self.blob = blob if blob is not None else init_weights(self.board_size_x, num_channels_1, seed)
        self._eng = _engine.Engine(self.board_size_x, max_games=max_batch, nodes_per_game=2, prior_mode=PRIOR_NET,
                                   device=device)
        self._eng.load_weights(self.blob, self.channels, precision)

    def set_weights(self, blob: np.ndarray):
        self.blob = np.ascontiguousarray(blob, dtype=np.float32)
        self._eng.load_weights(self.blob, self.channels, self.precision)

    def fp8_scales(self) -> dict:
        """Engine.fp8_scales of this (precision="fp8") net."""
        return self._eng.fp8_scales()

    def predict_batch(self, own, opp, want_logits: bool = False):
        """Canonical bitboards -> (pi [B,N*N], v [B]) (+ logits)."""
        pi, lg, v = self._eng.net_forward(own, opp, want_logits=want_logits)
        return (pi, lg, v) if want_logits else (pi, v)

    def predict(self, board):
        own, opp = boards_to_bits(board)
        pi, v = self.predict_batch(own, opp)
        return pi[0].reshape(self.board_size_x, self.board_size_y), np.float32(v[0])

    def train(self, examples, verbose=None, epochs: int = 10, batch_size: int = 32, lr: float = 1e-3,
              dropout: float = 0.3):
        """Net/NNet.py:53-68 with the compile settings of Net/OthelloNN.py:55-56 (PyTorch autograd; see train.py).
        The trained weights are folded and re-loaded onto the device tower."""
        from .train import train_blob
        blob, history = train_blob(self.blob, examples, self.board_size_x, self.channels, epochs=epochs,
                                   batch_size=batch_size, lr=lr, dropout=dropout, verbose=bool(verbose))
        self.set_weights(blob)
        return history

    def save_checkpoint(self, filepath):
        """Net/NNet.py:89-91.  '.h5' paths are written in Keras' save_weights layout (needs h5py); anything else is the
        native .npz (float32 blob in Keras get_weights() order)."""
        if str(filepath).endswith(".h5"):
            return save_keras_h5(filepath, self.blob, self.board_size_x, self.channels)
        np.savez(filepath, blob=self.blob, board_size=self.board_size_x, channels=self.channels)

    def load_checkpoint(self, filepath):
        """Net/NNet.py:93-96 ('.h5' = a Keras save_weights file of the reference's NNetWrapper; needs h5py)."""
        if str(filepath).endswith(".h5"):
            return self.set_weights(load_keras_h5(filepath, self.board_size_x, self.channels))
        d = np.load(filepath if str(filepath).endswith(".npz") else str(filepath) + ".npz")
        assert int(d["board_size"]) == self.board_size_x and int(d["channels"]) == self.channels
        self.set_weights(d["blob"])

    def copy(self):
        return B200NNet((self.board_size_x, self.board_size_y), self.channels, self.network_type, self.device,
                        self.max_batch, blob=self.blob.copy(), precision=self.precision)
