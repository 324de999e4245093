"""Weight files for the engine.

File format "FILMW1" (little-endian), read by csrc/film_weights.cpp without Python:

    8 bytes   magic  b"FILMW1\\0\\0"
    u32       number of tensors
    repeat:   u32 name_len, name bytes (utf-8), u32 ndim, u32 dims[ndim], f32 data[prod(dims)]

Tensor names and shapes are `spec.weight_table()`: Keras HWIO kernels + biases,
named after the reference's layers (`feature_extractor.py:118-123`,
`pyramid_flow_estimator.py:76-83,115,119`, `fusion.py:76-101`).

There is no pre-trained SavedModel and no TensorFlow in the build container
(SURVEY.md section 8c), so tests and benchmarks use `synthetic_weights()`: seeded
He-scaled tensors tuned so activations stay O(1) and level-0 flows are a few pixels
(otherwise the warps would be degenerate and parity vacuous). `from_named_arrays()`
is the import hook for real weights (a dict of numpy arrays keyed by the SavedModel
variable names, e.g. from `tf.train.load_checkpoint` on a machine that has TF).
"""
from __future__ import annotations

import hashlib
import os
import struct
from typing import Dict, Mapping

import numpy as np

from . import spec

MAGIC = b"FILMW1\0\0"


def save(path: str, tensors: Mapping[str, np.ndarray]) -> None:
    table = spec.weight_table()
    with open(path, "wb") as f:
        f.write(MAGIC)
        f.write(struct.pack("<I", len(table)))
        for name, shape in table:
            a = np.ascontiguousarray(tensors[name], dtype="<f4")
            if tuple(a.shape) != tuple(shape):
                raise ValueError(f"{name}: shape {a.shape} != expected {shape}")
            nb = name.encode()
            f.write(struct.pack("<I", len(nb)))
            f.write(nb)
            f.write(struct.pack("<I", a.ndim))
            f.write(struct.pack(f"<{a.ndim}I", *a.shape))
            f.write(a.tobytes())


def load(path: str) -> Dict[str, np.ndarray]:
    out: Dict[str, np.ndarray] = {}
    with open(path, "rb") as f:
        if f.read(8) != MAGIC:
            raise ValueError(f"{path}: not a FILMW1 weight file")
        (n,) = struct.unpack("<I", f.read(4))
        for _ in range(n):
            (ln,) = struct.unpack("<I", f.read(4))
            name = f.read(ln).decode()
            (nd,) = struct.unpack("<I", f.read(4))
            dims = struct.unpack(f"<{nd}I", f.read(4 * nd))
            cnt = int(np.prod(dims))
            out[name] = np.frombuffer(f.read(4 * cnt), dtype="<f4").reshape(dims).copy()
    expect = dict(spec.weight_table())
    if set(out) != set(expect):
        raise ValueError("weight file does not match the Style architecture table")
    for k, s in expect.items():
        if tuple(out[k].shape) != tuple(s):
            raise ValueError(f"{k}: shape {out[k].shape} != {s}")
    return out


def digest(tensors: Mapping[str, np.ndarray]) -> str:
    h = hashlib.sha256()
    for name, _ in spec.weight_table():
        h.update(name.encode())
        h.update(np.ascontiguousarray(tensors[name], dtype="<f4").tobytes())
    return h.hexdigest()


def synthetic_weights(seed: int = 1234) -> Dict[str, np.ndarray]:
    """Deterministic random-init weights of the Style architecture.

    He-normal for LeakyReLU(0.2) stacks; the last (linear) flow conv of every
    predictor is scaled so that per-level residual flows are ~0.1 px rms, which after
    the x2-per-level accumulation (pyramid_flow_estimator.py:154-161) gives level-0
    flows of several pixels. Biases are small but non-zero so bias-add is exercised.
    """
    rng = np.random.default_rng(seed)
    out: Dict[str, np.ndarray] = {}
    gain = float(np.sqrt(2.0 / (1.0 + spec.LEAKY_SLOPE ** 2)))
    for name, shape in spec.weight_table():
        if name.endswith("/bias"):
            out[name] = (0.05 * rng.standard_normal(shape)).astype(np.float32)
            continue
        kh, kw, cin, cout = shape
        fan_in = kh * kw * cin
        std = gain / np.sqrt(fan_in)
        if name.startswith("predict_flow/") and cout == 2:
            std = 0.12 / np.sqrt(fan_in)          # residual flow ~0.1 px rms
        elif name == "fusion/output_conv/kernel":
            std = 0.12 / np.sqrt(fan_in)          # RGB head, linear; output O(0.1) around the bias
        elif name.startswith("fusion/") and kh == 2:
            std = 1.0 / np.sqrt(fan_in)           # linear 2x2 conv (fusion.py:83-84)
        elif name.endswith("cfeat_conv_0/kernel"):
            std = 2.5 * gain / np.sqrt(fan_in)    # inputs live in [0,1], boost first layer
        out[name] = (std * rng.standard_normal(shape)).astype(np.float32)
    # output bias so the synthetic "image" sits in a plausible range
    out["fusion/output_conv/bias"] = np.array([0.45, 0.5, 0.55], np.float32)
    return out


def from_named_arrays(arrays: Mapping[str, np.ndarray], partial: bool = False) -> Dict[str, np.ndarray]:
    """Map SavedModel variable names to the engine's table.

    `partial=True` returns whatever could be mapped (no completeness / shape check): used by the
    TensorBundle importer to merge with keys it resolved another way.

    Accepts the reference's variable names. Feature-extractor and flow-predictor
    variables carry explicit layer names; fusion convs are unnamed Keras layers
    (`fusion.py:82-101`) whose auto-names depend on a global counter, so they are
    matched by creation order (conv2d, conv2d_1, ... sorted numerically) and shape.
    """
    out: Dict[str, np.ndarray] = {}
    table = dict(spec.weight_table())

    def strip(k: str) -> str:
        k = k.replace(":0", "")
        for pre in ("model/", "film_net/"):
            if k.startswith(pre):
                k = k[len(pre):]
        return k

    named = {strip(k): np.asarray(v, np.float32) for k, v in arrays.items()}
    fusion_layers: Dict[int, Dict[str, np.ndarray]] = {}
    for k, v in named.items():
        if k in table and not k.startswith("fusion/"):
            out[k] = v
            continue
        parts = k.split("/")
        if len(parts) >= 3 and parts[0] == "fusion" and parts[1].startswith("conv2d"):
            suffix = parts[1][len("conv2d"):].lstrip("_")
            idx = int(suffix) if suffix else 0
            fusion_layers.setdefault(idx, {})[parts[2]] = v
    order = sorted(fusion_layers)
    names = [f"fusion/level_{i}/conv_{j}" for i in range(spec.FUSION_PYRAMID_LEVELS - 1)
             for j in range(3)] + ["fusion/output_conv"]
    if order and len(order) != len(names):
        if partial:
            return out
        raise ValueError(f"expected {len(names)} fusion convs, found {len(order)}")
    for idx, nm in zip(order, names):
        layer = fusion_layers[idx]
        if "kernel" not in layer or "bias" not in layer:
            if partial:
                continue
            raise ValueError(f"fusion conv #{idx} is missing its kernel or bias")
        # creation order must also agree with the shapes (a reordered counter would be caught here)
        if tuple(layer["kernel"].shape) != tuple(table[nm + "/kernel"]):
            if partial:
                continue
            raise ValueError(f"fusion conv #{idx} ({nm}): kernel shape {layer['kernel'].shape} != {table[nm + '/kernel']}")
        out[nm + "/kernel"] = layer["kernel"]
        out[nm + "/bias"] = layer["bias"]
    if partial:
        return out
    missing = set(table) - set(out)
    if missing:
        raise ValueError(f"missing variables: {sorted(missing)[:5]} ...")
    for k, s in table.items():
        if tuple(out[k].shape) != tuple(s):
            raise ValueError(f"{k}: shape {out[k].shape} != {s}")
    return out


def ensure_synthetic_file(path: str | None = None, seed: int = 1234) -> str:
    """Write the synthetic weight file once (cache dir under the system temp dir) and return its path.

    The default cache dir is per user: on a shared host the temp dir is shared, and a cache dir another user
    created there is not writable."""
    if path is None:
        import tempfile
        root = os.environ.get("FILM_B200_CACHE",
                              os.path.join(tempfile.gettempdir(), f"film_b200_cache-{os.getuid()}"))
        os.makedirs(root, exist_ok=True)
        path = os.path.join(root, f"synthetic_seed{seed}.filmw")
    if not os.path.exists(path):
        tmp = f"{path}.tmp{os.getpid()}"
        save(tmp, synthetic_weights(seed))
        os.replace(tmp, path)
    return path
