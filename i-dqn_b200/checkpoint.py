"""On-disk checkpoint format: one directory per checkpoint, written as ``.<name>.tmp/`` and renamed to ``<name>/`` once
every file is on disk and ``manifest.json`` (format version, serial number, every file and its size) has been written
last.  A directory without a manifest is an interrupted save and is never read.  Arrays are ``.npy`` files; large ones
are streamed in chunks with plain file reads and writes.  Also the host restatement of the replay store's digest
(``idqn_replay_digest``, csrc/checkpoint.cu)."""
from __future__ import annotations

import json
import os
import shutil

import numpy as np

FORMAT_VERSION = 1
MANIFEST = "manifest.json"
CHUNK_BYTES = 256 << 20  # device <-> file streaming unit


def write_json(path: str, obj) -> None:
    with open(path, "w") as f:
        json.dump(obj, f, indent=1, default=lambda o: o.item())  # numpy scalars as Python numbers


def read_json(path: str):
    with open(path) as f:
        return json.load(f)


class NpyWriter:
    """A ``.npy`` file of ``shape``/``dtype`` filled by successive ``write(chunk)`` calls along the first axis."""

    def __init__(self, path: str, shape, dtype):
        self.f = open(path, "wb")
        np.lib.format.write_array_header_1_0(self.f, {"descr": np.lib.format.dtype_to_descr(np.dtype(dtype)),
                                                      "fortran_order": False, "shape": tuple(int(s) for s in shape)})

    def write(self, chunk: np.ndarray) -> None:
        self.f.write(np.ascontiguousarray(chunk).data)

    def close(self) -> None:
        self.f.close()


class NpyReader:
    """Reads a ``.npy`` file ``n`` leading-axis entries at a time (``read(n)``)."""

    def __init__(self, path: str):
        self.f = open(path, "rb")
        np.lib.format.read_magic(self.f)
        self.shape, fortran, self.dtype = np.lib.format.read_array_header_1_0(self.f)
        assert not fortran

    def read(self, n: int) -> np.ndarray:
        out = np.empty((n,) + tuple(self.shape[1:]), self.dtype)
        if self.f.readinto(memoryview(out.reshape(-1)).cast("B")) != out.nbytes:
            raise ValueError(f"{self.f.name}: file ends early")
        return out

    def close(self) -> None:
        self.f.close()


def rows_per_chunk(row_bytes: int) -> int:
    return max(1, CHUNK_BYTES // max(1, int(row_bytes)))


def _fsync(path: str, directory: bool = False) -> None:
    fd = os.open(path, os.O_RDONLY | (os.O_DIRECTORY if directory else 0))
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


def _complete(root: str):
    """(serial, name) of every complete checkpoint under root."""
    out = []
    for name in os.listdir(root) if os.path.isdir(root) else ():
        path = os.path.join(root, name, MANIFEST)
        if not name.startswith(".") and os.path.isfile(path):
            out.append((int(read_json(path)["serial"]), name))
    return sorted(out)


def begin(root: str, name: str) -> str:
    """A fresh ``root/.<name>.tmp`` directory to write checkpoint ``name`` into."""
    tmp = os.path.join(root, f".{name}.tmp")
    shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(tmp)
    return tmp


def commit(root: str, name: str, keep: int | None = None) -> str:
    """fsync every file of ``root/.<name>.tmp``, write its manifest last, rename it to ``root/<name>``; then delete all
    but the newest ``keep`` complete checkpoints."""
    tmp = os.path.join(root, f".{name}.tmp")
    files = {}
    for d, _, names in os.walk(tmp):
        for n in names:
            p = os.path.join(d, n)
            _fsync(p)
            files[os.path.relpath(p, tmp)] = os.path.getsize(p)
        _fsync(d, directory=True)
    serial = max((s for s, _ in _complete(root)), default=0) + 1
    write_json(os.path.join(tmp, MANIFEST), {"format": FORMAT_VERSION, "serial": serial, "files": dict(sorted(files.items()))})
    _fsync(os.path.join(tmp, MANIFEST))
    final = os.path.join(root, name)
    shutil.rmtree(final, ignore_errors=True)
    os.rename(tmp, final)
    _fsync(root, directory=True)
    if keep is not None:
        for _, old in _complete(root)[:-max(int(keep), 1)]:
            shutil.rmtree(os.path.join(root, old))
    return final


def latest_checkpoint(root: str) -> str | None:
    """The newest complete checkpoint under ``root`` (None if there is none); leftovers of interrupted saves are ignored."""
    done = _complete(root)
    return os.path.join(root, done[-1][1]) if done else None


def verify(path: str) -> None:
    """ValueError unless ``path`` is a complete checkpoint of this format whose files have their recorded sizes."""
    m = read_json(os.path.join(path, MANIFEST))
    if m.get("format") != FORMAT_VERSION:
        raise ValueError(f"{path}: checkpoint format {m.get('format')}, this version reads {FORMAT_VERSION}")
    for rel, size in m["files"].items():
        p = os.path.join(path, rel)
        if not os.path.isfile(p) or os.path.getsize(p) != size:
            raise ValueError(f"{path}: {rel} is missing or has the wrong size")


# ---- digest (idqn_replay_digest) --------------------------------------------------------------------------------------
def _splitmix64(z: np.ndarray) -> np.ndarray:
    z = z ^ (z >> np.uint64(30))
    z = z * np.uint64(0xBF58476D1CE4E5B9)
    z = z ^ (z >> np.uint64(27))
    z = z * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def digest(data) -> int:
    """``(sum_i splitmix64(w_i + (i+1) * 0x9E3779B97F4A7C15)) mod 2^64 XOR splitmix64(L)`` of a byte stream of length L
    read as zero-padded little-endian 64-bit words w_i."""
    if isinstance(data, (bytes, bytearray, memoryview)):
        b = np.frombuffer(data, np.uint8)
    else:
        b = np.ascontiguousarray(data).reshape(-1).view(np.uint8)
    n = len(b)
    words = np.zeros((n + 7) // 8 * 8, np.uint8)
    words[:n] = b
    w = words.view("<u8").astype(np.uint64)
    i = np.arange(1, len(w) + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        s = int(_splitmix64(w + i * np.uint64(0x9E3779B97F4A7C15)).sum(dtype=np.uint64))
        return s ^ int(_splitmix64(np.asarray([n], np.uint64))[0])


def frames_digest(frames: np.ndarray) -> int:
    """The digest of a run of frames ([n, ...]) as the frame store computes it: each frame zero-padded to 8 bytes."""
    f = np.ascontiguousarray(frames)
    f = f.reshape(len(f), int(np.prod(f.shape[1:]))).view(np.uint8)
    pad = (-f.shape[1]) % 8
    return digest(np.pad(f, ((0, 0), (0, pad))) if pad else f)
