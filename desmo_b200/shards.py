"""On-disk snapshot format for real data: VTK time series -> raw fp32 shards -> per-rank slabs on the device (SURVEY.md 8 f2).

The reference reads one ``.vtu`` file per time step with the ``vtk`` package and stacks the point array "velocity" into the data matrix
``X`` (rows = components at mesh points, columns = time steps; ``read_velocity_data``, CYL:39-85), then pre-processes ``X`` with numpy
on the host (CYL:88-149).  Here the time series is converted ONCE into a raw format that every rank can memory-map:

    <dir>/meta.json            {"n_points", "d_in", "m_in", "dtype": "float32" | "float64", "array", "files": [...], "steps_per_file"}
    <dir>/snapshots_00000.f32  records of n_points * d_in values, one record per time step (= the flattened "velocity" array of
                               that step = one row of X.T), ``steps_per_file`` records per file (.f64 when the source is float64)

``ShardReader.load_slab(rank, world)`` copies the columns of a rank's mesh-point slab (shard_bounds: multiples of the 128-point tile) out
of the memory maps into pinned host memory; ``DesmoEngine.preprocess_snapshot`` (desmo_preprocess: magnitude, mean removal, 1/sqrt(m),
time stride) then runs on the device, and ``pod_from_snapshot`` all-reduces the Gram across ranks.

``read_vtu_point_array`` is a dependency-free reader of the XML UnstructuredGrid files the reference consumes (the ``vtk`` package is not
needed): point-data ``DataArray``s in ascii, inline base64 ("binary", optionally zlib-compressed) and appended (raw or base64) encodings.
Host-side code only; nothing here runs on the hot path.
"""
from __future__ import annotations

import base64
import json
import os
import re
import struct
import zlib
from typing import Iterable, List, Optional, Tuple

import numpy as np

from .dist import shard_bounds

_VTK_TYPES = {"Float32": "f4", "Float64": "f8", "Int32": "i4", "Int64": "i8", "UInt32": "u4", "UInt64": "u8", "Int8": "i1", "UInt8": "u1",
              "Int16": "i2", "UInt16": "u2"}


def _decode_blocks(raw: bytes, header: str, compressed: bool, b64: bool) -> bytes:
    """Payload of a binary DataArray: [header | data] with header_type sizes; zlib blocks when a compressor is declared."""
    hs = np.dtype(header).itemsize
    if not compressed:
        if b64:
            whole = base64.b64decode(raw)
            n = int(np.frombuffer(whole[:hs], header, 1)[0])
            if len(whole) == hs:  # the size header was encoded on its own: decoding stopped at its padding
                return base64.b64decode(raw[len(base64.b64encode(whole)):])[:n]
            return whole[hs:hs + n]
        n = int(np.frombuffer(raw[:hs], header, 1)[0])
        return raw[hs:hs + n]
    # compressed: header = [nblocks, block_size, last_block_size, csize_0 .. csize_{nblocks-1}]
    if b64:
        first = base64.b64decode(raw[:((3 * hs + 2) // 3) * 4])
        nblocks = int(np.frombuffer(first, header, 1)[0])
        hbytes = (3 + nblocks) * hs
        hlen64 = ((hbytes + 2) // 3) * 4
        head = np.frombuffer(base64.b64decode(raw[:hlen64])[:hbytes], header)
        body = base64.b64decode(raw[hlen64:])
    else:
        nblocks = int(np.frombuffer(raw[:hs], header, 1)[0])
        hbytes = (3 + nblocks) * hs
        head = np.frombuffer(raw[:hbytes], header)
        body = raw[hbytes:]
    out, off = [], 0
    for c in head[3:3 + nblocks]:
        out.append(zlib.decompress(body[off:off + int(c)]))
        off += int(c)
    return b"".join(out)


def read_vtu_point_array(path: str, name: str = "velocity") -> np.ndarray:
    """The point-data array ``name`` of a VTK XML UnstructuredGrid file as (n_points, n_components) -- what
    ``VN.vtk_to_numpy(output.GetPointData().GetArray(name))`` returns in the reference (CYL:59-61)."""
    with open(path, "rb") as fh:
        blob = fh.read()
    head_end = blob.find(b"<AppendedData")
    xml_part = blob if head_end < 0 else blob[:head_end]
    text = xml_part.decode("latin-1")
    vf = re.search(r"<VTKFile([^>]*)>", text)
    if not vf:
        raise ValueError(f"{path}: not a VTK XML file")
    attrs = dict(re.findall(r'(\w+)\s*=\s*"([^"]*)"', vf.group(1)))
    header = _VTK_TYPES[attrs.get("header_type", "UInt32")]
    order = "<" if attrs.get("byte_order", "LittleEndian") == "LittleEndian" else ">"
    header = order + header
    compressed = "compressor" in attrs and "ZLib" in attrs["compressor"]
    pd = re.search(r"<PointData[^>]*>(.*?)</PointData>", text, re.S)
    if not pd:
        raise ValueError(f"{path}: no <PointData>")
    for m in re.finditer(r"<DataArray([^>]*?)(/>|>(.*?)</DataArray>)", pd.group(1), re.S):
        a = dict(re.findall(r'(\w+)\s*=\s*"([^"]*)"', m.group(1)))
        if a.get("Name") != name:
            continue
        dt = np.dtype(order + _VTK_TYPES[a["type"]])
        ncomp = int(a.get("NumberOfComponents", "1"))
        fmt = a.get("format", "ascii")
        if fmt == "ascii":
            arr = np.array(m.group(3).split(), dtype=np.float64).astype(dt)
        elif fmt == "binary":
            arr = np.frombuffer(_decode_blocks(m.group(3).strip().encode("latin-1"), header, compressed, True), dt)
        elif fmt == "appended":
            app = re.search(rb'<AppendedData[^>]*encoding\s*=\s*"(\w+)"[^>]*>\s*_', blob)
            if not app:
                raise ValueError(f"{path}: appended data section missing")
            start = app.end() + int(a["offset"])
            if app.group(1) == b"raw":
                arr = np.frombuffer(_decode_blocks(blob[start:], header, compressed, False), dt)
            else:
                end = blob.find(b"<", start)
                arr = np.frombuffer(_decode_blocks(blob[start:end].strip(), header, compressed, True), dt)
        else:
            raise ValueError(f"{path}: unknown DataArray format {fmt!r}")
        return np.ascontiguousarray(arr.reshape(-1, ncomp))
    raise KeyError(f"{path}: no point-data array named {name!r}")


def write_raw_shards(snapshots: Iterable[np.ndarray], out_dir: str, steps_per_file: int = 256, array: str = "velocity",
                     dtype: Optional[str] = None) -> dict:
    """Writes the raw shard format from an iterable of per-step arrays (n_points, d_in) (or flat n_points * d_in).  ``dtype`` is
    "float32" or "float64"; by default float64 sources stay float64 (the reference pre-processes in fp64 and casts afterwards,
    CYL:109-149,356 -- desmo_preprocess does the same on the device) and everything else is stored as float32."""
    os.makedirs(out_dir, exist_ok=True)
    files: List[str] = []
    fh = None
    n_points = d_in = None
    m_in = 0
    for step, snap in enumerate(snapshots):
        v = np.asarray(snap)
        if v.ndim == 1:
            v = v.reshape(-1, 1)
        if n_points is None:
            n_points, d_in = v.shape
            if dtype is None:
                dtype = "float64" if v.dtype == np.float64 else "float32"
            if dtype not in ("float32", "float64"):
                raise ValueError("dtype must be float32 or float64")
            ext, code = (".f64", "<f8") if dtype == "float64" else (".f32", "<f4")
        elif v.shape != (n_points, d_in):
            raise ValueError(f"step {step}: shape {v.shape} differs from the first step's {(n_points, d_in)}")
        if step % steps_per_file == 0:
            if fh:
                fh.close()
            files.append(f"snapshots_{len(files):05d}{ext}")
            fh = open(os.path.join(out_dir, files[-1]), "wb")
        fh.write(np.ascontiguousarray(v, dtype=code).tobytes())
        m_in += 1
    if fh:
        fh.close()
    if m_in == 0:
        raise ValueError("no snapshots")
    meta = {"n_points": int(n_points), "d_in": int(d_in), "m_in": int(m_in), "dtype": dtype, "array": array, "files": files,
            "steps_per_file": int(steps_per_file), "layout": "one record of n_points*d_in float32 per time step (row of X.T, CYL:68-72)"}
    with open(os.path.join(out_dir, "meta.json"), "w") as out:
        json.dump(meta, out, indent=1)
    return meta


def convert_vtu_series(input_dir: str, filename: str, t_1: int, t_n: int, out_dir: str, array: str = "velocity",
                       steps_per_file: int = 256) -> dict:
    """``read_velocity_data(input_dir, filename, reader, t_1, t_n)`` (CYL:39-85) as a one-off conversion: steps ``range(t_1, t_n)`` of
    ``input_dir + filename + str(i) + '.vtu'`` -> raw fp32 shards."""
    return write_raw_shards((read_vtu_point_array(os.path.join(input_dir, f"{filename}{i}.vtu"), array) for i in range(t_1, t_n)),
                            out_dir, steps_per_file, array)


class ShardReader:
    """Memory-maps a raw shard directory; hands out per-rank slabs of mesh points in the reader layout V[m_in][n_local * d_in]."""

    def __init__(self, shard_dir: str):
        with open(os.path.join(shard_dir, "meta.json")) as fh:
            self.meta = json.load(fh)
        self.dir = shard_dir
        self.n_points, self.d_in, self.m_in = self.meta["n_points"], self.meta["d_in"], self.meta["m_in"]
        rec = self.n_points * self.d_in
        self.np_dtype = "<f8" if self.meta.get("dtype", "float32") == "float64" else "<f4"
        self.maps = []
        left = self.m_in
        for f in self.meta["files"]:
            steps = min(left, self.meta["steps_per_file"])
            self.maps.append(np.memmap(os.path.join(shard_dir, f), dtype=self.np_dtype, mode="r", shape=(steps, rec)))
            left -= steps

    def slab_bounds(self, rank: int, world: int) -> Tuple[int, int]:
        return shard_bounds(self.n_points, world, rank)

    def load_slab(self, rank: int = 0, world: int = 1, out: Optional[np.ndarray] = None, pinned: bool = False):
        """(m_in, n_local * d_in) in the stored dtype: the rank's columns of every record.  ``pinned=True`` returns a pinned torch tensor."""
        lo, hi = self.slab_bounds(rank, world)
        cols = (hi - lo) * self.d_in
        if pinned:
            import torch

            t = torch.empty(self.m_in, cols, dtype=torch.float64 if self.np_dtype == "<f8" else torch.float32,
                            pin_memory=torch.cuda.is_available())
            out = t.numpy()
        elif out is None:
            out = np.empty((self.m_in, cols), self.np_dtype)
        row = 0
        for mp in self.maps:
            out[row:row + mp.shape[0]] = mp[:, lo * self.d_in:hi * self.d_in]
            row += mp.shape[0]
        return t if pinned else out

    def data_matrix(self) -> np.ndarray:
        """The reference's X (n_points * d_in rows, m_in columns, fp64; CYL:64-68) -- for tests and small cases only."""
        return np.concatenate([np.asarray(mp) for mp in self.maps], axis=0).T.astype(np.float64)


def model_from_shards(shard_dir: str, polyorder: int, r_DESMO: int, omega_init: float = 10000.0, *, d_use: Optional[int] = None,
                      magnitude: bool = True, subtract_mean: bool = True, scale_sqrt_m: bool = False, t_stride: int = 1, nF: Optional[int] = None,
                      period_init: float = 60.0, device=None, path: int = 0, snapshot_dtype=None):
    """Data ingest + pre-processing + POD init of the scripts (CYL:157-205, ANEU:143, TURB:189) for this rank's slab: returns
    (model, X_mean [n_local] fp64, singular values).  Under torch.distributed every rank calls it; the Gram is all-reduced.
    ``snapshot_dtype=torch.bfloat16`` pre-processes straight into bf16 storage (default: fp32)."""
    import torch
    import torch.distributed as dist

    from .model import DESMO, DESMOFourier

    rd = ShardReader(shard_dir)
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    lo, hi = rd.slab_bounds(rank, world)
    d_use = rd.d_in if d_use is None else d_use
    if not magnitude and rd.d_in != 1:
        raise ValueError("without magnitude every component is its own row: write the shards with d_in = 1")
    n_local, n_global = hi - lo, rd.n_points
    m = (rd.m_in + t_stride - 1) // t_stride
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    kw = dict(device=dev, n_global=n_global, path=path, snapshot_dtype=snapshot_dtype or torch.float32)
    model = (DESMOFourier(n_local, m, polyorder, r_DESMO, omega_init, nF, period_init=period_init, **kw) if nF
             else DESMO(n_local, m, polyorder, r_DESMO, omega_init, **kw))
    raw = rd.load_slab(rank, world, pinned=True).to(dev, non_blocking=True)
    mean = model.engine.preprocess_snapshot(raw, d_in=rd.d_in, d_use=d_use, magnitude=magnitude, subtract_mean=subtract_mean,
                                            scale_sqrt_m=scale_sqrt_m, t_stride=t_stride)
    sigma = model.engine.pod_from_snapshot()
    return model, mean, sigma
