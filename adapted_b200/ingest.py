"""File-level driver of the hot path: signal container -> GPU detection -> boundary tables.

Stands in for the part of ``adapted detect`` / ``adapted continue`` between the pod5 reader and the CSV files
(adapted/file_proc.py:143-214 producer, 217-266 worker, 312-457 saver threads, 97-140 continue logic).  ``pod5`` is
not installable in the build image (SURVEY.md section 8 f1), so the input is the native container -- the same
information a pod5 file holds per read: int16 ADC samples truncated to the preload window, the calibration pair, the
untruncated length and the read id.  Reads are cut into minibatches in file order (parser.py:95-99), results are
written 4000 reads per table like the reference's savers; a minibatch the reference loses on an exception outside its
per-read ``try`` (SURVEY.md A.11) is logged and appears in neither table, as there.
"""
from __future__ import annotations

import logging
import os
from typing import Any, Dict, Iterable, Iterator, List, Optional, Sequence, Set, Tuple

import numpy as np

from .config import flatten_config
from .output import BoundaryTableWriter

CONTAINER_KEYS = ("adc", "offsets", "full_lens", "calib_offset", "calib_scale", "read_ids")
_MAGIC = b"ADBSIG01"


def write_container(path: str, adc: np.ndarray, offsets: np.ndarray, full_lens: np.ndarray, calib_offset: np.ndarray,
                    calib_scale: np.ndarray, read_ids: Sequence[str]) -> str:
    """One file: magic, a JSON header, then 64-byte aligned raw sections (int64 offsets, int32 lengths, float32
    calibration pairs, fixed-width read ids, the int16 blob) -- read back as memory maps, nothing is parsed or copied."""
    import json

    if not path.endswith(".adbsig"):
        path += ".adbsig"
    ids = np.asarray([str(i).encode() for i in read_ids], dtype="S") if len(read_ids) else np.zeros(0, "S1")
    arrays = [("offsets", np.ascontiguousarray(offsets, np.int64)), ("full_lens", np.ascontiguousarray(full_lens, np.int32)),
              ("calib_offset", np.ascontiguousarray(calib_offset, np.float32)),
              ("calib_scale", np.ascontiguousarray(calib_scale, np.float32)), ("read_ids", ids),
              ("adc", np.ascontiguousarray(adc, np.int16))]
    pos, sections = 0, []
    for name, a in arrays:
        sections.append({"name": name, "dtype": a.dtype.str, "shape": list(a.shape), "offset": pos})
        pos += (a.nbytes + 63) & ~63
    header = json.dumps({"version": 1, "sections": sections}).encode()
    base = (len(_MAGIC) + 8 + len(header) + 63) & ~63
    with open(path, "wb") as f:
        f.write(_MAGIC)
        f.write(np.uint64(len(header)).tobytes())
        f.write(header)
        f.write(b"\0" * (base - f.tell()))
        for (name, a), sec in zip(arrays, sections):
            f.seek(base + sec["offset"])
            a.tofile(f)
        f.truncate(base + pos)
    return path


# ---- container version 2: binary header, compressed signal (the native pipeline's input, adb_files.cuh) ----------------
_MAGIC2 = b"ADBSIG02"
_HDR2 = np.dtype([("magic", "S8"), ("version", "<u4"), ("flags", "<u4"), ("n_reads", "<u8"), ("id_width", "<u4"),
                  ("reserved0", "<u4"), ("off_comp_offsets", "<u8"), ("off_n_samples", "<u8"), ("off_full_lens", "<u8"),
                  ("off_calib_offset", "<u8"), ("off_calib_scale", "<u8"), ("off_read_ids", "<u8"), ("off_blob", "<u8"),
                  ("blob_bytes", "<u8"), ("reserved", "u1", (32,))])
assert _HDR2.itemsize == 128
F_SVB16, F_ZSTD = 1, 2


def _zstd():
    import ctypes

    z = ctypes.CDLL("libzstd.so.1")
    z.ZSTD_compressBound.restype = ctypes.c_size_t
    z.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    z.ZSTD_compress.restype = ctypes.c_size_t
    z.ZSTD_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    z.ZSTD_decompress.restype = ctypes.c_size_t
    z.ZSTD_decompress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
    z.ZSTD_isError.restype = ctypes.c_uint
    z.ZSTD_isError.argtypes = [ctypes.c_size_t]
    return z


def write_container_v2(path: str, adc: np.ndarray, offsets: np.ndarray, full_lens: np.ndarray, calib_offset: np.ndarray,
                       calib_scale: np.ndarray, read_ids: Sequence[str], compress: bool = True, zstd: bool = False,
                       preload_size: Optional[int] = None, encoded=None) -> str:
    """"ADBSIG02": 128-byte binary header + 64-byte aligned sections.  Per read the first ``preload_size`` samples (all
    by default) as an svb16 + zig-zag + delta stream (``compress``; adapted_b200.svb16), optionally wrapped in one zstd
    frame per read (``zstd``: pod5's VBZ), or raw int16.  ``encoded`` = (comp, comp_offsets, n_samples) skips the
    encoder (bench.py encodes on the GPU)."""
    from . import svb16

    if not path.endswith(".adbsig"):
        path += ".adbsig"
    offsets = np.ascontiguousarray(offsets, np.int64)
    n = offsets.size - 1
    if encoded is not None:
        blob, coffs, ns = encoded
        flags = F_SVB16
    else:
        adc = np.ascontiguousarray(adc, np.int16)
        if preload_size is not None and n and int(np.diff(offsets).max(initial=0)) > preload_size:
            keep = np.minimum(np.diff(offsets), preload_size)
            adc = np.concatenate([adc[offsets[i]: offsets[i] + keep[i]] for i in range(n)])
            offsets = np.concatenate([[0], np.cumsum(keep)]).astype(np.int64)
        if compress:
            blob, coffs, ns = svb16.encode_reads(adc, offsets)
            flags = F_SVB16
        else:
            blob = adc[offsets[0]: offsets[-1]].view(np.uint8) if n else np.zeros(0, np.uint8)
            coffs = (offsets - offsets[0]) * 2
            ns = np.diff(offsets).astype(np.int32)
            flags = 0
    if zstd:
        blob, coffs = svb16.zstd_frames(blob, coffs, 1)
        flags |= F_ZSTD
    ids = np.asarray([str(i).encode() for i in read_ids], dtype="S") if len(read_ids) else np.zeros(0, "S1")
    ids = ids.astype(f"S{ids.dtype.itemsize + 1}")  # NUL terminated
    arrays = [("off_comp_offsets", np.ascontiguousarray(coffs, np.int64)), ("off_n_samples", np.ascontiguousarray(ns, np.int32)),
              ("off_full_lens", np.ascontiguousarray(full_lens, np.int32)), ("off_calib_offset", np.ascontiguousarray(calib_offset, np.float32)),
              ("off_calib_scale", np.ascontiguousarray(calib_scale, np.float32)), ("off_read_ids", ids),
              ("off_blob", np.ascontiguousarray(blob, np.uint8))]
    hdr = np.zeros(1, _HDR2)
    hdr["magic"], hdr["version"], hdr["flags"], hdr["n_reads"], hdr["id_width"] = _MAGIC2, 2, flags, n, ids.dtype.itemsize
    pos = 128
    for name, a in arrays:
        hdr[name] = pos
        pos += (a.nbytes + 63) & ~63
    hdr["blob_bytes"] = arrays[-1][1].nbytes
    with open(path, "wb") as f:
        f.write(hdr.tobytes())
        for name, a in arrays:
            f.seek(int(hdr[name][0]))
            a.tofile(f)
        f.truncate(pos)
    return path


def read_container_v2(path: str) -> Dict[str, Any]:
    """Memory maps of an ADBSIG02 container: comp, comp_offsets, n_samples, full_lens, calib_offset, calib_scale,
    read_ids (fixed-width bytes) and flags."""
    hdr = np.fromfile(path, dtype=_HDR2, count=1)
    if hdr.size != 1 or bytes(hdr["magic"][0]) != _MAGIC2:
        raise ValueError(f"{path}: not an ADBSIG02 signal container")
    h = hdr[0]
    n, w = int(h["n_reads"]), int(h["id_width"])

    def mm(off, dtype, count):
        return np.memmap(path, dtype=dtype, mode="r", offset=int(off), shape=(count,)) if count else np.zeros(0, dtype)

    return {"flags": int(h["flags"]), "comp_offsets": mm(h["off_comp_offsets"], np.int64, n + 1), "n_samples": mm(h["off_n_samples"], np.int32, n),
            "full_lens": mm(h["off_full_lens"], np.int32, n), "calib_offset": mm(h["off_calib_offset"], np.float32, n),
            "calib_scale": mm(h["off_calib_scale"], np.float32, n), "read_ids": mm(h["off_read_ids"], f"S{w}", n),
            "comp": mm(h["off_blob"], np.uint8, int(h["blob_bytes"]))}


def detect_files_native(files: Sequence[str], out_dir: str, spc: Any, model: Any = None, read_ids_incl: Optional[Set[str]] = None,
                        minibatch_size: int = 1000, batch_size_output: int = 4000, continue_run: bool = False, device: int = 0,
                        chunk_minibatches: int = 16, write_csv: bool = True, copy_threads: int = 0, format_threads: int = 0) -> Dict[str, Any]:
    """``adapted detect`` / ``continue`` between the reader and the tables through the native overlapped pipeline
    (adb_detect_files): ADBSIG02 containers -> pinned ring -> H2D (compressed) -> device decode -> detection -> records
    -> formatter threads.  Selection (file_proc.py:150-168) and the `continue` scan (file_proc.py:97-140) are resolved
    here into per-file keep masks and first table indices; everything per read runs in the library."""
    import ctypes as C

    from . import _lib
    from .detect import flatten_cnn_weights

    flat = flatten_config(spc)
    excl = processed_read_ids(out_dir) if continue_run else set()
    incl = set(read_ids_incl) if read_ids_incl else set()
    if incl and excl:
        incl, excl = incl.difference(excl), set()
    masks = []
    if incl or excl:
        for fn in files:
            ids = read_container_v2(fn)["read_ids"]
            w = ids.dtype.itemsize
            if incl:
                keep = np.isin(ids, np.asarray(sorted(x.encode() for x in incl), dtype=f"S{w}"))
            else:
                keep = ~np.isin(ids, np.asarray(sorted(x.encode() for x in excl), dtype=f"S{w}"))
            masks.append(np.ascontiguousarray(keep, dtype=np.uint8))
    bidx = {"pass": 0, "fail": 0}
    if continue_run:
        for key, sub, prefix in (("pass", "boundaries", "detected_boundaries_"), ("fail", "failed_reads", "failed_reads_")):
            d = os.path.join(out_dir, sub)
            idx = [int(f.split("_")[-1].split(".")[0]) for f in os.listdir(d) if f.startswith(prefix) and f.endswith(".csv")] \
                if os.path.isdir(d) else []
            bidx[key] = max(idx, default=-1) + 1
    paths = (C.c_char_p * len(files))(*[os.fsencode(f) for f in files])
    keep_arr = (C.c_void_p * len(files))(*[m.ctypes.data if m.size else None for m in masks]) if masks else None
    job = _lib.AdbFileJob(paths=paths, n_paths=len(files), minibatch_size=int(minibatch_size),
                          keep=keep_arr, out_dir=os.fsencode(out_dir), batch_size_output=int(batch_size_output),
                          chunk_batches=int(chunk_minibatches), bidx_pass=bidx["pass"], bidx_fail=bidx["fail"],
                          n_copy_threads=int(copy_threads), n_format_threads=int(format_threads), write_csv=int(bool(write_csv)))
    w = flatten_cnn_weights(model) if flat["primary_method"] == 1 else None
    cfg = _lib.fill_config(flat)
    st = _lib.AdbFileStats()
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_detect_files(ctx.handle, C.byref(job), C.byref(cfg), w.ctypes.data if w is not None else None, C.byref(st)))
    if st.lost:
        logging.error("%d reads in minibatches lost like the reference's handle_completed_future (file_proc.py:726-731)", st.lost)
    return {"reads": int(st.reads), "pass": int(st.n_pass), "fail": int(st.n_fail), "lost": int(st.lost), "files": int(st.files),
            "comp_bytes": int(st.comp_bytes), "h2d_bytes": int(st.h2d_bytes), "seconds": float(st.seconds),
            "reader_busy_s": float(st.read_s), "writer_wait_gpu_s": float(st.gpu_wait_s), "writer_busy_s": float(st.write_s)}


def read_container(path: str) -> Dict[str, np.ndarray]:
    """Memory maps of the sections (read-only); ``read_ids`` comes back as a fixed-width bytes array."""
    import json

    with open(path, "rb") as f:
        if f.read(len(_MAGIC)) != _MAGIC:
            raise ValueError(f"{path}: not an adapted_b200 signal container")
        hlen = int(np.frombuffer(f.read(8), np.uint64)[0])
        header = json.loads(f.read(hlen).decode())
    base = (len(_MAGIC) + 8 + hlen + 63) & ~63
    out = {}
    for sec in header["sections"]:
        shape = tuple(sec["shape"])
        if int(np.prod(shape)) == 0:
            out[sec["name"]] = np.zeros(shape, dtype=np.dtype(sec["dtype"]))
        else:
            out[sec["name"]] = np.memmap(path, dtype=np.dtype(sec["dtype"]), mode="r", offset=base + sec["offset"], shape=shape)
    return out


def _id_str(x) -> str:
    return x.decode() if isinstance(x, (bytes, np.bytes_)) else str(x)


class ContainerSource:
    """Reads of one native container, in file order: (read_id, int16 samples, calibration offset, scale, num_samples)."""

    def __init__(self, path: str):
        self.path = path

    def reads(self, selection: Optional[Set[str]] = None):
        c = read_container(self.path)
        off = c["offsets"]
        for i in range(c["full_lens"].size):
            rid = _id_str(c["read_ids"][i])
            if selection is not None and rid not in selection:
                continue
            yield rid, c["adc"][off[i]: off[i + 1]], float(c["calib_offset"][i]), float(c["calib_scale"][i]), int(c["full_lens"][i])


class Pod5Source:
    """The same interface over a pod5 file through the ``pod5`` package (``Reader.reads(selection=..., missing_ok=True)``,
    ``ReadRecord.signal`` / ``.calibration`` / ``.num_samples`` / ``.read_id`` -- the calls of file_proc.py:164-175 with
    the raw ADC signal instead of ``signal_pa``).  ``pod5`` is not installable in the build image: this adapter is
    written against the package's documented API and is UNTESTED here (parity unpinned, DESIGN.md)."""

    def __init__(self, path: str):
        self.path = path

    def reads(self, selection: Optional[Set[str]] = None):
        import pod5  # noqa: F401 -- raises ImportError where the package is missing

        with pod5.Reader(self.path) as reader:
            it = reader.reads(selection=list(selection), missing_ok=True) if selection else reader.reads()
            for rr in it:
                cal = rr.calibration
                yield str(rr.read_id), np.asarray(rr.signal, dtype=np.int16), float(cal.offset), float(cal.scale), int(rr.num_samples)


def open_source(path: str):
    return Pod5Source(path) if path.endswith(".pod5") else ContainerSource(path)


def yield_minibatches(files: Iterable[str], read_ids_incl: Optional[Set[str]], read_ids_excl: Optional[Set[str]],
                      batch_size: int, preload_size: int) -> Iterator[Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray,
                                                                             np.ndarray, List[str]]]:
    """yield_signals_from_pod5 (file_proc.py:143-190) for the int16 ingest: minibatches of ``batch_size`` reads in file
    order, running across file boundaries, every read truncated to ``preload_size`` samples; yields
    (adc blob, offsets [n+1], full_lens, calib_offset, calib_scale, read_ids).  Selection semantics as there: with both
    sets given the exclusions are taken out of the inclusions; an inclusion set selects, an exclusion set skips."""
    incl = set(read_ids_incl) if read_ids_incl else set()
    excl = set(read_ids_excl) if read_ids_excl else set()
    if incl and excl:
        incl = incl.difference(excl)
        excl = set()
    selection = incl if incl else None
    m = int(preload_size)

    def fresh():
        return [], [0], [], [], [], []

    chunks, offs, lens, coff, cscale, ids = fresh()
    for fn in files:
        for rid, sig, c_off, c_scale, n_samples in open_source(fn).reads(selection):
            if rid in excl:
                continue
            k = min(m, int(n_samples), int(sig.size))
            chunks.append(np.asarray(sig[:k], dtype=np.int16))
            offs.append(offs[-1] + k)
            lens.append(int(n_samples))
            coff.append(c_off)
            cscale.append(c_scale)
            ids.append(rid)
            if len(ids) == batch_size:
                yield (np.concatenate(chunks) if chunks else np.zeros(0, np.int16), np.asarray(offs, np.int64),
                       np.asarray(lens, np.int32), np.asarray(coff, np.float32), np.asarray(cscale, np.float32), ids)
                chunks, offs, lens, coff, cscale, ids = fresh()
    if ids:
        yield (np.concatenate(chunks), np.asarray(offs, np.int64), np.asarray(lens, np.int32), np.asarray(coff, np.float32),
               np.asarray(cscale, np.float32), ids)


def detect_files(files: Sequence[str], out_dir: str, spc: Any, model: Any = None, read_ids_incl: Optional[Set[str]] = None,
                 minibatch_size: int = 1000, batch_size_output: int = 4000, continue_run: bool = False, device: int = 0,
                 minibatches_per_call: int = 64) -> Dict[str, int]:
    """``adapted detect`` / ``continue`` between the reader and the tables for any number of input files (containers or,
    where the package exists, pod5): minibatches run across file boundaries like the reference's producer; groups of
    ``minibatches_per_call`` go through the CUDA library in one call (pipelined H2D inside)."""
    from .detect import detect_reads

    flat = flatten_config(spc)
    if len(files) == 1 and not str(files[0]).endswith(".pod5"):
        # one container: whole groups of minibatches are sliced out of the blob, no per-read python work
        c = read_container(files[0])
        if int(np.diff(c["offsets"]).max(initial=0)) <= flat["sig_preload_size"]:
            return detect_file(files[0], out_dir, spc, model=model, minibatch_size=minibatch_size,
                               batch_size_output=batch_size_output, continue_run=continue_run, device=device,
                               reads_per_call=minibatches_per_call * minibatch_size, read_ids_incl=read_ids_incl, container=c)
    method = flat["primary_method"]
    log = "" if method == 0 else None
    excl = processed_read_ids(out_dir) if continue_run else None
    if continue_run:
        writer = BoundaryTableWriter.continue_from(out_dir, method, batch_size_output=batch_size_output, llr_detect_log=log)
    else:
        writer = BoundaryTableWriter(os.path.join(out_dir, "boundaries"), os.path.join(out_dir, "failed_reads"), method,
                                     batch_size_output=batch_size_output, llr_detect_log=log)
    stats = {"reads": 0, "pass": 0, "fail": 0, "lost": 0}

    def run(group):
        adc = np.concatenate([g[0] for g in group])
        lens_per = [g[1][-1] for g in group]
        off = np.zeros(sum(len(g[5]) for g in group) + 1, dtype=np.int64)
        pos, base = 1, 0
        for g, tot in zip(group, lens_per):
            off[pos: pos + len(g[5])] = g[1][1:] + base
            pos += len(g[5])
            base += int(tot)
        ids = [i for g in group for i in g[5]]
        recs, status, over = detect_reads(adc, off, np.concatenate([g[2] for g in group]), np.concatenate([g[3] for g in group]),
                                          np.concatenate([g[4] for g in group]), spc, model=model, minibatch_size=minibatch_size,
                                          device=device, return_records=True, return_overflow=True)
        n = len(ids)
        stats["reads"] += n
        for bi, st in enumerate(status):
            a, b = bi * minibatch_size, min((bi + 1) * minibatch_size, n)
            if st != 0:
                logging.error("minibatch of %d reads lost (status %d), like the reference's handle_completed_future", b - a, int(st))
                stats["lost"] += b - a
                continue
            writer.add(recs[a:b], ids[a:b], {i - a: v for i, v in over.items() if a <= i < b} if over else None)
            ok = int((recs[a:b]["success"] != 0).sum())
            stats["pass"] += ok
            stats["fail"] += (b - a) - ok

    with writer:
        group = []
        for mbatch in yield_minibatches(files, read_ids_incl, excl, minibatch_size, flat["sig_preload_size"]):
            group.append(mbatch)
            # only complete minibatches may be followed by another one inside a call
            if len(group) == minibatches_per_call or len(mbatch[5]) < minibatch_size:
                run(group)
                group = []
        if group:
            run(group)
    stats["files"] = len(writer.files)
    return stats


def processed_read_ids(continue_from: str, failed_only: bool = False) -> Set[str]:
    """Read ids already present in the tables of a previous run (scan_processed_reads, file_proc.py:103-130)."""
    done: Set[str] = set()
    subs = [("failed_reads", "failed_reads_")] + ([] if failed_only else [("boundaries", "detected_boundaries_")])
    for sub, prefix in subs:
        d = os.path.join(continue_from, sub)
        if not os.path.isdir(d):
            continue
        for fn in os.listdir(d):
            if fn.startswith(prefix) and fn.endswith(".csv"):
                with open(os.path.join(d, fn)) as f:
                    done.update(line.split(",")[0] for line in f.readlines()[1:])
    return done


def detect_file(path: str, out_dir: str, spc: Any, model: Any = None, minibatch_size: int = 1000,
                batch_size_output: int = 4000, continue_run: bool = False, device: int = 0,
                reads_per_call: int = 64000, read_ids_incl: Optional[Set[str]] = None,
                container: Optional[Dict[str, np.ndarray]] = None) -> Dict[str, int]:
    """Run the detection over every read of a container and write ``<out_dir>/boundaries/detected_boundaries_<i>.csv``
    and ``<out_dir>/failed_reads/failed_reads_<i>.csv``.  ``continue_run`` skips reads already in the tables of
    ``out_dir`` and continues the file numbering (``adapted continue``)."""
    from .detect import detect_reads

    c = container if container is not None else read_container(path)
    ids = np.asarray(c["read_ids"])
    keep = np.arange(ids.size)

    def as_ids(strings):
        return np.asarray(sorted(x.encode() for x in strings), dtype=ids.dtype if ids.dtype.kind == "S" else None)

    if read_ids_incl:
        keep = keep[np.isin(ids, as_ids(read_ids_incl))]
    if continue_run:
        done = processed_read_ids(out_dir)
        if done:
            keep = keep[~np.isin(ids[keep], as_ids(done))]
    flat = flatten_config(spc)
    method = flat["primary_method"]
    log = "" if method == 0 else None
    if continue_run:
        writer = BoundaryTableWriter.continue_from(out_dir, method, batch_size_output=batch_size_output, llr_detect_log=log)
    else:
        writer = BoundaryTableWriter(os.path.join(out_dir, "boundaries"), os.path.join(out_dir, "failed_reads"), method,
                                     batch_size_output=batch_size_output, llr_detect_log=log)
    offsets = c["offsets"]
    stats = {"reads": int(keep.size), "pass": 0, "fail": 0, "lost": 0}
    per_call = max(minibatch_size, reads_per_call // minibatch_size * minibatch_size)
    with writer:
        for s in range(0, keep.size, per_call):
            sel = keep[s: s + per_call]
            # compact the selected reads into one ragged batch (file order)
            lens = (offsets[sel + 1] - offsets[sel]).astype(np.int64)
            off = np.zeros(sel.size + 1, dtype=np.int64)
            np.cumsum(lens, out=off[1:])
            if sel.size and sel[-1] - sel[0] + 1 == sel.size:
                adc = c["adc"][offsets[sel[0]]: offsets[sel[-1] + 1]]
            else:
                adc = np.concatenate([c["adc"][offsets[i]: offsets[i + 1]] for i in sel]) if sel.size else np.zeros(0, np.int16)
            recs, status, over = detect_reads(adc, off, c["full_lens"][sel], c["calib_offset"][sel], c["calib_scale"][sel], spc,
                                              model=model, minibatch_size=minibatch_size, device=device, return_records=True,
                                              return_overflow=True)
            for bi, st in enumerate(status):
                a, b = bi * minibatch_size, min((bi + 1) * minibatch_size, sel.size)
                if st != 0:
                    logging.error("minibatch of %d reads lost (status %d), like the reference's handle_completed_future",
                                  b - a, int(st))
                    stats["lost"] += b - a
                    continue
                r = recs[a:b]
                writer.add(r, [_id_str(x) for x in ids[sel[a:b]]],
                           {i - a: v for i, v in over.items() if a <= i < b} if over else None)
                n_ok = int((r["success"] != 0).sum())
                stats["pass"] += n_ok
                stats["fail"] += (b - a) - n_ok
    stats["files"] = len(writer.files)
    return stats
