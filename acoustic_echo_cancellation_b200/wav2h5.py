"""Drop-in for the reference's wav -> h5 generators with the stage-1 canceller inserted.

    create_h5(args)        <-> ``create_h5(args)`` of all three scripts (dispatches on the arguments like the
                               scripts' own ``main()`` do)
    create_h5_train(args)  <-> Stage2_lhm/generate_h5files/train_wav2h5.py:10-52
    create_h5_test(args)   <-> Stage2_lhm/generate_h5files/test_wav2h5.py:10-64
    create_h5_val(args)    <-> Stage2_lhm/generate_h5files/val_wav2h5.py:10-59

Same argparse flags (``--train_path``/``--val_path``, ``--h5_path``, ``--list_path``, ``--sr``), same file
names (``tr/tr_<idx>.ex``, ``tt/test.ex``, ``tt/test2.ex``, ``tr_list.txt``, ``tt_list.txt``, ``tt_list2.txt``,
``filename.txt``) and the same dataset keys (``nearend_speech``/``nearend_mic``/``farend_speech``/``echo``;
``mic``/``ref``/``near``/``echo`` for the val form), so the reference readers (Stage2_lhm/scripts/train1.py:33-40,
scripts/test.py:20-33, scripts/utils/data_utils.py:31-34) keep working; two datasets are ADDED beside them:
``stage1_error`` and ``stage1_echo``.  In ``test.ex`` / ``test2.ex`` they go INSIDE each numbered group because
``ValidateDataset`` counts root members (scripts/test.py:23).  With far-end alignment on (``--stage1_align_max_delay``,
``Stage1Runner(align=...)``) stage 1 runs on the far end delayed by its estimated bulk delay, and a third dataset,
``stage1_far_shift`` (float32, one element: that delay in samples), goes beside them; ``farend_speech`` stays as
recorded.

How a run is organised (the reference is one serial loop: decode 4 wavs, write, next utterance):

    decode batch k+1  (thread pool, 16-bit PCM read straight into page-locked int16 batch buffers: ingest.py)
    stage 1 on batch k (``aec_stage1_run_host[_pcm16]``: H2D / kernel / D2H pipelined in slices; one C call,
                        GIL released)
    write batch k-1    (thread pool; one file per utterance for the train form, one ordered writer for test / val)

all three overlapped, three buffer sets cycling.  With ``torch.distributed`` initialised each rank converts a
contiguous shard of the SORTED id list on its own GPU (LOCAL_RANK) and rank 0 writes the merged list.

The ``.ex`` files are HDF5.  ``h5py`` is used when it is installed (the reference's own writer); it is absent from the
build image, and then ``h5lite`` -- this package's own writer of the HDF5 subset those files need (superblock v0,
symbol-table groups, contiguous float32 datasets; h5lite.py) -- writes them, so the generators produce files the
reference's readers open either way.  ``h5=`` selects a container explicitly: ``h5lite``, the ``h5py`` module, or the
two non-HDF5 stand-ins kept for measurements (``NpzStore``: one uncompressed ``.npz`` per file; ``RawStore``: raw
bytes + JSON index), whose files are NOT readable by the reference's readers.
"""
from __future__ import annotations

import argparse
import glob
import os
import time
from concurrent.futures import ThreadPoolExecutor
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from . import ingest
from .ingest import load_wav  # noqa: F401  (re-exported: the reference-shaped single-file loader)

KEYS = ("nearend_speech", "nearend_mic", "farend_speech", "echo")
WAV_PATTERNS = {
    "nearend_speech": "nearend_speech_fileid_{idx}.wav",
    "nearend_mic": "nearend_mic_fileid_{idx}.wav",
    "farend_speech": "farend_speech_fileid_{idx}.wav",
    "echo": "echo_fileid_{idx}.wav",
}
# val_wav2h5.py:11-14,33-36,43-46: sub-directory per signal, older key names
VAL_KEYS = {"mic": "nearend_mic", "ref": "farend_speech", "near": "nearend_speech", "echo": "echo"}


def list_utterance_ids(folder: str, pattern: str = "nearend_speech_fileid_*.wav") -> List[str]:
    """ids in the order ``glob`` yields them (train_wav2h5.py:13-17)."""
    ids = []
    for p in glob.glob(os.path.join(folder, pattern)):
        ids.append(os.path.basename(p).split(".wav")[0].split("_")[-1])
    return ids


def as_pcm16(x: np.ndarray) -> Optional[np.ndarray]:
    """The int16 samples ``x`` was decoded from, if ``x`` is exactly ``pcm / 32768`` (what ``librosa.load`` /
    ``wavfile.read`` give for a 16-bit PCM wav at its native rate, train_wav2h5.py:20-23), else None.  Lossless by
    construction: the check is ``x * 32768`` being integers inside the int16 range."""
    q = np.asarray(x, dtype=np.float32) * np.float32(32768.0)
    if q.size and (np.any(q != np.rint(q)) or q.max() > 32767.0 or q.min() < -32768.0):
        return None
    return q.astype(np.int16)


def _stage1_batch(far: List[np.ndarray], mic: List[np.ndarray], runner: Callable):
    """Zero-pad a ragged list to [B, Lmax] (like collate_fn, train1.py:52-61), run, un-pad.

    When every far-end and microphone signal of the batch is exact 16-bit PCM (the usual case: the corpus is wav files)
    the batch goes to the runner as int16, which the host-buffer C ABI uploads as such and converts on the GPU
    (``aec_stage1_run_host_pcm16``): half the host-to-device bytes of a PCIe-bound pipeline, bit-identical results."""
    n = np.array([len(x) for x in far], dtype=np.int64)
    lmax = int(n.max())
    pcm = [(as_pcm16(f), as_pcm16(m[:len(f)])) for f, m in zip(far, mic)]
    use_pcm = all(a is not None and b is not None for a, b in pcm)
    dt = np.int16 if use_pcm else np.float32
    fa = np.zeros((len(far), lmax), dtype=dt)
    mi = np.zeros((len(far), lmax), dtype=dt)
    for i, (f, m) in enumerate(zip(far, mic)):
        fa[i, :len(f)] = pcm[i][0] if use_pcm else f
        mm = pcm[i][1] if use_pcm else m[:len(f)]
        mi[i, :len(mm)] = mm
    err, echo = runner(fa, mi, n)
    return [err[i, :n[i]] for i in range(len(far))], [echo[i, :n[i]] for i in range(len(far))]


def _local_device() -> int:
    """CUDA device of this rank: LOCAL_RANK under torchrun, else the current device."""
    if "LOCAL_RANK" in os.environ:
        return int(os.environ["LOCAL_RANK"])
    try:
        import torch

        return int(torch.cuda.current_device()) if torch.cuda.is_available() else 0
    except Exception:
        return 0


class Stage1Runner:
    """``runner(far, mic, n) -> (err, echo)`` backed by ``aec_stage1_run_host`` / ``_pcm16`` (no CPU fallback).
    With ``align`` (a ``DelayConfig``) the far end is aligned to the microphone first (``aec_stage1_run_host_ex``) and
    the runner returns ``(err, echo, shift)``, ``shift`` int32 [B] the samples each far end was delayed by.

    Inputs that are not page-locked (arrays a caller got from ``librosa.load`` and stacked with numpy) are staged
    through page-locked buffers first: a ``cudaMemcpyAsync`` from pageable memory is staged by the driver and
    serialises the slices of the pipeline.  Outputs are page-locked buffers owned by the runner, valid until the
    call after next (two sets alternate), which is what lets a writer thread drain batch k while batch k+1 runs."""

    def __init__(self, cfg=None, slice_utterances: int = 128, device: Optional[int] = None, want_echo: bool = True,
                 align=None):
        from .stage1 import Stage1Config

        self.cfg = cfg or Stage1Config()
        self.align = align
        self.slice_utterances = int(slice_utterances)
        self.device = _local_device() if device is None else int(device)
        self.want_echo = want_echo
        self.pipe = None
        self._in: Dict[str, np.ndarray] = {}
        self._out: List[Dict[str, np.ndarray]] = [{}, {}]
        self._flip = 0
        self.seconds = 0.0          # time spent inside the C call (for the pipeline report)

    def _pinned(self, store: dict, key: str, shape, dtype) -> np.ndarray:
        from .stage1 import pinned_empty

        buf = store.get(key)
        if buf is None or buf.dtype != np.dtype(dtype) or buf.shape[0] < shape[0] or buf.shape[1] < shape[1]:
            rows = max(shape[0], buf.shape[0] if buf is not None and buf.dtype == np.dtype(dtype) else 0)
            cols = max(shape[1], buf.shape[1] if buf is not None and buf.dtype == np.dtype(dtype) else 0)
            import torch

            with torch.cuda.device(self.device):
                buf = pinned_empty((rows, cols), dtype)
            store[key] = buf
        return buf[:shape[0], :shape[1]]

    def __call__(self, far: np.ndarray, mic: np.ndarray, n: np.ndarray):
        from .stage1 import HostPipeline, is_pinned

        if self.pipe is None or self.pipe.max_samples < far.shape[1]:
            if self.pipe is not None:
                self.pipe.close()
            self.pipe = HostPipeline(self.slice_utterances, far.shape[1], self.device)
        if not (is_pinned(far) and is_pinned(mic)):
            sf = self._pinned(self._in, "far", far.shape, far.dtype)
            sm = self._pinned(self._in, "mic", mic.shape, mic.dtype)
            np.copyto(sf, far)
            np.copyto(sm, mic)
            far, mic = sf, sm
        out = self._out[self._flip]
        self._flip ^= 1
        err = self._pinned(out, "err", far.shape, np.float32)
        echo = self._pinned(out, "echo", far.shape, np.float32) if self.want_echo else None
        shift = np.zeros(far.shape[0], dtype=np.int32) if self.align is not None else None
        t0 = time.perf_counter()
        self.pipe.run(far, mic, self.cfg, n_samples=n, err=err, echo=echo, align=self.align, shift=shift)
        self.seconds += time.perf_counter() - t0
        return (err, echo) if shift is None else (err, echo, shift)

    def buffers_pinned(self) -> bool:
        """True when every staging / output buffer this runner has allocated is page-locked (tested on the GPU)."""
        from .stage1 import is_pinned

        bufs = list(self._in.values()) + [b for o in self._out for b in o.values()]
        return bool(bufs) and all(is_pinned(b) for b in bufs)

    def close(self):
        if self.pipe is not None:
            self.pipe.close()
            self.pipe = None


def default_runner(cfg=None, slice_utterances: int = 128, device: Optional[int] = None, align=None) -> Callable:
    """Runner backed by ``aec_stage1_run_host`` on this rank's GPU (LOCAL_RANK under torchrun)."""
    return Stage1Runner(cfg, slice_utterances, device, align=align)


def _h5py():
    """the module whose ``File(name, 'w')`` writes the ``.ex`` files: h5py when installed, else this package's own
    HDF5 writer (same call surface, same names / shapes / types / values on disk, contiguous storage)"""
    try:
        import h5py  # type: ignore
        return h5py
    except ImportError:  # pragma: no cover - depends on the box
        from . import h5lite
        return h5lite


class _NpzGroup:
    def __init__(self, root: "_NpzFile", prefix: str):
        self._root, self._prefix = root, prefix

    def create_dataset(self, name, data=None, shape=None, chunks=None):
        self._root._members[self._prefix + name] = np.ascontiguousarray(data)

    def create_group(self, name):
        return _NpzGroup(self._root, self._prefix + str(name) + "/")


class _NpzFile(_NpzGroup):
    def __init__(self, path: str):
        super().__init__(self, "")
        self._path, self._members = path, {}

    def close(self):
        with open(self._path, "wb") as f:          # exact file name (np.savez would append ".npz" to a str path)
            np.savez(f, **self._members)
        self._members = {}


class _RawGroup:
    def __init__(self, root: "_RawFile", prefix: str):
        self._root, self._prefix = root, prefix

    def create_dataset(self, name, data=None, shape=None, chunks=None):
        a = np.ascontiguousarray(data)
        f = self._root._f
        self._root._index.append((self._prefix + name, a.dtype.str, list(a.shape), f.tell()))
        f.write(memoryview(a).cast("B"))                  # (the write releases the GIL)

    def create_group(self, name):
        return _RawGroup(self._root, self._prefix + str(name) + "/")


class _RawFile(_RawGroup):
    def __init__(self, path: str):
        super().__init__(self, "")
        self._f = open(path, "wb", buffering=0)
        self._f.write(b"AECRAW01" + b"\0" * 8)            # magic + offset of the index (patched on close)
        self._index = []

    def close(self):
        import json

        pos = self._f.tell()
        self._f.write(json.dumps(self._index).encode())
        self._f.seek(8)
        self._f.write(int(pos).to_bytes(8, "little"))
        self._f.close()


class RawStore:
    """Second stand-in container for boxes without h5py, built for speed: the datasets' bytes one after the other
    plus a JSON index at the end (``RawStore.load(path)`` reads it back).  What the file-pipeline measurement
    (tools/config5_files.py) writes; like ``NpzStore`` it is NOT readable by the reference's readers."""

    def File(self, name, mode):
        assert mode == "w"
        return _RawFile(name)

    @staticmethod
    def load(path: str) -> Dict[str, np.ndarray]:
        import json

        with open(path, "rb") as f:
            blob = f.read()
        assert blob[:8] == b"AECRAW01"
        pos = int.from_bytes(blob[8:16], "little")
        out = {}
        for name, dt, shape, off in json.loads(blob[pos:].decode()):
            n = int(np.prod(shape)) if shape else 1
            out[name] = np.frombuffer(blob, dtype=np.dtype(dt), count=n, offset=off).reshape(shape)
        return out


class NpzStore:
    """Stand-in container with the slice of the ``h5py`` surface the generators use, for boxes without h5py:
    one uncompressed npz (zip of .npy) per ``File``, member names ``<group>/<dataset>``."""

    def File(self, name, mode):
        assert mode == "w"
        return _NpzFile(name)


def _dist():
    try:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            return dist
    except Exception:
        pass
    return None


def _shard(ids: List[str]):
    """This rank's contiguous shard of the SORTED id list (glob order is filesystem-dependent: ranks on different
    nodes could otherwise see different orders and drop / duplicate utterances).  A single process keeps the glob
    order, like the reference."""
    from .sharding import shard_range

    dist = _dist()
    if dist is not None and dist.get_world_size() > 1:
        ordered = sorted(ids, key=lambda s: (len(s), s))
        lo, hi = shard_range(len(ordered), dist.get_rank(), dist.get_world_size())
        return ordered[lo:hi], dist.get_rank()
    return ids, 0


def _create_dataset(g, name: str, a: np.ndarray, shape=None):
    """``create_dataset(name, data=a.astype(float32), shape=a.shape, chunks=True)`` as the reference writes it;
    h5py rejects ``chunks=True`` for an empty dataset (an utterance shorter than one hop has an empty stage-1
    output), so those are written contiguous."""
    a = ingest.as_float32(a)
    shape = a.shape if shape is None else shape
    if a.size == 0 or int(np.prod(shape)) == 0:
        g.create_dataset(name, data=a, shape=shape)
    else:
        g.create_dataset(name, data=a, shape=shape, chunks=True)


class _Engine:
    """decode | stage 1 | write, overlapped.  ``emit(k, ids, batch, errs, echos)`` writes one finished batch."""

    def __init__(self, sr: int, runner: Optional[Callable], batch: int, decode_threads: int, pinned: bool):
        alloc = None
        if pinned:
            from .stage1 import pinned_empty

            alloc = lambda shape, dtype: pinned_empty(shape, dtype)      # noqa: E731
        self.runner = runner or default_runner()
        self.decoder = ingest.BatchDecoder(sr, threads=decode_threads, alloc=alloc, sets=3)
        self.batch = int(batch)
        self.stats = {"decode_s": 0.0, "stage1_s": 0.0, "write_s": 0.0, "wall_s": 0.0, "utterances": 0,
                      "pcm16_batches": 0, "float32_batches": 0}

    def _decode(self, paths):
        t0 = time.perf_counter()
        b = self.decoder.decode(paths["far"], paths["mic"], paths["extra"])
        self.stats["decode_s"] += time.perf_counter() - t0
        return b

    def _run(self, b: ingest.DecodedBatch):
        t0 = time.perf_counter()
        res = self.runner(b.far, b.mic, b.n)
        err, echo = res[0], res[1]
        self.stats["stage1_s"] += time.perf_counter() - t0
        self.stats["pcm16_batches" if b.pcm16 else "float32_batches"] += 1
        nb = len(b.n)
        # a runner that aligns the far end returns its per-utterance shift third
        shifts = [np.array([res[2][i]], dtype=np.float32) for i in range(nb)] if len(res) > 2 else None
        return [err[i, :b.n[i]] for i in range(nb)], [echo[i, :b.n[i]] for i in range(nb)], shifts

    def run(self, ids: Sequence[str], paths_of: Callable[[Sequence[str]], dict], emit: Callable):
        t_start = time.perf_counter()
        chunks = [list(ids[i:i + self.batch]) for i in range(0, len(ids), self.batch)]
        with ThreadPoolExecutor(1, thread_name_prefix="aec-decode") as dec, \
                ThreadPoolExecutor(1, thread_name_prefix="aec-gpu") as gpu, \
                ThreadPoolExecutor(1, thread_name_prefix="aec-write") as wr:

            def timed_emit(*a):
                t0 = time.perf_counter()
                emit(*a)
                self.stats["write_s"] += time.perf_counter() - t0

            writes = []
            fut_dec = dec.submit(self._decode, paths_of(chunks[0])) if chunks else None
            for k, chunk in enumerate(chunks):
                b = fut_dec.result()
                # batch k-2 must be on disk before its buffers are reused: the decoder cycles three buffer sets
                # (batch k+1 decodes into the set of batch k-2) and the runner's output sets alternate (batch k
                # writes where batch k-2 did)
                if k >= 2:
                    writes[k - 2].result()
                if k + 1 < len(chunks):
                    fut_dec = dec.submit(self._decode, paths_of(chunks[k + 1]))
                errs, echos, shifts = gpu.submit(self._run, b).result()
                writes.append(wr.submit(timed_emit, k, chunk, b, errs, echos, shifts))
                self.stats["utterances"] += len(chunk)
            for w in writes:
                w.result()
        self.decoder.close()
        self.stats["wall_s"] = time.perf_counter() - t_start
        return self.stats


def _train_paths(folder: str):
    def paths_of(chunk):
        p = lambda k: [os.path.join(folder, WAV_PATTERNS[k].format(idx=i)) for i in chunk]      # noqa: E731
        return {"far": p("farend_speech"), "mic": p("nearend_mic"),
                "extra": {"nearend_speech": p("nearend_speech"), "echo": p("echo")}}
    return paths_of


def _signal(b: ingest.DecodedBatch, key: str, j: int) -> np.ndarray:
    return b.signals[{"farend_speech": "__far__", "nearend_mic": "__mic__"}.get(key, key)][j]


def write_ex_batch(paths: Sequence[str], names: Sequence[str], rows: Sequence[Sequence[np.ndarray]], threads: int = 8):
    """``rows[f][d]`` (1-D float32, or int16 PCM stored as float32 = s / 32768) -> dataset ``names[d]`` of the HDF5 file
    ``paths[f]``; the native batched form of the reference's per-utterance writer block (train_wav2h5.py:35-44),
    ``aec_ex_write_batch``."""
    import ctypes as C

    from . import _lib

    lib = _lib.load()
    nf, nd = len(paths), len(names)
    keep = []                                       # arrays that had to be made contiguous / converted stay alive
    ptrs = (C.c_void_p * (nf * nd))()
    lens = np.zeros(nf * nd, dtype=np.int64)
    fmts = np.zeros(nd, dtype=np.int32)
    for d in range(nd):
        if nf and all(rows[f][d].dtype == np.int16 for f in range(nf)):
            fmts[d] = 1
    for f in range(nf):
        for d in range(nd):
            a = rows[f][d]
            want = np.int16 if fmts[d] == 1 else np.float32
            if a.dtype != want:
                a = ingest.as_float32(a)
            if a.ndim != 1 or not a.flags.c_contiguous:
                a = np.ascontiguousarray(a).reshape(-1)
            keep.append(a)
            ptrs[f * nd + d] = a.ctypes.data
            lens[f * nd + d] = a.shape[0]
    cpaths = (C.c_char_p * nf)(*[os.fsencode(p) for p in paths])
    cnames = (C.c_char_p * nd)(*[n.encode() for n in names])
    _lib.check(lib.aec_ex_write_batch(cpaths, nf, nd, cnames, ptrs, lens.ctypes.data, fmts.ctypes.data, int(threads)),
               "aec_ex_write_batch")


def create_h5_train(args, runner: Optional[Callable] = None, batch: int = 256, h5=None, decode_threads: int = 8,
                    write_threads: int = 8, pinned: Optional[bool] = None, stats: Optional[dict] = None,
                    native_writer: bool = True):
    """``create_h5(args)`` of train_wav2h5.py with stage 1 inserted.  One ``tr_<idx>.ex`` per utterance.  With the
    package's own HDF5 container (``h5lite``: the default where h5py is not installed) the files of a batch are
    written by one native call (``aec_ex_write_batch``); ``native_writer=False`` keeps the per-file Python writer."""
    h5 = h5 or _h5py()
    ids, rank = _shard(list_utterance_ids(args.train_path))
    os.makedirs(os.path.join(args.h5_path, "tr"), exist_ok=True)
    train_list = [str(os.path.join(args.h5_path, "tr", "tr_" + idx + ".ex")) for idx in ids]
    eng = _Engine(args.sr, runner, batch, decode_threads, pinned=(runner is None) if pinned is None else pinned)
    pool = ThreadPoolExecutor(max(1, write_threads), thread_name_prefix="aec-h5")

    def write_one(name, b, j, err, echo, shift):
        w = h5.File(name, "w")
        for k in KEYS:                                                   # train_wav2h5.py:39-42
            _create_dataset(w, k, _signal(b, k, j))
        _create_dataset(w, "stage1_error", err)
        _create_dataset(w, "stage1_echo", echo)
        if shift is not None:
            _create_dataset(w, "stage1_far_shift", shift)
        w.close()

    def emit(k, chunk, b, errs, echos, shifts):
        futs = [pool.submit(write_one, os.path.join(args.h5_path, "tr", "tr_" + idx + ".ex"), b, j, errs[j], echos[j],
                            shifts[j] if shifts is not None else None)
                for j, idx in enumerate(chunk)]
        for f in futs:
            f.result()

    def emit_native(k, chunk, b, errs, echos, shifts):
        # the whole batch in ONE C call (aec_ex_write_batch: C++ threads, int16 -> float32 on the way out, no
        # interpreter between the files); same bytes as write_one through h5lite
        names = KEYS + ("stage1_error", "stage1_echo") + (("stage1_far_shift",) if shifts is not None else ())
        rows = [[_signal(b, key, j) for key in KEYS] + [errs[j], echos[j]] + ([shifts[j]] if shifts is not None else [])
                for j in range(len(chunk))]
        write_ex_batch([os.path.join(args.h5_path, "tr", "tr_" + idx + ".ex") for idx in chunk], names, rows,
                       threads=max(1, write_threads))

    from . import h5lite

    if h5 is h5lite and native_writer:
        emit = emit_native                                               # noqa: F811
    st = eng.run(ids, _train_paths(args.train_path), emit)
    pool.shutdown()
    if stats is not None:
        stats.update(st)
    from .sharding import merge_filelists

    merged = merge_filelists(train_list)
    if rank == 0:
        with open(os.path.join(args.list_path, "tr_list.txt"), "w") as f:     # train_wav2h5.py:48-51
            f.write("\n".join(merged))
    return merged


def _single_file(args, ids, paths_of, keymap, h5, runner, batch, filename, list_name, names, decode_threads, pinned,
                 stats, echo_shape_of_near: bool):
    """Shared body of the test / val forms: ONE file, one numbered group per utterance, written in order by one
    writer (call it on one rank)."""
    h5 = h5 or _h5py()
    os.makedirs(os.path.join(args.h5_path, "tt"), exist_ok=True)
    path = os.path.join(args.h5_path, "tt", filename)
    w = h5.File(path, "w")
    count = [0]
    eng = _Engine(args.sr, runner, batch, decode_threads, pinned=(runner is None) if pinned is None else pinned)

    def emit(k, chunk, b, errs, echos, shifts):
        for j in range(len(chunk)):
            g = w.create_group(str(count[0]))                                # test_wav2h5.py:44, val_wav2h5.py:42
            for out_key, src_key in keymap.items():
                a = _signal(b, src_key, j)
                shape = None
                if echo_shape_of_near and out_key == "echo":                 # val_wav2h5.py:46: shape=near.shape
                    shape = _signal(b, "nearend_speech", j).shape
                    a = ingest.as_float32(a)
                    if a.shape != shape:                                     # h5py would broadcast-or-raise; keep the data
                        shape = a.shape
                _create_dataset(g, out_key, a, shape)
            _create_dataset(g, "stage1_error", errs[j])
            _create_dataset(g, "stage1_echo", echos[j])
            if shifts is not None:
                _create_dataset(g, "stage1_far_shift", shifts[j])
            count[0] += 1

    st = eng.run(ids, paths_of, emit)
    w.close()
    if stats is not None:
        stats.update(st)
    with open(os.path.join(args.list_path, list_name), "w") as f:             # test_wav2h5.py:55-58
        f.write(str(path))
    with open(os.path.join(args.list_path, "filename.txt"), "w") as f:        # test_wav2h5.py:60-62
        f.write("\n".join(names))
    return path


def create_h5_test(args, runner: Optional[Callable] = None, batch: int = 256, h5=None, filename: str = "test.ex",
                   decode_threads: int = 8, pinned: Optional[bool] = None, stats: Optional[dict] = None):
    """``create_h5(args)`` of test_wav2h5.py with stage 1 inserted: ``tt/test.ex``, groups "0", "1", ... with the
    four reference datasets + the two stage-1 ones; ``tt_list.txt``; ``filename.txt`` holds the ids."""
    ids = list_utterance_ids(args.val_path)
    return _single_file(args, ids, _train_paths(args.val_path), {k: k for k in KEYS}, h5, runner, batch, filename,
                        "tt_list.txt", ids, decode_threads, pinned, stats, echo_shape_of_near=False)


def create_h5_val(args, runner: Optional[Callable] = None, batch: int = 256, h5=None, filename: str = "test2.ex",
                  decode_threads: int = 8, pinned: Optional[bool] = None, stats: Optional[dict] = None):
    """``create_h5(args)`` of val_wav2h5.py with stage 1 inserted: one sub-directory per signal under
    ``--val_path`` (``farend_speech/``, ``nearend_speech/``, ``nearend_mic/``, ``echo/``), utterances enumerated
    from ``nearend_mic/*.wav`` (val_wav2h5.py:24), keys ``mic`` / ``ref`` / ``near`` / ``echo`` (:43-46),
    ``tt/test2.ex``, ``tt_list2.txt``; ``filename.txt`` holds the microphone BASENAMES (:28)."""
    mic_dir = os.path.join(args.val_path, "nearend_mic")
    names, ids = [], []
    for p in glob.glob(os.path.join(mic_dir, "*.wav")):
        base = os.path.basename(p)
        names.append(base)
        ids.append(base.split("_")[-1].split(".wav")[0])                      # val_wav2h5.py:27-30
    name_of = dict(zip(ids, names))

    def paths_of(chunk):
        sub = lambda d, k: [os.path.join(args.val_path, d, WAV_PATTERNS[k].format(idx=i)) for i in chunk]   # noqa: E731
        return {"far": sub("farend_speech", "farend_speech"),
                "mic": [os.path.join(mic_dir, name_of[i]) for i in chunk],
                "extra": {"nearend_speech": sub("nearend_speech", "nearend_speech"), "echo": sub("echo", "echo")}}

    return _single_file(args, ids, paths_of, dict(VAL_KEYS), h5, runner, batch, filename, "tt_list2.txt", names,
                        decode_threads, pinned, stats, echo_shape_of_near=True)


def create_h5(args, **kw):
    """The one name all three reference scripts export.  ``args.train_path`` -> the train form; ``args.val_path``
    -> the val form when it holds the per-signal sub-directories of val_wav2h5.py:11-14, else the test form."""
    if getattr(args, "train_path", None):
        return create_h5_train(args, **kw)
    if getattr(args, "val_path", None):
        if os.path.isdir(os.path.join(args.val_path, "nearend_mic")):
            return create_h5_val(args, **kw)
        return create_h5_test(args, **kw)
    raise ValueError("args needs train_path (train_wav2h5.py) or val_path (test_wav2h5.py / val_wav2h5.py)")


def build_parser(kind: str) -> argparse.ArgumentParser:
    """The reference's flags and defaults (train_wav2h5.py:55-73, test_wav2h5.py:67-86, val_wav2h5.py:62-86)."""
    p = argparse.ArgumentParser(description=f"wav -> h5 ({kind}) with the stage-1 echo canceller",
                                formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    if kind == "train":
        p.add_argument("--train_path", type=str, default="/data/lihaoming/datasets/synthetic/train_set")
        p.add_argument("--h5_path", type=str, default="/data/lihaoming/datasets/synthetic/h5")
    elif kind == "val":
        p.add_argument("--val_path", type=str, default="/data/lihaoming/gen_data/data/test_sets")
        p.add_argument("--h5_path", type=str, default="/data/lihaoming/gen_data/data/h5")
    else:
        p.add_argument("--val_path", type=str, default="/data/lihaoming/datasets/synthetic/test_set")
        p.add_argument("--h5_path", type=str, default="/data/lihaoming/datasets/synthetic/h5")
    p.add_argument("--list_path", type=str, default="../examples/filelists")
    p.add_argument("--sr", type=int, default=16000)
    # not in the reference (which has no stage 1): which filter produces stage1_error / stage1_echo
    p.add_argument("--stage1_algo", choices=sorted(STAGE1_ALGOS), default="nlms",
                   help="nlms / kalman: STFT-domain recurrence; ols-nlms / ols-kalman: overlap-save PBFDAF (frame 512, 1-16 partitions)")
    p.add_argument("--stage1_partitions", type=int, default=4)
    p.add_argument("--stage1_align_max_delay", type=int, default=0,
                   help="0: off; else the largest far-end delay (samples, a power of two in 256..8192) searched per "
                        "utterance -- stage 1 then runs on the far end delayed by the estimate, and each utterance "
                        "gets a stage1_far_shift dataset (samples)")
    # not in the reference (which always writes through h5py): who writes the .ex (HDF5) files
    p.add_argument("--ex_writer", choices=["auto", "h5py", "native"], default="auto",
                   help="auto: h5py when installed (chunked storage, as the reference writes), else the package's own HDF5 "
                        "writer; native: the package's writer even when h5py is there (contiguous storage, batched C++ "
                        "writer for the per-utterance training files)")
    return p


def container_from_args(args):
    """the module whose ``File`` writes the .ex files, per ``--ex_writer`` (None -> the default of ``_h5py()``)"""
    which = getattr(args, "ex_writer", "auto")
    if which == "native":
        from . import h5lite
        return h5lite
    if which == "h5py":
        import h5py  # type: ignore
        return h5py
    return None


STAGE1_ALGOS = {"nlms": 0, "kalman": 1, "ols-nlms": 2, "ols-kalman": 3}


def runner_from_args(args) -> Optional[Callable]:
    """the stage-1 runner the command-line flags ask for; None (-> library default) when they are absent"""
    if not hasattr(args, "stage1_algo"):
        return None
    from .stage1 import DelayConfig, Stage1Config

    n = int(getattr(args, "stage1_align_max_delay", 0) or 0)
    return default_runner(Stage1Config(algo=STAGE1_ALGOS[args.stage1_algo], partitions=int(args.stage1_partitions)),
                          align=DelayConfig(max_delay=n) if n > 0 else None)


def main(kind: str = "train", argv=None):
    args = build_parser(kind).parse_args(argv)
    os.makedirs(args.h5_path, exist_ok=True)
    return {"train": create_h5_train, "test": create_h5_test, "val": create_h5_val}[kind](
        args, runner=runner_from_args(args), h5=container_from_args(args))
