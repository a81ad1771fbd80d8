"""CPU: host-side logic -- utterance sharding, the world_size-2 metric gather (gloo), ragged
batching and the h5 schema of the create_h5 drop-in (with an in-memory stand-in for h5py, which is
not installed in the build image)."""
import os
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from acoustic_echo_cancellation_b200 import hostutil, sharding, wav2h5


def test_shard_range_partitions_exactly():
    for n in (0, 1, 7, 1024, 100000):
        for world in (1, 2, 3, 8):
            spans = [sharding.shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        sharding.shard_range(4, 2, 2)


def _worker(rank, world, port, n_items, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lo, hi = sharding.shard_range(n_items, rank, world)
    local = torch.arange(lo, hi, dtype=torch.float32) * 0.5      # stands for per-utterance ERLE
    full = sharding.gather_metrics(local, n_items)
    full_async, work = sharding.gather_metrics(local, n_items, async_op=True)    # overlapped form used by bench.py
    if work is not None:
        work.wait()
    assert torch.equal(full, full_async)
    even, work = sharding.gather_metrics(torch.full((3,), float(rank)), 3 * world, async_op=True)   # equal shards
    if work is not None:
        work.wait()
    assert even.tolist() == [float(r) for r in range(world) for _ in range(3)]
    files = sharding.merge_filelists([f"tr_{i}.ex" for i in range(lo, hi)])
    ret[rank] = (full.tolist(), files)
    dist.destroy_process_group()


def test_gather_metrics_world_size_2_gloo():
    n_items, world = 7, 2
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 29500 + os.getpid() % 2000
    mp.spawn(_worker, args=(world, port, n_items, ret), nprocs=world, join=True)
    for r in range(world):
        full, files = ret[r]
        assert full == [0.5 * i for i in range(n_items)]
        assert files == [f"tr_{i}.ex" for i in range(n_items)]


def test_gather_metrics_single_process_passthrough():
    x = torch.arange(5, dtype=torch.float32)
    assert torch.equal(sharding.gather_metrics(x, 5), x)
    y, work = sharding.gather_metrics(x, 5, async_op=True)
    assert work is None and torch.equal(y, x)


def test_ragged_batching_pads_and_unpads():
    far = [np.arange(5, dtype=np.float32), np.arange(3, dtype=np.float32)]
    mic = [np.ones(5, dtype=np.float32), np.ones(3, dtype=np.float32)]
    seen = {}

    def runner(fa, mi, n):
        seen["shape"], seen["n"] = fa.shape, n.tolist()
        assert (fa[1, 3:] == 0).all()
        return fa + 1, mi * 2

    errs, echos = wav2h5._stage1_batch(far, mic, runner)
    assert seen == {"shape": (2, 5), "n": [5, 3]}
    assert [len(e) for e in errs] == [5, 3] and np.array_equal(errs[1], far[1] + 1)
    assert np.array_equal(echos[0], 2 * mic[0])


class _FakeGroup(dict):
    def create_dataset(self, name, data=None, shape=None, chunks=None):
        assert shape == data.shape and data.dtype == np.float32
        assert chunks is True or data.size == 0            # h5py rejects chunks=True for an empty dataset
        self[name] = np.array(data)

    def create_group(self, name):
        g = _FakeGroup()
        self[name] = g
        return g


class _FakeH5:
    def __init__(self):
        self.files = {}

    def File(self, name, mode):
        assert mode == "w"
        f = _FakeGroup()
        f.close = lambda: None
        self.files[name] = f
        return f


def _write_wavs(folder, ids, n=2000, sr=16000, subdirs=False, dtype=np.int16):
    from scipy.io import wavfile

    rng = np.random.default_rng(0)
    data = {}
    for i in ids:
        for k, pat in wav2h5.WAV_PATTERNS.items():
            if dtype == np.int16:
                x = (rng.standard_normal(n + 10 * int(i)) * 3000).astype(np.int16)
            else:
                x = (rng.standard_normal(n + 10 * int(i)) * 0.1).astype(np.float32)
            d = os.path.join(folder, k) if subdirs else folder
            os.makedirs(d, exist_ok=True)
            wavfile.write(os.path.join(d, pat.format(idx=i)), sr, x)
            data[(i, k)] = x
    return data


def _fake_runner(fa, mi, n):          # stand-in for the CUDA runner: like the C ABI it takes float32 or 16-bit PCM
    if fa.dtype == np.int16:          # (the test wavs are 16-bit, so this is the branch create_h5 takes)
        fa, mi = fa.astype(np.float32) / np.float32(32768), mi.astype(np.float32) / np.float32(32768)
    return fa * np.float32(0.5), mi * np.float32(0.25)


def test_create_h5_three_forms_schema(tmp_path):
    """a6: the train / test / val generators (train_wav2h5.py, test_wav2h5.py, val_wav2h5.py) -- file names, keys,
    list files, stage-1 datasets inside the groups -- and the one `create_h5` name that dispatches to them."""
    wav_dir, val_dir, h5_dir, list_dir = tmp_path / "wav", tmp_path / "val", tmp_path / "h5", tmp_path / "lists"
    for d in (wav_dir, val_dir, h5_dir, list_dir):
        d.mkdir()
    ids = ["3", "11", "7", "20", "5"]
    data = _write_wavs(str(wav_dir), ids)
    fake = _FakeH5()
    args = types.SimpleNamespace(train_path=str(wav_dir), h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    st = {}
    paths = wav2h5.create_h5(args, runner=_fake_runner, batch=2, h5=fake, stats=st)       # -> train form
    assert sorted(os.path.basename(p) for p in paths) == sorted(f"tr_{i}.ex" for i in ids)
    assert open(list_dir / "tr_list.txt").read().split("\n") == paths
    assert st["utterances"] == 5 and st["pcm16_batches"] == 3 and st["float32_batches"] == 0
    for p in paths:
        f = fake.files[p]
        idx = os.path.basename(p)[3:-3]
        assert set(f) == {"nearend_speech", "nearend_mic", "farend_speech", "echo", "stage1_error", "stage1_echo"}
        for k in wav2h5.KEYS:                                   # exactly what librosa.load gives for a 16-bit wav
            assert np.array_equal(f[k], data[(idx, k)].astype(np.float32) / np.float32(32768))
        assert f["stage1_error"].shape == f["farend_speech"].shape
        assert np.array_equal(f["stage1_error"], np.float32(0.5) * f["farend_speech"])
        assert np.array_equal(f["stage1_echo"], np.float32(0.25) * f["nearend_mic"])
    # test form
    fake = _FakeH5()
    args = types.SimpleNamespace(val_path=str(wav_dir), h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    path = wav2h5.create_h5(args, runner=_fake_runner, batch=2, h5=fake)                 # -> test form (flat folder)
    assert os.path.basename(path) == "test.ex"
    root = fake.files[path]
    assert sorted(root, key=int) == ["0", "1", "2", "3", "4"]     # ONLY numbered groups at the root (test.py:23)
    names = open(list_dir / "filename.txt").read().split("\n")
    assert sorted(names) == sorted(ids)
    for g, idx in zip(sorted(root, key=int), names):              # group order == filename.txt order
        assert set(root[g]) == set(wav2h5.KEYS) | {"stage1_error", "stage1_echo"}
        assert np.array_equal(root[g]["echo"], data[(idx, "echo")].astype(np.float32) / np.float32(32768))
    assert open(list_dir / "tt_list.txt").read() == path
    # val form: sub-directory per signal, keys mic/ref/near/echo, tt/test2.ex, tt_list2.txt, basenames in filename.txt
    vdata = _write_wavs(str(val_dir), ["4", "9", "1"], subdirs=True)
    fake = _FakeH5()
    args = types.SimpleNamespace(val_path=str(val_dir), h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    path = wav2h5.create_h5(args, runner=_fake_runner, batch=2, h5=fake)                 # -> val form
    assert os.path.basename(path) == "test2.ex" and open(list_dir / "tt_list2.txt").read() == path
    root = fake.files[path]
    names = open(list_dir / "filename.txt").read().split("\n")
    assert sorted(names) == sorted(f"nearend_mic_fileid_{i}.wav" for i in ("4", "9", "1"))
    assert sorted(root, key=int) == ["0", "1", "2"]
    for g, base in zip(sorted(root, key=int), names):
        idx = base.split("_")[-1].split(".wav")[0]
        assert set(root[g]) == {"mic", "ref", "near", "echo", "stage1_error", "stage1_echo"}
        for out_key, src in wav2h5.VAL_KEYS.items():
            assert np.array_equal(root[g][out_key], vdata[(idx, src)].astype(np.float32) / np.float32(32768))
        assert np.array_equal(root[g]["stage1_error"], np.float32(0.5) * root[g]["ref"])


def test_create_h5_float_wavs_take_the_float32_path_and_npz_store_round_trips(tmp_path):
    wav_dir, h5_dir, list_dir = tmp_path / "wav", tmp_path / "h5", tmp_path / "lists"
    for d in (wav_dir, h5_dir, list_dir):
        d.mkdir()
    data = _write_wavs(str(wav_dir), ["1", "2"], dtype=np.float32)       # IEEE-float wavs: not the PCM16 fast path
    args = types.SimpleNamespace(train_path=str(wav_dir), h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    st = {}
    paths = wav2h5.create_h5_train(args, runner=_fake_runner, batch=4, h5=wav2h5.NpzStore(), stats=st)
    assert st["float32_batches"] == 1 and st["pcm16_batches"] == 0
    for p in paths:
        idx = os.path.basename(p)[3:-3]
        with np.load(p) as z:
            assert set(z.files) == set(wav2h5.KEYS) | {"stage1_error", "stage1_echo"}
            assert np.array_equal(z["farend_speech"], data[(idx, "farend_speech")])
            assert np.array_equal(z["stage1_error"], np.float32(0.5) * z["farend_speech"])
    args.val_path, args.train_path = args.train_path, None
    path = wav2h5.create_h5(args, runner=_fake_runner, batch=1, h5=wav2h5.RawStore())     # test form, raw container
    z = wav2h5.RawStore.load(path)
    names = open(list_dir / "filename.txt").read().split("\n")
    assert sorted(z) == sorted(f"{g}/{k}" for g in range(2) for k in wav2h5.KEYS + ("stage1_error", "stage1_echo"))
    for g, idx in enumerate(names):
        assert np.array_equal(z[f"{g}/echo"], data[(idx, "echo")])
        assert np.array_equal(z[f"{g}/stage1_echo"], np.float32(0.25) * z[f"{g}/nearend_mic"])


def test_wav_probe_and_pcm16_fast_read(tmp_path):
    from scipy.io import wavfile

    from acoustic_echo_cancellation_b200 import ingest

    x = (np.random.default_rng(1).standard_normal(1234) * 5000).astype(np.int16)
    p = str(tmp_path / "a.wav")
    wavfile.write(p, 16000, x)
    info = ingest.probe_wav(p)
    assert (info.rate, info.channels, info.bits, info.fmt, info.frames) == (16000, 1, 16, 1, 1234)
    assert info.fast(16000) and not info.fast(8000)
    row = np.full(2000, 7, dtype=np.int16)
    assert ingest.read_pcm16_into(p, info, row) == 1234
    assert np.array_equal(row[:1234], x) and (row[1234:] == 0).all()
    assert np.array_equal(ingest.pcm16_to_float32(x), ingest.load_wav(p, 16000))     # == librosa's x / 32768
    wavfile.write(p, 16000, np.stack([x, x], axis=1))
    assert not ingest.probe_wav(p).fast(16000)                   # stereo -> general loader
    with open(str(tmp_path / "bad.wav"), "wb") as f:
        f.write(b"not a wav file at all")
    with pytest.raises(ValueError):
        ingest.probe_wav(str(tmp_path / "bad.wav"))
    # ragged microphone: shorter than the far end is zero-padded, longer is cut on upload but stored in full
    far, mic_short, mic_long = str(tmp_path / "f.wav"), str(tmp_path / "ms.wav"), str(tmp_path / "ml.wav")
    wavfile.write(far, 16000, x)
    wavfile.write(mic_short, 16000, x[:1000])
    wavfile.write(mic_long, 16000, np.concatenate([x, x[:50]]))
    dec = ingest.BatchDecoder(16000, threads=2)
    b = dec.decode([far, far], [mic_short, mic_long], {"echo": [far, far]})
    assert b.pcm16 and b.n.tolist() == [1234, 1234] and b.far.shape == (2, 1234)
    assert np.array_equal(b.mic[0, :1000], x[:1000]) and (b.mic[0, 1000:] == 0).all()
    assert np.array_equal(b.mic[1], x)
    assert len(b.signals["__mic__"][0]) == 1000 and len(b.signals["__mic__"][1]) == 1284
    dec.close()
    # the native reader of libaec_b200.so (C++ threads) and the Python reader give the same batch
    assert dec.native, "libaec_b200.so must be built for the CPU suite (make -C .../csrc)"
    py = ingest.BatchDecoder(16000, threads=2, native=False)
    c = py.decode([far, far], [mic_short, mic_long], {"echo": [far, far]})
    assert c.pcm16 and np.array_equal(c.far, b.far) and np.array_equal(c.mic, b.mic) and np.array_equal(c.n, b.n)
    for key in ("__far__", "__mic__", "echo"):
        assert all(np.array_equal(x, y) for x, y in zip(b.signals[key], c.signals[key])), key
    py.close()
    infos = ingest.probe_batch([far, mic_short], 2)
    assert [(i.rate, i.channels, i.bits, i.fmt, i.frames) for i in infos] == [(16000, 1, 16, 1, 1234), (16000, 1, 16, 1, 1000)]
    assert ingest.probe_batch([far], 1)[0] == ingest.probe_wav(far)
    with pytest.raises(ValueError):
        ingest.probe_batch([str(tmp_path / "bad.wav")], 1)
    with pytest.raises(IOError):
        ingest.probe_batch([str(tmp_path / "missing.wav")], 1)
    dst = np.full((1, 1500), 9, dtype=np.int16)
    wavfile.write(p, 8000, x)                                    # wrong rate -> not the fast path
    assert ingest.read_pcm16_batch([p], dst, 16000, 1) is None


def test_wav_probe_handles_extra_chunks_and_extensible_headers(tmp_path):
    """RIFF files in the wild: a LIST chunk (odd size -> pad byte) before `data`, WAVE_FORMAT_EXTENSIBLE with the PCM
    sub-format, a data chunk size of 0xFFFFFFFF (streamed) -- Python and native probes must agree and read the samples"""
    import struct

    from acoustic_echo_cancellation_b200 import ingest

    x = (np.random.default_rng(2).standard_normal(777) * 4000).astype(np.int16)
    body = x.tobytes()
    fmt_ext = struct.pack("<HHIIHHHHIH14s", 0xFFFE, 1, 16000, 32000, 2, 16, 22, 16, 4, 1,
                          bytes.fromhex("000000001000800000aa00389b71"))
    lst = b"LIST" + struct.pack("<I", 7) + b"INFOabc" + b"\0"                # odd-sized chunk + pad byte
    p1 = str(tmp_path / "ext.wav")
    with open(p1, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", 4 + 8 + len(fmt_ext) + len(lst) + 8 + len(body)) + b"WAVE")
        f.write(b"fmt " + struct.pack("<I", len(fmt_ext)) + fmt_ext + lst)
        f.write(b"data" + struct.pack("<I", 0xFFFFFFFF) + body)
    for info in (ingest.probe_wav(p1), ingest.probe_batch([p1], 1)[0]):
        assert (info.rate, info.channels, info.bits, info.fmt, info.frames) == (16000, 1, 16, 1, 777)
        assert info.fast(16000)
    dst = np.zeros((1, 800), dtype=np.int16)
    fr = ingest.read_pcm16_batch([p1], dst, 16000, 2)
    assert fr.tolist() == [777] and np.array_equal(dst[0, :777], x) and (dst[0, 777:] == 0).all()
    row = np.zeros(800, dtype=np.int16)
    ingest.read_pcm16_into(p1, ingest.probe_wav(p1), row)
    assert np.array_equal(row, dst[0])
    # truncated on purpose: shorter row than the file -> the first row_samples samples, true length still reported
    short = np.zeros((1, 100), dtype=np.int16)
    assert ingest.read_pcm16_batch([p1], short, 16000, 1).tolist() == [777] and np.array_equal(short[0], x[:100])


def _shard_worker(rank, world, port, folder, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ids = wav2h5.list_utterance_ids(folder)
    if rank == 1:
        ids = ids[::-1]                       # ranks may see the directory in different orders
    mine, r = wav2h5._shard(ids)
    ret[rank] = list(mine)
    dist.destroy_process_group()


def _gen_worker(rank, world, port, wav_dir, h5_dir, list_dir, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    args = types.SimpleNamespace(train_path=wav_dir, h5_path=h5_dir, list_path=list_dir, sr=16000)
    st = {}
    merged = wav2h5.create_h5(args, runner=_fake_runner, batch=2, h5=wav2h5.RawStore(), stats=st)
    ret[rank] = (merged, st["utterances"])
    dist.destroy_process_group()


def test_two_rank_generation_writes_every_utterance_once(tmp_path):
    """config 5 shape on two ranks (gloo): each rank converts its shard of the sorted id list, the union is the corpus,
    rank 0 writes the merged tr_list.txt, every listed file exists and holds its own utterance"""
    wav_dir, h5_dir, list_dir = tmp_path / "wav", tmp_path / "h5", tmp_path / "lists"
    for d in (wav_dir, h5_dir, list_dir):
        d.mkdir()
    ids = [str(i) for i in (5, 17, 2, 40, 8, 23, 11)]
    data = _write_wavs(str(wav_dir), ids, n=700)
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 33500 + os.getpid() % 2000
    mp.spawn(_gen_worker, args=(2, port, str(wav_dir), str(h5_dir), str(list_dir), ret), nprocs=2, join=True)
    merged0, n0 = ret[0]
    merged1, n1 = ret[1]
    assert merged0 == merged1 and n0 + n1 == len(ids) and abs(n0 - n1) <= 1
    assert [os.path.basename(p) for p in merged0] == [f"tr_{i}.ex" for i in sorted(ids, key=int)]
    assert open(list_dir / "tr_list.txt").read().split("\n") == merged0
    for p in merged0:
        idx = os.path.basename(p)[3:-3]
        z = wav2h5.RawStore.load(p)
        assert np.array_equal(z["echo"], data[(idx, "echo")].astype(np.float32) / np.float32(32768))
        assert np.array_equal(z["stage1_error"], np.float32(0.5) * z["farend_speech"])


def test_two_rank_shards_are_disjoint_and_complete(tmp_path):
    ids = [str(i) for i in (12, 3, 100, 7, 45, 9, 1)]
    _write_wavs(str(tmp_path), ids, n=64)
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 31500 + os.getpid() % 2000
    mp.spawn(_shard_worker, args=(2, port, str(tmp_path), ret), nprocs=2, join=True)
    a, b = ret[0], ret[1]
    assert not (set(a) & set(b)) and sorted(a + b, key=int) == sorted(ids, key=int)
    assert abs(len(a) - len(b)) <= 1
    assert a + b == sorted(ids, key=int)      # numeric order of the ids: contiguous shards of one sorted list


def test_cli_flags_match_the_reference():
    a = wav2h5.build_parser("train").parse_args([])
    assert (a.train_path, a.h5_path, a.list_path, a.sr) == (
        "/data/lihaoming/datasets/synthetic/train_set", "/data/lihaoming/datasets/synthetic/h5",
        "../examples/filelists", 16000)
    b = wav2h5.build_parser("test").parse_args(["--val_path", "x", "--sr", "8000"])
    assert b.val_path == "x" and b.sr == 8000
    c = wav2h5.build_parser("val").parse_args([])              # val_wav2h5.py:66-84
    assert (c.val_path, c.h5_path, c.sr) == ("/data/lihaoming/gen_data/data/test_sets",
                                             "/data/lihaoming/gen_data/data/h5", 16000)


def test_cpulist_parser_and_bind_is_harmless_without_gpu():
    assert hostutil._parse_cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11]
    assert hostutil._parse_cpulist("") == []
    if not torch.cuda.is_available():
        assert hostutil.gpu_local_cpus(0) is None and hostutil.bind_to_gpu_numa(0) is None


def test_stage1_batch_sends_exact_pcm16_as_int16_and_everything_else_as_float32():
    rng = np.random.default_rng(0)
    pcm = [rng.integers(-32768, 32768, size=n, dtype=np.int16) for n in (700, 512)]
    far = [p.astype(np.float32) / 32768.0 for p in pcm]            # what librosa.load returns for a 16-bit wav
    mic = [np.roll(f, 3) for f in far]
    seen = {}

    def runner(fa, mi, n):
        seen["dtype"], seen["far"], seen["n"] = fa.dtype, fa.copy(), n.copy()
        z = np.zeros(fa.shape, dtype=np.float32)
        return z, z

    errs, _ = wav2h5._stage1_batch(far, mic, runner)
    assert seen["dtype"] == np.int16 and [len(e) for e in errs] == [700, 512]
    assert np.array_equal(seen["far"][0, :700], pcm[0]) and np.array_equal(seen["far"][1, :512], pcm[1])
    assert (seen["far"][1, 512:] == 0).all()
    far[1] = far[1] + np.float32(1e-6)                             # not representable as PCM16 any more
    wav2h5._stage1_batch(far, mic, runner)
    assert seen["dtype"] == np.float32
    assert wav2h5.as_pcm16(np.array([1.0], dtype=np.float32)) is None          # +1.0 would be 32768: out of range
    assert wav2h5.as_pcm16(np.array([-1.0, 0.5], dtype=np.float32)).tolist() == [-32768, 16384]


def test_row_stride_helper_copies_overlapping_rows_only():
    """the [B, L] row handling of ConvSTFT, batch_shift and the stage-1 entries: the kernels read row b at
    b * row_stride, so rows that overlap or are broadcast (row stride < L) must become a copy, while disjoint
    unit-stride rows (a column slice of a wider tensor) go through as they are, with their own stride"""
    from acoustic_echo_cancellation_b200.stage1 import _disjoint_rows, _shared_rows

    sig = torch.arange(20000, dtype=torch.float32)
    chunks = sig.unfold(0, 4096, 1000)                     # chunks of a long recording: rows 1000 apart, 4096 long
    assert chunks.stride() == (1000, 1)
    x, s = _disjoint_rows(chunks)
    assert s == 4096 and x.stride() == (4096, 1) and x.data_ptr() != chunks.data_ptr() and torch.equal(x, chunks)
    rep = sig[:513].expand(5, 513)                         # one signal broadcast to five rows
    assert rep.stride() == (0, 1)
    x, s = _disjoint_rows(rep)
    assert s == 513 and x.stride() == (513, 1) and torch.equal(x, rep)
    wide = torch.arange(4 * 700, dtype=torch.float32).reshape(4, 700)
    cols = wide[:, 3:515]                                  # disjoint rows 700 apart: no copy
    x, s = _disjoint_rows(cols)
    assert x is cols and s == 700
    for one in (wide[1:2, 3:515], chunks[2:3], rep[:1]):  # one row: its stride is never used, no copy
        x, s = _disjoint_rows(one)
        assert x is one and s == one.shape[1]
    for strided in (wide[:, ::2], wide[:1, ::2]):         # non-unit inner stride: copy
        x, s = _disjoint_rows(strided)
        assert x.is_contiguous() and s == 350 and torch.equal(x, strided)
    assert _disjoint_rows(torch.zeros(6, 1))[1] == 1
    # the stage-1 entries take one stride for both signals: kept when they agree, contiguous copies when not
    far, mic, s = _shared_rows(cols, wide[:, 100:612])
    assert far is cols and s == 700 and mic.data_ptr() == wide[:, 100:612].data_ptr()
    far, mic, s = _shared_rows(cols, torch.zeros(4, 512))
    assert s == 512 and far.is_contiguous() and torch.equal(far, cols) and mic.is_contiguous()
    far, mic, s = _shared_rows(chunks[:4, :512], cols)
    assert s == 512 and far.is_contiguous() and mic.is_contiguous() and torch.equal(far, chunks[:4, :512])
