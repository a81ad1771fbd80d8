"""h5lite: the package's own writer / reader of the HDF5 subset the reference's ``.ex`` files need (h5py and libhdf5 are
not in the image).  The reader is pinned on a file libhdf5 itself produced; the writer is checked by that reader, by an
independent structural walk of the bytes (B-tree key invariants, sorted symbol tables, sibling links, alignment, end-of-
file address), through the three ``create_h5`` generators, and -- where AEC_REFERENCE_DIR names a checkout of the
reference -- by the reference's own ``TrainDataset`` / ``ValidateDataset`` with h5lite standing in for h5py."""
import os
import struct
import subprocess
import sys
import types

import numpy as np
import pytest

from acoustic_echo_cancellation_b200 import h5lite, wav2h5
from test_host_logic import _fake_runner, _write_wavs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _libhdf5_sample():
    # a copy of scipy's test file scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat (BSD-3-Clause), written by libhdf5
    return os.path.join(ROOT, "tests", "golden", "testhdf5_7.4_GLNX86.mat")


def test_reader_on_a_file_written_by_libhdf5():
    """MATLAB 7.3 file = HDF5 behind a 512-byte user block: superblock v0 at 512, base address 512, one dataset
    `testdouble` = linspace(0, 2 pi, 9) as a (9, 1) float64 array (what scipy's own tests expect of it), object header with
    seven messages incl. attribute / modification time / NIL padding, version-2 layout message"""
    with h5lite.File(_libhdf5_sample(), "r") as f:
        assert list(f) == ["testdouble"] and len(f) == 1 and "testdouble" in f and "nope" not in f
        d = f["testdouble"]
        assert d.shape == (9, 1) and d.dtype == np.float64
        assert np.array_equal(d[:].ravel(), np.linspace(0, 2 * np.pi, 9))
        assert np.array_equal(np.array(f["/testdouble"]), d[...])
        with pytest.raises(KeyError):
            f["missing"]


# ---- an independent walk of the bytes: nothing below uses h5lite's reader -------------------------------------------
def _walk_group(b, btree, heap, sizes):
    """returns [(name, object header address, cache type, scratch)] in B-tree order and checks the group invariants"""
    assert b[heap:heap + 4] == b"HEAP" and b[heap + 4] == 0
    dsize, free, daddr = struct.unpack_from("<QQQ", b, heap + 8)
    assert free == 1 and dsize % 8 == 0 and daddr % 8 == 0 and daddr + dsize <= len(b)
    hd = b[daddr:daddr + dsize]
    assert hd[:8] == b"\0" * 8                                  # offset 0: the empty name of key 0

    def name(off):
        return hd[off:hd.index(b"\0", off)]

    out = []

    def node(addr, lo_name, level_expected=None):
        """names in this subtree lie in (lo_name, returned hi_name]"""
        assert addr % 8 == 0
        if b[addr:addr + 4] == b"SNOD":
            ver, _, n = struct.unpack_from("<BBH", b, addr + 4)
            assert ver == 1 and 1 <= n <= 8 and addr + sizes["snod"] <= len(b)
            prev = lo_name
            for i in range(n):
                off, oh, cache, _r = struct.unpack_from("<QQII", b, addr + 8 + 40 * i)
                nm = name(off)
                assert nm > prev, "symbol-table entries must be strictly ascending in strcmp order"
                prev = nm
                out.append((nm.decode(), oh, cache, b[addr + 32 + 40 * i:addr + 48 + 40 * i]))
            assert b[addr + 8 + 40 * n:addr + sizes["snod"]] == b"\0" * (sizes["snod"] - 8 - 40 * n)
            return prev, None
        assert b[addr:addr + 4] == b"TREE"
        ntype, level, used = struct.unpack_from("<BBH", b, addr + 4)
        left, right = struct.unpack_from("<QQ", b, addr + 8)
        assert ntype == 0 and used <= 32 and addr + sizes["tree"] <= len(b)
        if level_expected is not None:
            assert level == level_expected
        key = name(struct.unpack_from("<Q", b, addr + 24)[0])
        assert key == lo_name
        o = addr + 32
        for _ in range(used):
            child, koff = struct.unpack_from("<QQ", b, o)
            hi, _ = node(child, key, level - 1 if level else None)
            assert hi == name(koff), "key i+1 is the largest name of child i"
            key = hi
            o += 16
        return key, (left, right, level)

    node(btree, b"")
    return out


def _walk_file(path):
    b = open(path, "rb").read()
    assert b[:8] == h5lite.SIGNATURE and b[8:16] == bytes([0, 0, 0, 0, 0, 8, 8, 0])
    lk, ik, flags = struct.unpack_from("<HHI", b, 16)
    base, free, eof, drv = struct.unpack_from("<QQQQ", b, 24)
    assert (lk, ik, flags, base, free, drv) == (4, 16, 0, 0, h5lite.UNDEF, h5lite.UNDEF) and eof == len(b)
    name_off, oh, cache, _r, bt, hp = struct.unpack_from("<QQIIQQ", b, 56)
    assert name_off == 0 and cache == 1
    sizes = {"snod": 8 + 2 * lk * 40, "tree": 24 + (2 * ik + 1) * 8 + 2 * ik * 8}
    found = {}

    def header(addr):
        assert addr % 8 == 0
        ver, _, n, ref, size = struct.unpack_from("<BBHII", b, addr)
        assert ver == 1 and ref == 1 and size % 8 == 0 and addr + 16 + size <= len(b)
        msgs, pos = [], addr + 16
        while pos < addr + 16 + size:
            t, s, fl = struct.unpack_from("<HHB", b, pos)
            assert s % 8 == 0
            msgs.append((t, b[pos + 8:pos + 8 + s]))
            pos += 8 + s
        assert len(msgs) == n and pos == addr + 16 + size
        return msgs

    def group(oh, bt, hp, prefix):
        (mt, md), = header(oh)
        assert mt == 0x11 and struct.unpack("<QQ", md) == (bt, hp)           # cached scratch == the header's message
        for nm, coh, cache, scratch in _walk_group(b, bt, hp, sizes):
            msgs = dict(header(coh))
            if cache == 1:
                cbt, chp = struct.unpack("<QQ", scratch)
                group(coh, cbt, chp, prefix + nm + "/")
                continue
            assert set(msgs) == {0x1, 0x3, 0x5, 0x8}
            sp, ty, fill, lay = msgs[0x1], msgs[0x3], msgs[0x5], msgs[0x8]
            rank = sp[1]
            assert sp[0] == 1 and sp[2] == 0
            shape = struct.unpack_from(f"<{rank}Q", sp, 8)
            assert fill[:8] == bytes([2, 1, 2, 1, 0, 0, 0, 0])
            assert lay[0] == 3 and lay[1] == 1
            addr, nbytes = struct.unpack_from("<QQ", lay, 2)
            size = struct.unpack_from("<I", ty, 4)[0]
            assert nbytes == int(np.prod(shape)) * size
            if nbytes:
                assert addr % 8 == 0 and 96 <= addr and addr + nbytes <= len(b)
            else:
                assert addr == h5lite.UNDEF
            if ty[0] == 0x11 and size == 4:
                assert ty[:4] == bytes([0x11, 0x20, 31, 0]) and ty[8:20] == struct.pack("<HHBBBBI", 0, 32, 23, 8, 0, 23, 127)
                dt = np.float32
            elif ty[0] == 0x11:
                assert ty[:4] == bytes([0x11, 0x20, 63, 0]) and ty[8:20] == struct.pack("<HHBBBBI", 0, 64, 52, 11, 0, 52, 1023)
                dt = np.float64
            else:
                assert ty[0] == 0x10 and ty[8:12] == struct.pack("<HH", 0, 8 * size)
                dt = np.dtype(("i" if ty[1] & 8 else "u") + str(size))
            found[prefix + nm] = (np.frombuffer(b, dtype=dt, count=nbytes // size, offset=addr if nbytes else 0)
                                  .reshape(shape))

    group(oh, bt, hp, "")
    return found


@pytest.mark.parametrize("n_groups", [0, 1, 8, 9, 300])
def test_writer_structures_and_round_trip(tmp_path, n_groups):
    """8 entries = one full symbol-table node, 9 = two, 300 = 38 nodes under a two-level B-tree"""
    rng = np.random.default_rng(n_groups)
    path = str(tmp_path / "t.ex")
    ref = {}
    with h5lite.File(path, "w") as w:
        for i in range(n_groups):
            g = w.create_group(str(i))
            for k in wav2h5.KEYS + ("stage1_error", "stage1_echo"):
                a = rng.standard_normal(50 + i).astype(np.float32)
                g.create_dataset(k, data=a, shape=a.shape, chunks=True)
                ref[f"{i}/{k}"] = a
        ref["pcm"] = np.arange(-3, 4, dtype=np.int16)
        ref["empty"] = np.zeros(0, np.float32)
        ref["matrix"] = np.arange(12, dtype=np.float64).reshape(3, 4)
        ref["u8"] = np.arange(5, dtype=np.uint8)
        for k in ("pcm", "empty", "matrix", "u8"):
            w.create_dataset(k, data=ref[k])
        with pytest.raises(ValueError):
            w.create_dataset("pcm", data=ref["pcm"])                        # h5py: name already exists
        with pytest.raises(ValueError):
            w.create_dataset("bad", data=np.zeros(4, np.float32), shape=(5,))
        with pytest.raises(TypeError):
            w.create_dataset("cplx", data=np.zeros(2, np.complex64))
        assert len(w) == n_groups + 4 and "pcm" in w and w["pcm"].shape == (7,)
    assert h5lite.is_hdf5(path)
    found = _walk_file(path)                                                # independent of h5lite's reader
    assert set(found) == set(ref)
    for k, a in ref.items():
        assert found[k].dtype == a.dtype and np.array_equal(found[k], a), k
    with h5lite.File(path, "r") as r:                                       # and through the reader
        assert len(r) == n_groups + 4
        assert sorted(r) == sorted([str(i) for i in range(n_groups)] + ["pcm", "empty", "matrix", "u8"])
        for k, a in ref.items():
            d = r[k]
            assert d.shape == a.shape and d.dtype == a.dtype and np.array_equal(d[:], a)
        if n_groups:
            assert set(r["0"].keys()) == set(wav2h5.KEYS) | {"stage1_error", "stage1_echo"}
            assert len(r["0"]["echo"]) == 50 and np.array_equal(np.array(r["0"]["echo"]), ref["0/echo"])


def test_three_level_group_btree(tmp_path):
    """more than 8 * 32 * 32 = 8192 names need a third B-tree level (a test set of that size in one test.ex)"""
    path = str(tmp_path / "big.ex")
    with h5lite.File(path, "w") as w:
        for i in range(8300):
            w.create_dataset(f"d{i}", data=np.full(1, i, np.int32))
    found = _walk_file(path)
    assert len(found) == 8300 and all(int(found[f"d{i}"][0]) == i for i in range(0, 8300, 97))
    with h5lite.File(path, "r") as r:
        assert len(r) == 8300 and int(r["d8299"][0]) == 8299


def test_unfinished_and_foreign_files_are_rejected(tmp_path):
    p = tmp_path / "x.ex"
    w = h5lite.File(str(p), "w")
    w.create_dataset("a", data=np.ones(3, np.float32))
    w._fh.close()                                                           # never closed properly: no superblock
    w._closed = True
    with pytest.raises(OSError):
        h5lite.File(str(p), "r")
    with pytest.raises(ValueError):
        h5lite.File(str(p), "a")


def _make_sets(tmp_path):
    wav_dir, val_dir, h5_dir, list_dir = tmp_path / "wav", tmp_path / "val", tmp_path / "h5", tmp_path / "lists"
    for d in (wav_dir, val_dir, h5_dir, list_dir):
        d.mkdir()
    ids = [str(i) for i in range(11)]
    data = _write_wavs(str(wav_dir), ids)
    vdata = _write_wavs(str(val_dir), ids[:3], subdirs=True)
    return wav_dir, val_dir, h5_dir, list_dir, ids, data, vdata


def test_create_h5_writes_real_hdf5_without_h5py(tmp_path):
    """a6 / f1 with the DEFAULT container of a box without h5py: every .ex file the three generators write is an HDF5
    file with the reference's names, float32 datasets and the stage-1 datasets inside the groups"""
    pytest.importorskip("scipy")
    try:
        import h5py  # noqa: F401
        pytest.skip("h5py is installed: the generators use it")
    except ImportError:
        pass
    wav_dir, val_dir, h5_dir, list_dir, ids, data, vdata = _make_sets(tmp_path)
    f32 = lambda x: x.astype(np.float32) / np.float32(32768)            # noqa: E731
    args = types.SimpleNamespace(train_path=str(wav_dir), h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    paths = wav2h5.create_h5(args, runner=_fake_runner, batch=4)
    assert len(paths) == len(ids) == len(open(list_dir / "tr_list.txt").read().split())
    for p in paths:
        idx = os.path.basename(p)[3:-3]
        z = _walk_file(p)
        assert set(z) == set(wav2h5.KEYS) | {"stage1_error", "stage1_echo"}
        for k in wav2h5.KEYS:
            assert z[k].dtype == np.float32 and np.array_equal(z[k], f32(data[(idx, k)]))
        assert np.array_equal(z["stage1_error"], np.float32(0.5) * z["farend_speech"])
    targs = types.SimpleNamespace(val_path=str(wav_dir), train_path=None, h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    tpath = wav2h5.create_h5(targs, runner=_fake_runner, batch=4)
    names = open(list_dir / "filename.txt").read().split("\n")
    with h5lite.File(tpath, "r") as r:
        assert len(r) == len(ids)                                            # ValidateDataset counts root members
        for g, idx in enumerate(names):
            assert set(r[str(g)]) == set(wav2h5.KEYS) | {"stage1_error", "stage1_echo"}
            assert np.array_equal(r[str(g)]["nearend_mic"][:], f32(data[(idx, "nearend_mic")]))
    vargs = types.SimpleNamespace(val_path=str(val_dir), h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    vpath = wav2h5.create_h5_val(vargs, runner=_fake_runner, batch=2)
    z = _walk_file(vpath)
    assert sorted(z) == sorted(f"{g}/{k}" for g in range(3) for k in list(wav2h5.VAL_KEYS) + ["stage1_error", "stage1_echo"])


# a checkout of SZU-Speech/Acoustic-Echo-Cancellation; its sources are not part of this repository
REFERENCE_SCRIPTS = os.path.join(os.environ.get("AEC_REFERENCE_DIR", ""), "Stage2_lhm", "scripts")


@pytest.mark.skipif(not os.environ.get("AEC_REFERENCE_DIR") or not os.path.isdir(REFERENCE_SCRIPTS),
                    reason="needs the reference's sources: set AEC_REFERENCE_DIR to a checkout of it")
def test_reference_readers_open_the_generated_files(tmp_path):
    """a7 with the reference's OWN code: TrainDataset (train1.py:29-42) and ValidateDataset (test.py:19-33), imported
    unmodified in a subprocess with h5lite standing in for the absent h5py, read the files create_h5 wrote"""
    wav_dir, val_dir, h5_dir, list_dir, ids, data, vdata = _make_sets(tmp_path)
    args = types.SimpleNamespace(train_path=str(wav_dir), h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    wav2h5.create_h5(args, runner=_fake_runner, batch=4, h5=h5lite)
    targs = types.SimpleNamespace(val_path=str(wav_dir), train_path=None, h5_path=str(h5_dir), list_path=str(list_dir), sr=16000)
    tpath = wav2h5.create_h5(targs, runner=_fake_runner, batch=4, h5=h5lite)
    out = str(tmp_path / "read.npz")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "golden", "run_reference_readers.py"), ROOT,
                        REFERENCE_SCRIPTS, str(list_dir / "tr_list.txt"), tpath, out],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    z = np.load(out)
    f32 = lambda x: x.astype(np.float32) / np.float32(32768)            # noqa: E731
    tr_paths = [ln.strip() for ln in open(list_dir / "tr_list.txt") if ln.strip()]
    assert int(z["train_len"]) == len(ids) and int(z["val_len"]) == len(ids)
    for i, p in enumerate(tr_paths):
        idx = os.path.basename(p)[3:-3]
        for k in wav2h5.KEYS:
            assert np.array_equal(z[f"train/{i}/{k}"], f32(data[(idx, k)]))
    names = open(list_dir / "filename.txt").read().split("\n")
    for g, idx in enumerate(names):
        for k in wav2h5.KEYS:
            assert np.array_equal(z[f"val/{g}/{k}"], f32(data[(idx, k)]))
        assert int(z[f"val/{g}/n_samples"]) == len(data[(idx, "nearend_speech")])


def test_native_batch_writer_is_byte_identical_to_h5lite(tmp_path):
    """aec_ex_write_batch (C++ threads, csrc/aec_exio.cu) and the Python writer are two implementations of the same
    layout: same bytes for float32 and 16-bit PCM sources, odd lengths (alignment padding), empty datasets, names in
    any creation order; bad arguments are refused, an unwritable path is an I/O error"""
    from acoustic_echo_cancellation_b200 import _lib, ingest

    rng = np.random.default_rng(5)
    names = ("nearend_speech", "nearend_mic", "farend_speech", "echo", "stage1_error", "stage1_echo")
    lens = [160000, 1001, 1, 0, 255, 4097, 7]
    rows, paths = [], []
    for f, n in enumerate(lens):
        row = [(rng.standard_normal(n) * 3000).astype(np.int16) for _ in range(4)]
        row += [rng.standard_normal(max(n - 3, 0)).astype(np.float32), rng.standard_normal(n).astype(np.float32)]
        rows.append(row)
        paths.append(str(tmp_path / f"native_{f}.ex"))
    wav2h5.write_ex_batch(paths, names, rows, threads=3)
    for f, p in enumerate(paths):
        q = str(tmp_path / f"python_{f}.ex")
        with h5lite.File(q, "w") as w:
            for k, a in zip(names, rows[f]):
                a = ingest.as_float32(a)
                w.create_dataset(k, data=a, shape=a.shape, chunks=True)
        assert open(p, "rb").read() == open(q, "rb").read(), f
        found = _walk_file(p)
        assert set(found) == set(names)
        assert np.array_equal(found["echo"], rows[f][3].astype(np.float32) / np.float32(32768))
    # float32-only rows, two datasets, reverse-sorted creation order
    a, b = rng.standard_normal(33).astype(np.float32), rng.standard_normal(5).astype(np.float32)
    p = str(tmp_path / "two.ex")
    wav2h5.write_ex_batch([p], ("zeta", "alpha"), [[a, b]], threads=1)
    with h5lite.File(str(tmp_path / "two_py.ex"), "w") as w:
        w.create_dataset("zeta", data=a)
        w.create_dataset("alpha", data=b)
    assert open(p, "rb").read() == open(tmp_path / "two_py.ex", "rb").read()
    with h5lite.File(p, "r") as r:
        assert list(r) == ["alpha", "zeta"] and np.array_equal(r["zeta"][:], a)
    with pytest.raises(_lib.AecError):
        wav2h5.write_ex_batch([p], ("same", "same"), [[a, b]])
    with pytest.raises(_lib.AecError):
        wav2h5.write_ex_batch([p], ("a/b", "c"), [[a, b]])
    with pytest.raises(_lib.AecError):
        wav2h5.write_ex_batch([p], tuple(f"d{i}" for i in range(9)), [[a] * 9])
    with pytest.raises(_lib.AecError):
        wav2h5.write_ex_batch([str(tmp_path / "no_such_dir" / "x.ex")], ("a",), [[a]])


def test_create_h5_train_native_and_python_writers_agree(tmp_path):
    wav_dir, val_dir, h5_dir, list_dir, ids, data, vdata = _make_sets(tmp_path)
    out = {}
    for native in (True, False):
        d = tmp_path / f"h5_{native}"
        d.mkdir()
        args = types.SimpleNamespace(train_path=str(wav_dir), h5_path=str(d), list_path=str(list_dir), sr=16000)
        paths = wav2h5.create_h5_train(args, runner=_fake_runner, batch=4, h5=h5lite, native_writer=native)
        out[native] = {os.path.basename(p): open(p, "rb").read() for p in paths}
    assert out[True] == out[False] and len(out[True]) == len(ids)


def test_ex_writer_flag_selects_the_container():
    a = wav2h5.build_parser("train").parse_args(["--ex_writer", "native"])
    assert wav2h5.container_from_args(a) is h5lite
    assert wav2h5.container_from_args(wav2h5.build_parser("val").parse_args([])) is None
    assert wav2h5.container_from_args(types.SimpleNamespace()) is None            # the reference's own argparse namespace


def test_random_trees_round_trip_property():
    """hypothesis: random group trees (names incl. UTF-8, shared prefixes, up to 40 members per group -> several
    symbol-table nodes), random dtypes / shapes -> the structural walk and the reader both return what went in"""
    hyp = pytest.importorskip("hypothesis")
    import tempfile

    from hypothesis import strategies as st

    names = st.text(alphabet=st.characters(blacklist_characters="/\x00", blacklist_categories=("Cs",)), min_size=1, max_size=12)
    dtypes = st.sampled_from([np.float32, np.float64, np.int16, np.int32, np.int64, np.uint8])
    shapes = st.one_of(st.tuples(st.integers(0, 40)), st.tuples(st.integers(0, 5), st.integers(1, 4)))
    leaf = st.tuples(dtypes, shapes, st.integers(0, 2 ** 31 - 1))
    tree = st.dictionaries(names, st.one_of(leaf, st.dictionaries(names, leaf, max_size=12)), max_size=40)

    def build(w, spec, prefix, ref):
        for name, v in spec.items():
            if isinstance(v, dict):
                build(w.create_group(name), v, prefix + name + "/", ref)
            else:
                dt, shape, seed = v
                a = (np.random.default_rng(seed).standard_normal(shape) * 100).astype(dt)
                w.create_dataset(name, data=a)
                ref[prefix + name] = a

    @hyp.settings(max_examples=40, deadline=None)
    @hyp.given(tree)
    def check(spec):
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "t.h5")
            ref = {}
            with h5lite.File(path, "w") as w:
                build(w, spec, "", ref)
            found = _walk_file(path)
            assert set(found) == set(ref)
            with h5lite.File(path, "r") as r:
                assert sorted(r) == sorted(spec)
                for k, a in ref.items():
                    assert found[k].dtype == a.dtype and np.array_equal(found[k], a)
                    got = r[k][...]
                    assert got.shape == a.shape and got.dtype == a.dtype and np.array_equal(got, a)

    check()
