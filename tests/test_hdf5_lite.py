"""CPU tier: the built-in HDF5 reader (digdriver_b200/hdf5_lite.py) on a real HDF5 file (SciPy's MATLAB v7.3 test file,
written by libhdf5 through MATLAB) and on round trips through its own classic-format writer, including the pandas
fixed-format layout and the reference's per-element groups (SURVEY.md section 8 f-1)."""
import os
import struct
import zlib

import numpy as np
import pandas as pd
import pytest

from conftest import GOLDEN
from digdriver_b200 import hdf5_lite, storage

# a copy of scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat from SciPy 1.18.1 (BSD-3-Clause), 4 KB
SCIPY_MAT = os.path.join(GOLDEN, "testhdf5_7.4_GLNX86.mat")


def test_reads_a_real_libhdf5_file():
    with hdf5_lite.File(SCIPY_MAT) as f:
        assert f.base == 512 and f.keys("/") == ["testdouble"] and not f.is_group("testdouble")
        assert f.attrs("testdouble") == {"MATLAB_class": "double"}
        x = f["testdouble"]
        assert x.shape == (9, 1) and x.dtype == np.float64
        np.testing.assert_allclose(x[:, 0], np.linspace(0, 2 * np.pi, 9), rtol=1e-15)
        assert "nope" not in f and "testdouble" in f
        with pytest.raises(KeyError):
            f["nope"]


def test_writer_reader_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    many = {"e%04d" % i: ('data', np.arange(i, i + 3), {}) for i in range(700)}          # three B-tree levels
    tree = {"attrs": {"n_up": np.int64(1), "mappability_threshold": 0.5, "note": "hello"},
            "children": {"idx": ('data', rng.integers(0, 10 ** 6, (50, 3)).astype(np.int32), {"unit": "bp"}),
                         "mappability": ('data', rng.random(50), {}),
                         "flags": ('data', rng.random(20) < 0.5, {}),
                         "substitution_idx": ('data', np.array(["ACA>AAA", "TTT>TGT"]), {}),
                         "empty": ('data', np.zeros((0, 3)), {}),
                         "window_10000": {"attrs": {}, "children": {"K": {"attrs": {"k": np.int64(7)}, "children": many}}}}}
    path = str(tmp_path / "t.h5")
    hdf5_lite.hdf5_write(path, tree)
    assert storage._is_hdf5_file(path)
    with hdf5_lite.File(path) as f:
        assert f.keys("/") == sorted(tree["children"])
        a = f.attrs("/")
        assert a["n_up"] == 1 and a["mappability_threshold"] == 0.5 and a["note"] == "hello"
        for k in ("idx", "mappability", "flags", "empty"):
            want = tree["children"][k][1]
            got = f[k]
            assert got.dtype == want.dtype and np.array_equal(got, want), k
        assert f.attrs("idx") == {"unit": "bp"}
        assert [s.decode() for s in f["substitution_idx"]] == ["ACA>AAA", "TTT>TGT"]
        assert f.is_group("window_10000/K") and f.attrs("window_10000/K")["k"] == 7
        assert f.keys("window_10000/K") == sorted(many)
        assert np.array_equal(f["window_10000/K/e0456"], np.arange(456, 459))


def test_store_reads_hdf5_through_the_builtin_reader(tmp_path):
    """A directory store exported to HDF5 (pandas fixed-format groups, arrays, attributes, per-element groups) reads
    back identically through Store -> hdf5_lite, which is also the path a reference-produced .h5 takes here."""
    rng = np.random.default_rng(1)
    d = str(tmp_path / "store")
    st = storage.Store(d, "w")
    n = 40
    rp = pd.DataFrame({"CHROM": rng.integers(1, 23, n), "START": np.arange(n) * 10000, "END": np.arange(1, n + 1) * 10000,
                       "Y_TRUE": rng.poisson(20, n), "Y_PRED": rng.gamma(2.0, 10.0, n), "STD": rng.uniform(0.5, 5, n),
                       "FLAG": rng.random(n) < 0.2}, index=["chr1:%d-%d" % (i * 10000, (i + 1) * 10000) for i in range(n)])
    m192 = pd.DataFrame({"MUT_TYPE": ["A>C", "C>T", "G>A"], "CONTEXT": ["AAA", "ACG", "TGT"], "COUNT": [3.0, 0.0, 7.0],
                         "FREQ": [1e-6, 0.0, 2.5e-6]})
    totals = pd.Series(rng.integers(0, 10 ** 6, 64), index=["".join(t) for t in __import__("itertools").product("ACGT", repeat=3)])
    st.write_table("region_params", rp)
    st.write_table("sequence_model_192", m192)
    st.write_table("genome_counts", totals)
    st.write_array("idx", rp[["CHROM", "START", "END"]].values, dtype=np.int32)
    st.set_attrs(N_MUT_CDS=1234, N_SAMPLES=56, mappability_threshold=0.5)
    names = ["eltA", "eltB"]
    L, R = rng.integers(0, 9, (2, 192)).astype(np.float64), rng.integers(0, 999, (2, 192))
    ov = [[(1, 0, 10000), (1, 10000, 20000)], [(7, 50000, 60000)]]
    st.write_element_groups("window_10000/K1", names, L, R, ov)
    out = storage.export_hdf5(d, str(tmp_path / "model.h5"))
    h = storage.Store(out, "r")
    assert h.lite is not None or storage._have_hdf5()
    got = h.read_table("region_params")
    assert list(got.columns) == list(rp.columns) and list(got.index) == list(rp.index)
    for c in rp.columns:
        assert got[c].dtype == rp[c].dtype and np.array_equal(got[c].values, rp[c].values), c
    g192 = h.read_table("sequence_model_192")
    assert list(g192.MUT_TYPE) == list(m192.MUT_TYPE) and list(g192.CONTEXT) == list(m192.CONTEXT)
    assert np.array_equal(g192.FREQ.values, m192.FREQ.values) and list(g192.index) == [0, 1, 2]
    gt = h.read_table("genome_counts")
    assert list(gt.index) == list(totals.index) and np.array_equal(gt.values, totals.values)
    assert np.array_equal(h.read_array("idx"), rp[["CHROM", "START", "END"]].values) and h.read_array("idx").dtype == np.int32
    assert h.get_attrs() == {"N_MUT_CDS": 1234, "N_SAMPLES": 56, "mappability_threshold": 0.5}
    assert h.has("region_params") and h.has("idx") and not h.has("nope")
    n2, L2, R2, ov2 = h.read_element_groups("window_10000/K1", ["eltB", "eltA"])
    assert n2 == ["eltB", "eltA"] and np.array_equal(L2, L[::-1]) and np.array_equal(R2, R[::-1]) and ov2 == ov[::-1]
    with pytest.raises(RuntimeError):
        storage.Store(out, "a")                      # read-only without h5py


def _chunked_file(path, arr, chunk, shuffle):
    """A hand-assembled classic-format file with ONE chunked, deflate(+shuffle)-compressed 2-D dataset 'x', laid out as
    h5py's create_dataset(compression='gzip', shuffle=...) does (layout v3 class 2, B-tree v1 node type 1, filter
    pipeline v1) -- exercises the parts of the reader that hdf5_write never produces."""
    w = hdf5_lite._Writer()
    w.buf += b"\x00" * 96
    es = arr.dtype.itemsize
    entries = []
    for i in range(0, arr.shape[0], chunk[0]):
        for j in range(0, arr.shape[1], chunk[1]):
            c = np.zeros(chunk, dtype=arr.dtype)
            part = arr[i:i + chunk[0], j:j + chunk[1]]
            c[:part.shape[0], :part.shape[1]] = part
            raw = c.tobytes()
            if shuffle:
                raw = np.frombuffer(raw, dtype=np.uint8).reshape(-1, es).T.tobytes()
            z = zlib.compress(raw)
            entries.append(((i, j), len(z), w.alloc(z)))
    node = b"TREE" + struct.pack("<BBHQQ", 1, 0, len(entries), hdf5_lite.UNDEF, hdf5_lite.UNDEF)
    for (i, j), n, addr in entries:
        node += struct.pack("<IIQQQ", n, 0, i, j, 0) + struct.pack("<Q", addr)
    node += struct.pack("<IIQQQ", 0, 0, arr.shape[0], arr.shape[1], 0)
    btree = w.alloc(node)
    layout = struct.pack("<BBBQ", 3, 2, 3, btree) + struct.pack("<III", chunk[0], chunk[1], es)
    filt = b""
    nf = 0
    if shuffle:
        filt += struct.pack("<HHHH", 2, 0, 1, 1) + struct.pack("<I", es) + b"\x00" * 4
        nf += 1
    filt += struct.pack("<HHHH", 1, 0, 1, 1) + struct.pack("<I", 6) + b"\x00" * 4
    nf += 1
    pipeline = struct.pack("<BB6x", 1, nf) + filt
    ds = w.header([(0x01, hdf5_lite._ds_message(arr.shape)), (0x03, hdf5_lite._dt_message(arr.dtype)), (0x0B, pipeline),
                   (0x08, layout)])
    root, bt, heap = w.group({"attrs": {}, "children": {}})
    # replace the empty root by one holding 'x': simplest is to build the group by hand through the writer's pieces
    w2 = hdf5_lite._Writer()
    w2.buf = w.buf
    heap_data = bytearray(b"\x00" * 8) + b"x\x00" + b"\x00" * 6
    hd = w2.alloc(bytes(heap_data))
    hp = w2.alloc(b"HEAP" + struct.pack("<B3xQQQ", 0, len(heap_data), hdf5_lite.UNDEF, hd))
    sn = w2.alloc(b"SNOD" + struct.pack("<BxH", 1, 1) + struct.pack("<QQII16x", 8, ds, 0, 0) + b"\x00" * (40 * 7))
    tr = w2.alloc(b"TREE" + struct.pack("<BBHQQ", 0, 0, 1, hdf5_lite.UNDEF, hdf5_lite.UNDEF) + struct.pack("<QQQ", 0, sn, 8) +
                  b"\x00" * (16 * 31))
    rh = w2.header([(0x11, struct.pack("<QQ", tr, hp))])
    sb = hdf5_lite.SIGNATURE + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, 4, 16, 0)
    sb += struct.pack("<QQQQ", 0, hdf5_lite.UNDEF, len(w2.buf), hdf5_lite.UNDEF) + struct.pack("<QQII", 0, rh, 1, 0) + struct.pack("<QQ", tr, hp)
    w2.buf[0:96] = sb
    open(path, "wb").write(bytes(w2.buf))


@pytest.mark.parametrize("shuffle", [False, True])
def test_chunked_deflate_dataset(tmp_path, shuffle):
    arr = np.random.default_rng(3).integers(0, 50, (37, 3)).astype(np.int32)       # `idx`: int32 [Nw, 3], gzip
    path = str(tmp_path / "c.h5")
    _chunked_file(path, arr, (16, 2), shuffle)
    with hdf5_lite.File(path) as f:
        got = f["x"]
    assert got.dtype == np.int32 and np.array_equal(got, arr)


def test_variable_length_data_through_the_global_heap(tmp_path):
    """h5py stores str attributes as variable-length strings and PyTables stores pandas' object blocks as a VLArray of
    ONE pickled ndarray: both live in a global heap collection (GCOL).  Hand-assembled file, read back."""
    import pickle
    w = hdf5_lite._Writer()
    w.buf += b"\x00" * 96
    obj = np.array([["A>C", "AAA"], ["C>T", "ACG"]], dtype=object)
    blob = pickle.dumps(obj, protocol=2)
    items = [b"UTF-8 text \xc3\xa9", blob]
    body = b""
    for i, it in enumerate(items, start=1):
        body += struct.pack("<HHIQ", i, 1, 0, len(it)) + it + b"\x00" * (-len(it) % 8)
    body += struct.pack("<HHIQ", 0, 0, 0, 0)
    gcol = w.alloc(b"GCOL" + struct.pack("<B3xQ", 1, 16 + len(body)) + body)
    vl_str = struct.pack("<BBBBI", 0x10 | 9, 0x01 | (1 << 4), 0x01, 0, 16) + hdf5_lite._dt_message(np.dtype("S1"))
    vl_u8 = struct.pack("<BBBBI", 0x10 | 9, 0x00, 0, 0, 16) + hdf5_lite._dt_message(np.uint8)
    nm = b"title\x00"
    ds0 = hdf5_lite._ds_message(())
    attr = struct.pack("<BxHHH", 1, len(nm), len(vl_str), len(ds0)) + hdf5_lite._pad8(nm) + hdf5_lite._pad8(vl_str) + \
        hdf5_lite._pad8(ds0) + struct.pack("<IQI", len(items[0]), gcol, 1)
    raw = w.alloc(struct.pack("<IQI", len(blob), gcol, 2))
    layout = struct.pack("<BBQQ", 3, 1, raw, 16)
    ds = w.header([(0x01, hdf5_lite._ds_message((1,))), (0x03, vl_u8), (0x08, layout), (0x0C, attr)])
    heap_data = bytearray(b"\x00" * 8) + b"block1_values\x00" + b"\x00" * 2
    hd = w.alloc(bytes(heap_data))
    hp = w.alloc(b"HEAP" + struct.pack("<B3xQQQ", 0, len(heap_data), hdf5_lite.UNDEF, hd))
    sn = w.alloc(b"SNOD" + struct.pack("<BxH", 1, 1) + struct.pack("<QQII16x", 8, ds, 0, 0) + b"\x00" * (40 * 7))
    tr = w.alloc(b"TREE" + struct.pack("<BBHQQ", 0, 0, 1, hdf5_lite.UNDEF, hdf5_lite.UNDEF) + struct.pack("<QQQ", 0, sn, 8) +
                 b"\x00" * (16 * 31))
    rh = w.header([(0x11, struct.pack("<QQ", tr, hp))])
    sb = hdf5_lite.SIGNATURE + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, 4, 16, 0)
    sb += struct.pack("<QQQQ", 0, hdf5_lite.UNDEF, len(w.buf), hdf5_lite.UNDEF) + struct.pack("<QQII", 0, rh, 1, 0) + struct.pack("<QQ", tr, hp)
    w.buf[0:96] = sb
    path = str(tmp_path / "v.h5")
    open(path, "wb").write(bytes(w.buf))
    with hdf5_lite.File(path) as f:
        assert f.attrs("block1_values") == {"title": "UTF-8 text é"}
        got = f._pandas_values("block1_values")
    assert got.dtype == object and got.tolist() == obj.tolist()


def test_new_style_structures(tmp_path):
    """Superblock v2, version-2 object headers ('OHDR', with a continuation chunk 'OCHK'), compact groups made of link
    messages, version-3 attributes and a version-2 dataspace: what libhdf5 writes with libver='latest' as long as a
    group stays compact.  Hand-assembled, read back."""
    U = hdf5_lite.UNDEF
    buf = bytearray(b"\x00" * 48)                                   # superblock v2: 8 + 4 + 4*8 + 4 = 48 bytes

    def alloc(b):
        buf.extend(b"\x00" * (-len(buf) % 8))
        a = len(buf)
        buf.extend(b)
        return a

    def msg(mtype, data):
        return struct.pack("<BHB", mtype, len(data), 0) + data

    def ohdr(messages, cont=None):
        body = b"".join(messages)
        if cont is not None:
            body += msg(0x10, struct.pack("<QQ", cont[0], cont[1]))
        return alloc(b"OHDR" + struct.pack("<BBH", 2, 0x01, len(body)) + body + b"\x00" * 4)

    arr = np.arange(12, dtype=np.float64).reshape(3, 4) * 0.5
    data = alloc(arr.tobytes())
    ds2 = struct.pack("<BBBB", 2, 2, 0, 1) + struct.pack("<QQ", 3, 4)             # dataspace v2, simple, rank 2
    layout = struct.pack("<BBQQ", 3, 1, data, arr.nbytes)
    note = np.array(b"new style")
    a_dt, a_ds = hdf5_lite._dt_message(note.dtype), struct.pack("<BBBB", 2, 0, 0, 0)  # scalar dataspace v2
    attr3 = struct.pack("<BBHHHB", 3, 0, 5, len(a_dt), len(a_ds), 0) + b"note\x00" + a_dt + a_ds + note.tobytes()
    # the attribute lives in a continuation chunk of the dataset's header
    och_body = msg(0x0C, attr3)
    och = alloc(b"OCHK" + och_body + b"\x00" * 4)
    dset = ohdr([msg(0x01, ds2), msg(0x03, hdf5_lite._dt_message(arr.dtype)), msg(0x08, layout)],
                cont=(och, 4 + len(och_body) + 4))
    link = lambda name, addr: msg(0x06, struct.pack("<BBB", 1, 0, len(name)) + name.encode() + struct.pack("<Q", addr))  # noqa: E731
    linfo = msg(0x02, struct.pack("<BBQQ", 0, 0, U, U))                          # link info: no dense storage
    sub = ohdr([linfo, link("values", dset)])
    root = ohdr([linfo, link("grp", sub), link("also_values", dset)])
    sb = hdf5_lite.SIGNATURE + struct.pack("<BBBB", 2, 8, 8, 0) + struct.pack("<QQQQ", 0, U, len(buf), root) + b"\x00" * 4
    buf[0:48] = sb
    path = str(tmp_path / "n.h5")
    open(path, "wb").write(bytes(buf))
    with hdf5_lite.File(path) as f:
        assert f.keys("/") == ["also_values", "grp"] and f.keys("grp") == ["values"] and f.is_group("grp")
        assert np.array_equal(f["grp/values"], arr) and np.array_equal(f["also_values"], arr)
        assert f.attrs("grp/values") == {"note": "new style"}
