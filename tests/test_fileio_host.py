"""CPU: bioen_b200.fileio -- the reference's pickle / HDF5 interface (bioen/fileio.py) and the problem-file layout of
its optimisation tests (test/optimize/test_fileio_logw.py, test_fileio_forces.py)."""
import pickle
import struct

import numpy as np
import pytest


def _logw_list(rng, m=5, n=7):
    w0 = np.full((n, 1), 1.0 / n)
    return [rng.standard_normal((n, 1)), np.zeros((n, 1)), rng.standard_normal((m, n)), rng.standard_normal((m, n)),
            rng.standard_normal((1, m)), w0, 3.5]


def test_pickle_roundtrip_and_problem_layout(tmp_path):
    from bioen_b200 import fileio as fio
    rng = np.random.default_rng(0)
    data = _logw_list(rng)
    fn = str(tmp_path / "p.pkl")
    fio.dump(fn, data)
    back = fio.load(fn)
    assert len(back) == 7 and all(np.array_equal(a, b) for a, b in zip(data, back))
    P = fio.load_problem(fn)
    assert P["kind"] == "logw" and P["theta"] == 3.5 and P["yTilde"].shape == (5, 7) and P["YTilde"].shape == (1, 5)
    forces = [np.zeros((5, 1)), data[5], data[2], data[3], data[4], 0.25]
    fn2 = str(tmp_path / "f.pkl")
    fio.dump_pickle(fn2, forces)
    P2 = fio.load_problem(fn2)
    assert P2["kind"] == "forces" and P2["forces_init"].shape == (5, 1) and P2["theta"] == 0.25
    # np.matrix entries (what the reference's analyze layer and its legacy files hold) come back as plain ndarrays
    fio.dump_pickle(fn2, [np.matrix(a) if isinstance(a, np.ndarray) else a for a in forces])
    assert type(fio.load_problem(fn2)["yTilde"]) is np.ndarray
    with pytest.raises(ValueError):
        fio.load(str(tmp_path / "x.txt"))
    with pytest.raises(ValueError):
        fio.dump(str(tmp_path / "x.txt"), data)
    fio.dump_pickle(fn2, data[:3])
    with pytest.raises(ValueError):
        fio.load_problem(fn2, kind="logw")


def test_hdf5_interface(tmp_path):
    from bioen_b200 import fileio as fio
    rng = np.random.default_rng(1)
    data = _logw_list(rng)
    fn = str(tmp_path / "p.h5")
    try:
        import h5py  # noqa: F401
    except ImportError:
        with pytest.raises(ImportError, match="h5py"):       # a clear error, at call time (not at import time)
            fio.dump(fn, data, fio.LOGW_KEYS)
        with pytest.raises(ImportError, match="h5py"):
            fio.load(fn)
        return
    fio.dump(fn, data, fio.LOGW_KEYS)                         # test_fileio_logw.py:37-52
    back = fio.load(fn, hdf5_keys=fio.LOGW_KEYS)
    assert all(np.array_equal(a, b) for a, b in zip(data, back))
    P = fio.load_problem(fn)
    assert P["kind"] == "logw" and np.array_equal(P["yTilde"], data[3])
    fio.dump(fn, data)                                        # artificial sortable labels AA, AB, ...
    assert all(np.array_equal(a, b) for a, b in zip(data, fio.load(fn)))
    fio.dump(fn, {"a": data[2], "g": {"b": data[3]}})
    deep = fio.load(fn, hdf5_deep_mode=True)
    assert np.array_equal(deep["a"], data[2]) and np.array_equal(deep["g"]["b"], data[3])
    pk = str(tmp_path / "p.pkl")
    fio.dump(pk, data)
    fio.convert_to_hdf5(pk, fn, fio.LOGW_KEYS)
    assert np.array_equal(fio.load(fn, hdf5_keys=["yTilde"])[0], data[3])


def _py2_pickle(items):
    """A list pickled the way Python 2 wrote the reference's problem files (protocol 2): np.matrix objects whose
    dtype codes and raw data are Python 2 `str`s (SHORT_BINSTRING / BINSTRING), floats as BINFLOAT.  Python 3
    reads such a file only with encoding="latin1"."""
    def s(b):
        return b"U" + bytes([len(b)]) + b if len(b) < 256 else b"T" + struct.pack("<i", len(b)) + b

    def i(v):
        return b"K" + bytes([v]) if 0 <= v < 256 else b"J" + struct.pack("<i", v)

    def matrix(a):
        a = np.ascontiguousarray(a, dtype="<f8")
        dtype = (b"cnumpy\ndtype\n" + s(b"f8") + i(0) + i(1) + b"\x87R(" + i(3) + s(b"<") + b"NNN" + i(-1) + i(-1)
                 + i(0) + b"tb")
        return (b"cnumpy.core.multiarray\n_reconstruct\ncnumpy.matrixlib.defmatrix\nmatrix\n" + i(0) + b"\x85" + s(b"b")
                + b"\x87R(" + i(1) + b"(" + b"".join(i(n) for n in a.shape) + b"t" + dtype + b"\x89" + s(a.tobytes())
                + b"tb")
    body = b"".join(matrix(v) if isinstance(v, np.ndarray) else b"G" + struct.pack(">d", v) for v in items)
    return b"\x80\x02](" + body + b"e."


def test_reference_problem_files_load(tmp_path):
    """The reference's legacy (Python 2) problem files: data_deer_test_logw_M808xN10.pkl and data_forces_M64xN64.pkl,
    rebuilt in Python 2's pickle layout from their entries stored in tests/golden."""
    from conftest import load_golden
    from bioen_b200 import fileio as fio
    d = load_golden("data_deer_test_logw_M808xN10")
    fn = tmp_path / "data_deer_test_logw_M808xN10.pkl"
    fn.write_bytes(_py2_pickle([d[k] for k in fio.LOGW_KEYS[:-1]] + [float(d["theta"])]))
    with pytest.raises(UnicodeDecodeError):
        pickle.loads(fn.read_bytes())
    P = fio.load_problem(str(fn))
    assert P["kind"] == "logw" and P["yTilde"].shape[0] == 808 and P["GInit"].shape == (P["yTilde"].shape[1], 1)
    assert all(np.array_equal(P[k], d[k]) for k in fio.LOGW_KEYS[:-1]) and P["theta"] == d["theta"]
    d = load_golden("data_forces_M64xN64")
    fn = tmp_path / "data_forces_M64xN64.pkl"
    fn.write_bytes(_py2_pickle([d[k] for k in fio.FORCES_KEYS[:-1]] + [float(d["theta"])]))
    F = fio.load_problem(str(fn))
    assert F["kind"] == "forces" and F["yTilde"].shape == (64, 64) and F["forces_init"].shape == (64, 1)
    assert all(np.array_equal(F[k], d[k]) for k in fio.FORCES_KEYS[:-1]) and F["theta"] == d["theta"]


def test_open_matrix_npy(tmp_path):
    from bioen_b200 import fileio as fio
    a = np.random.default_rng(2).standard_normal((6, 9))
    fn = str(tmp_path / "m.npy")
    np.save(fn, a)
    mm = fio.open_matrix(fn)
    assert isinstance(mm, np.memmap) and mm.shape == (6, 9) and np.array_equal(mm[2:5], a[2:5])
    assert fio.open_matrix(a) is a
    with pytest.raises(ValueError):
        fio.open_matrix(str(tmp_path / "m.bin"))
