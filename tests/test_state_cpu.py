"""CPU: the native state file (checkpoint.save_state / load_state) and the writer of the reference's PE checkpoint
(checkpoint.write_pe_checkpoint), read back by read_pe_checkpoint; where the reference source tree
(CMBPO_REFERENCE_ROOT) is present, the layer lines are compared with the reference's own FC.__repr__
(models/pens/fc.py:46-50)."""
import os
import struct
import zipfile

import numpy as np
import pytest

from oracle import cmbpo_oracle as orc, ref_stubs
from cmbpo_b200 import checkpoint as ck


def _state():
    rs = np.random.RandomState(7)
    rs.standard_normal()                              # a cached gaussian in the state
    name, keys, pos, has_gauss, cached = rs.get_state()
    rng = np.random.default_rng(3)
    return {
        "f32": rng.standard_normal((3, 4)).astype(np.float32),
        "f64_special": np.array([np.nan, -0.0, np.inf, -np.inf, 5e-324, 1.0 / 3.0]),
        "ints": {"i8": np.arange(-4, 4, dtype=np.int8), "u32": np.array([0, 2 ** 32 - 1], np.uint32),
                 "i64": np.array([-(2 ** 63), 2 ** 63 - 1], np.int64)},
        "bool_arr": np.array([[True, False]]),
        "empty": np.zeros((0, 5), np.float32),
        "zero_d": np.array(2.5, np.float16),
        "strided": rng.standard_normal((4, 6))[:, ::2],
        "np_scalars": [np.float32(0.1), np.int64(-3), np.float64(np.pi), np.bool_(True)],
        "plain": [None, True, False, 0, -(10 ** 30), 1.5, -0.0, 1e-310, float("inf"), "", "Ωmega/πk", []],
        "nested": {"list_of_arrays": [np.ones(2, np.float32), {"deep": [np.arange(3)]}], "empty": {}},
        "rng": {"name": name, "keys": keys, "pos": pos, "has_gauss": has_gauss, "cached_gaussian": cached},
    }


def _same(a, b, path="state"):
    assert type(a) is type(b), (path, type(a), type(b))
    if isinstance(a, dict):
        assert list(a) == list(b), path
        for k in a:
            _same(a[k], b[k], path + "/" + k)
    elif isinstance(a, list):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, "%s/%d" % (path, i))
    elif isinstance(a, (np.ndarray, np.generic)):
        assert a.dtype == b.dtype and np.shape(a) == np.shape(b), path
        assert np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes(), path
    elif isinstance(a, float):
        assert struct.pack("<d", a) == struct.pack("<d", b), path
    else:
        assert a == b, path


def test_roundtrip_every_leaf_type_bit_for_bit(tmp_path):
    path = str(tmp_path / "state.npz")
    st = _state()
    ck.save_state(path, st)
    got = ck.load_state(path)
    _same(st, got)
    rs = np.random.RandomState()
    r = got["rng"]
    rs.set_state((r["name"], r["keys"], r["pos"], r["has_gauss"], r["cached_gaussian"]))
    want = np.random.RandomState(7)
    want.standard_normal()
    assert np.array_equal(rs.standard_normal(5), want.standard_normal(5))
    # every entry is a plain .npy array that numpy reads without pickle
    with zipfile.ZipFile(path) as zf:
        names = zf.namelist()
    assert all(n.endswith(".npy") for n in names)
    with np.load(path, allow_pickle=False) as z:
        assert all(z[n].dtype != object for n in z.files)
    assert os.listdir(str(tmp_path)) == ["state.npz"]


@pytest.mark.parametrize("bad", [(1, 2), {1, 2}, object(), {3: "int key"}, b"bytes"])
def test_unsupported_leaves_are_refused(tmp_path, bad):
    with pytest.raises(TypeError):
        ck.save_state(str(tmp_path / "s.npz"), {"x": [bad]})
    assert os.listdir(str(tmp_path)) == []


def _entries(path):
    with np.load(path, allow_pickle=False) as z:
        return {n: z[n] for n in z.files}


def test_load_refuses_unknown_version_missing_entries_and_wrong_shapes(tmp_path):
    good = str(tmp_path / "good.npz")
    ck.save_state(good, {"W": np.ones((2, 3), np.float32), "n": 4})
    assert ck.load_state(good)["n"] == 4
    e = _entries(good)
    bad = str(tmp_path / "bad.npz")

    def refused(entries, match):
        np.savez(bad, **entries)
        with pytest.raises(ValueError, match=match):
            ck.load_state(bad)

    refused(dict(e, format_version=np.array(2, np.int64)), "version")
    refused({k: v for k, v in e.items() if k != "format_version"}, "not a state file")
    refused({k: v for k, v in e.items() if k != "meta"}, "not a state file")
    refused({k: v for k, v in e.items() if k != "a0"}, "missing")
    refused(dict(e, a0=np.ones((3, 2), np.float32)), "shape")
    refused(dict(e, a0=np.ones((2, 3), np.float64)), "shape")


def test_a_failed_save_leaves_the_previous_file(tmp_path):
    path = str(tmp_path / "ck.npz")
    first = {"step": 1, "W": np.arange(12, dtype=np.float32).reshape(3, 4)}
    ck.save_state(path, first)
    # the object array fails while the file is being written, after the arrays before it were
    with pytest.raises(ValueError):
        ck.save_state(path, {"step": 2, "W": np.zeros((512, 512), np.float32), "z": np.array([object()], dtype=object)})
    _same(first, ck.load_state(path))
    assert os.listdir(str(tmp_path)) == ["ck.npz"]


# ---- write_pe_checkpoint -> read_pe_checkpoint ----------------------------------------------------------------------
def _pe_state(ens, scalers, decay):
    """The fields of B200PE.state_dict() that write_pe_checkpoint reads."""
    E = ens.W[0].shape[0]
    return {"layers": [{"W": W, "b": b.reshape(E, -1)} for W, b in zip(ens.W, ens.b)], "acts": list(ens.acts),
            "probabilistic": ens.probabilistic,
            "scalers": {k: (getattr(ens, k) if k.split("_")[1] in scalers else None)
                        for k in ("mu_in", "var_in", "mu_out", "var_out")},
            "train": None if decay is None else {"decay": decay}}


def _problem(kind):
    dyn, _, v, _ = orc.make_problem(5, 17, 6, hidden=(32, 48), vf_hidden=(16, 16))
    return {"both": (dyn, ("in", "out"), 1e-4), "one": (dyn, ("out",), 3e-5), "value": (v, (), None)}[kind]


@pytest.mark.parametrize("kind", ["both", "one", "value"])
def test_written_checkpoint_reads_back_identical(tmp_path, kind):
    ens, scalers, decay = _problem(kind)
    ck.write_pe_checkpoint(str(tmp_path), "BNN", 12, _pe_state(ens, scalers, decay))
    got = ck.read_pe_checkpoint(str(tmp_path), "BNN", 12)
    assert got["probabilistic"] is ens.probabilistic and got["acts"] == list(ens.acts)
    assert len(got["W"]) == len(ens.W)
    for a, w in zip(got["W"], ens.W):
        assert a.dtype == np.float32 and np.array_equal(a, w)
    for a, b in zip(got["b"], ens.b):
        assert np.array_equal(a, b.reshape(b.shape[0], -1))
    for k in ("mu_in", "var_in", "mu_out", "var_out"):
        if k.split("_")[1] in scalers:
            assert np.array_equal(got[k], getattr(ens, k).reshape(1, -1)), k
        else:
            assert got[k] is None, k
    assert got["max_logvar"] is None
    layers = ck.parse_nns(str(tmp_path / "BNN_12.nns"))
    last = ens.W[-1].shape[2] // (2 if ens.probabilistic else 1)
    assert [l[0] for l in layers] == [w.shape[2] for w in ens.W[:-1]] + [last]
    wds = [line.split("weight_decay=")[1].split(",")[0] for line in open(str(tmp_path / "BNN_12.nns"))]
    n = len(ens.W)
    want = ["None"] * n if decay is None else [repr(decay / 4)] + [repr(decay / 2)] * (n - 2) + [repr(decay)]
    assert wds == want


@pytest.mark.skipif(not ref_stubs.reference_available(), reason="reference source tree not present")
def test_written_layer_lines_are_the_references_repr(tmp_path):
    ref = ref_stubs.load()
    import importlib
    FC = importlib.import_module("models.pens.fc").FC
    ens, scalers, decay = _problem("both")
    ck.write_pe_checkpoint(str(tmp_path), "R", 2, _pe_state(ens, scalers, decay))
    n = len(ens.W)
    wds = [decay / 4] + [decay / 2] * (n - 2) + [decay]
    want = [repr(FC(w.shape[2] // (2 if l == n - 1 else 1), input_dim=w.shape[1], activation=ens.acts[l],
                    weight_decay=wds[l], ensemble_size=w.shape[0])) for l, w in enumerate(ens.W)]
    assert open(str(tmp_path / "R_2.nns")).read().splitlines() == want
    del ref
