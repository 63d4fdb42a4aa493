"""CPU: the PE checkpoint reader (cmbpo_b200/checkpoint.py) against files laid out like PE.save
(models/pens/pe.py:736-764) writes them; where the reference source tree (CMBPO_REFERENCE_ROOT) is present, the layer
descriptions are also produced by the reference's own FC.__repr__ (models/pens/fc.py:46-50)."""
import os

import numpy as np
import pytest
from scipy.io import savemat

from oracle import cmbpo_oracle as orc, ref_stubs
from cmbpo_b200 import checkpoint as ck


def fc_repr(out, inp, act, wd, E):
    return "FC(output_dim=%r, input_dim=%r, activation=%r, weight_decay=%r, ensemble_size=%r)" % (out, inp, act, wd, E)


def write_like_pe_save(d, name, step, ens, scalers, nll=False, repr_fn=fc_repr):
    """nonoptvars (scalers) + optvars (W, b[E,1,out] per layer, then logvar bounds for NLL) -> .mat"""
    n_l = len(ens.W)
    with open(os.path.join(d, "%s_%s.nns" % (name, step)), "w+") as f:
        for l in range(n_l):
            out = ens.W[l].shape[2]
            act = ens.acts[l]
            if l == n_l - 1 and ens.probabilistic:
                out //= 2
            f.write("%s\n" % repr_fn(out, ens.W[l].shape[1], act, 2.5e-05 * (l + 1), ens.W[0].shape[0]))
    arrs = []
    if "in" in scalers:
        arrs += [ens.mu_in.reshape(1, -1), ens.var_in.reshape(1, -1)]
    if "out" in scalers:
        arrs += [ens.mu_out.reshape(1, -1), ens.var_out.reshape(1, -1)]
    for W, b in zip(ens.W, ens.b):
        arrs += [W, b.reshape(b.shape[0], 1, -1)]
    if nll:
        D = ens.W[-1].shape[2] // 2
        arrs += [np.full((1, D), 0.5, np.float32), np.full((1, D), -10.0, np.float32)]
    savemat(os.path.join(d, "%s_%s.mat" % (name, step)), {str(i): a for i, a in enumerate(arrs)})


@pytest.mark.parametrize("scalers,nll", [(("in", "out"), False), (("in", "out"), True), (("in",), False),
                                         (("out",), False), ((), False)])
def test_roundtrip_dynamics(tmp_path, scalers, nll):
    dyn, actor, v, vc = orc.make_problem(5, 17, 6, hidden=(32, 48))
    write_like_pe_save(str(tmp_path), "BNN", 40, dyn, scalers, nll)
    got = ck.read_pe_checkpoint(str(tmp_path), "BNN", 40)
    assert got["probabilistic"] is True and got["acts"] == list(dyn.acts)
    for a, b in zip(got["W"], dyn.W):
        assert np.array_equal(a, b) and a.dtype == np.float32
    for a, b in zip(got["b"], dyn.b):
        assert np.array_equal(a, b.reshape(b.shape[0], -1))
    for key, used in (("mu_in", "in" in scalers), ("var_in", "in" in scalers),
                      ("mu_out", "out" in scalers), ("var_out", "out" in scalers)):
        if used:
            assert np.array_equal(got[key].ravel(), getattr(dyn, key).ravel()), key
        else:
            assert got[key] is None, key
    assert (got["max_logvar"] is not None) == nll


def test_roundtrip_value_ensemble(tmp_path):
    dyn, actor, v, vc = orc.make_problem(6, 29, 8, hidden=(32, 32), vf_hidden=(16, 16))
    write_like_pe_save(str(tmp_path), "VEnsemble", 3, v, ("in", "out"))
    got = ck.read_pe_checkpoint(str(tmp_path), "VEnsemble", 3)
    assert got["probabilistic"] is False and len(got["W"]) == len(v.W)
    assert np.array_equal(got["W"][-1], v.W[-1])


def test_malformed_files_fail_loudly(tmp_path):
    dyn, *_ = orc.make_problem(7, 17, 6, hidden=(8, 8))
    write_like_pe_save(str(tmp_path), "M", 1, dyn, ("in", "out"))
    with open(os.path.join(str(tmp_path), "M_1.nns"), "a") as f:
        f.write("Dense(units=3)\n")
    with pytest.raises(ValueError):
        ck.read_pe_checkpoint(str(tmp_path), "M", 1)


@pytest.mark.skipif(not ref_stubs.reference_available(), reason="reference source tree not present")
def test_layer_lines_are_the_references_repr(tmp_path):
    ref = ref_stubs.load()
    import importlib
    FC = importlib.import_module("models.pens.fc").FC
    dyn, *_ = orc.make_problem(8, 17, 6, hidden=(24, 24))
    write_like_pe_save(str(tmp_path), "R", 2, dyn, ("in", "out"),
                       repr_fn=lambda out, inp, act, wd, E: repr(FC(out, input_dim=inp, activation=act,
                                                                     weight_decay=wd, ensemble_size=E)))
    got = ck.read_pe_checkpoint(str(tmp_path), "R", 2)
    assert got["acts"] == list(dyn.acts) and np.array_equal(got["W"][1], dyn.W[1])
    del ref
