"""Checkpoints: the native state file that resumes a run, and the reference's PE checkpoints (SURVEY.md
section 8f-3) in both directions, so that ensembles trained by the TF code base can drive the B200 rollout
and ensembles trained here can go back to it.

`save_state` / `load_state` write and read one `.npz` holding a nested dict of numpy arrays and plain values:
the `state_dict()` of B200PE, B200Policy, DeviceArchive and ModelSampler, and whatever else the caller adds
(the numpy random state its training loop draws from, say).  See INTEGRATION.md, "Checkpoint and resume".

`PE.save` (models/pens/pe.py:736-764) writes two files per model:
  * `<name>_<timestep>.nns`  -- one `repr(FC)` per layer (models/pens/fc.py:46-50), the last one with
    the end activation and, for a probabilistic model, HALF the real output width;
  * `<name>_<timestep>.mat`  -- scipy `savemat` of `sess.run(nonoptvars + optvars)` under the keys
    "0", "1", ...: nonoptvars = scaler_in (mu, var) then scaler_out (mu, var), each only if used
    (pe.py:203-213, pens/utils.py:189-194); optvars = per layer (weights [E,in,out], biases
    [E,1,out]) (fc.py:172-175), then (max_logvar, min_logvar) only for the NLL loss.
Elite indices are not part of the checkpoint (they are recomputed by `PE.train`, pe.py:396-399):
pass them in.  `write_pe_checkpoint` writes the same two files (PE.save does not write the Adam slots
either).
"""
import json
import os
import re
import zipfile

import numpy as np

from .pe import B200PE, layer_decays

# ---- the native state file --------------------------------------------------------------------------------------
STATE_FORMAT = 1
_VERSION_KEY, _META_KEY = "format_version", "meta"


def _encode(node, arrays, path):
    """The JSON description of `node`; its arrays (numpy scalars as 0-d arrays) go to `arrays` as (entry, array)."""
    if isinstance(node, dict):
        for k in node:
            if not isinstance(k, str):
                raise TypeError("%s: key %r is not a string" % (path or "state", k))
        return {"dict": {k: _encode(v, arrays, path + "/" + k) for k, v in node.items()}}
    if isinstance(node, list):
        return {"list": [_encode(v, arrays, "%s/%d" % (path, i)) for i, v in enumerate(node)]}
    if isinstance(node, (np.ndarray, np.generic)):
        a = np.asarray(node)
        arrays.append(("a%d" % len(arrays), a))
        return {"array": arrays[-1][0], "shape": list(a.shape), "dtype": a.dtype.str,
                "scalar": isinstance(node, np.generic)}
    if node is None or isinstance(node, (bool, int, float, str)):
        return {"value": node}
    raise TypeError("%s: cannot save a %s" % (path or "state", type(node).__name__))


def _decode(node, z, path):
    if not isinstance(node, dict):
        raise ValueError("%s: malformed metadata" % (path or "state"))
    if "dict" in node:
        return {k: _decode(v, z, path + "/" + k) for k, v in node["dict"].items()}
    if "list" in node:
        return [_decode(v, z, "%s/%d" % (path, i)) for i, v in enumerate(node["list"])]
    if "value" in node:
        return node["value"]
    if not {"array", "shape", "dtype", "scalar"} <= set(node):
        raise ValueError("%s: malformed metadata" % (path or "state"))
    if node["array"] not in z.files:
        raise ValueError("%s: the array is missing from the file" % path)
    a = z[node["array"]]
    if list(a.shape) != node["shape"] or a.dtype.str != node["dtype"]:
        raise ValueError("%s: array of shape %s / %s, recorded %s / %s"
                         % (path, list(a.shape), a.dtype.str, node["shape"], node["dtype"]))
    return a[()] if node["scalar"] else a


def save_state(path, state):
    """Write the nested dict `state` to `path` (.npz): dicts with string keys, lists, numpy arrays and scalars, and
    None / bool / int / float / str leaves.  Arrays are stored bit for bit and read back without pickle; the other
    leaves and the tree go to a JSON entry.  The file is written beside `path` and moved over it with os.replace
    once complete, so an interrupted save leaves the previous checkpoint intact."""
    if not isinstance(state, dict):
        raise TypeError("the state is a dict, not a %s" % type(state).__name__)
    arrays = []
    meta = json.dumps(_encode(state, arrays, ""))
    entries = [(_VERSION_KEY, np.array(STATE_FORMAT, np.int64)),
               (_META_KEY, np.frombuffer(meta.encode("utf-8"), np.uint8))] + arrays
    tmp = "%s.tmp%d" % (path, os.getpid())
    try:
        with open(tmp, "wb") as f:
            with zipfile.ZipFile(f, "w", zipfile.ZIP_STORED, allowZip64=True) as zf:
                for name, a in entries:
                    with zf.open(name + ".npy", "w", force_zip64=True) as fh:
                        np.lib.format.write_array(fh, a, allow_pickle=False)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.unlink(tmp)
        raise
    try:                                     # make the rename itself durable
        fd = os.open(os.path.dirname(os.path.abspath(path)), os.O_RDONLY)
    except OSError:
        return
    try:
        os.fsync(fd)
    except OSError:
        pass
    finally:
        os.close(fd)


def load_state(path):
    """The nested dict save_state() wrote.  Raises ValueError on an unknown format version, an array the metadata
    names that is missing, or an array whose shape or dtype differs from the recorded one."""
    with np.load(path, allow_pickle=False) as z:
        if _VERSION_KEY not in z.files or _META_KEY not in z.files:
            raise ValueError("%s is not a state file (no %s / %s entry)" % (path, _VERSION_KEY, _META_KEY))
        version = z[_VERSION_KEY]
        if version.shape != () or int(version) != STATE_FORMAT:
            raise ValueError("%s: unknown state format version %s (this code reads %d)" % (path, version, STATE_FORMAT))
        tree = json.loads(z[_META_KEY].tobytes().decode("utf-8"))
        if "dict" not in tree:
            raise ValueError("%s: malformed metadata" % path)
        return _decode(tree, z, "")


# ---- the reference's PE checkpoint ------------------------------------------------------------------------------
_FC = re.compile(r"FC\(output_dim=(?P<out>\d+), input_dim=(?P<inp>None|\d+), activation=(?P<act>None|'[^']*'|\"[^\"]*\"), "
                 r"weight_decay=(?P<wd>[^,]+), ensemble_size=(?P<E>\d+)\)")


def parse_nns(path):
    """[(output_dim, input_dim or None, activation or None, ensemble_size)] per layer."""
    layers = []
    with open(path) as f:
        for line in f:
            line = line.strip()
            if not line:
                continue
            m = _FC.fullmatch(line)
            if m is None:
                raise ValueError("unrecognised layer description in %s: %r" % (path, line))
            act = m.group("act")
            layers.append((int(m.group("out")), None if m.group("inp") == "None" else int(m.group("inp")),
                           None if act == "None" else act.strip("'\""), int(m.group("E"))))
    if not layers:
        raise ValueError("%s describes no layers" % path)
    return layers


def read_pe_checkpoint(model_dir, name, timestep):
    """Returns dict(W, b, acts, probabilistic, mu_in, var_in, mu_out, var_out, max_logvar, min_logvar)
    as plain numpy arrays (scalers None when the model was saved without them)."""
    from scipy.io import loadmat

    stem = os.path.join(model_dir, "%s_%s" % (name, timestep))
    layers = parse_nns(stem + ".nns")
    mat = loadmat(stem + ".mat")
    n = len([k for k in mat if k.isdigit()])
    arrs = [np.asarray(mat[str(i)], np.float32) for i in range(n)]
    L_ = len(layers)
    n_extra = n - 2 * L_                       # scalers (0 / 2 / 4) + logvar bounds (0 / 2)
    if n_extra not in (0, 2, 4, 6):
        raise ValueError("%s.mat holds %d arrays for %d layers" % (stem, n, L_))
    # the optimised variables are the LAST 2L (+2) arrays; decide by shape: layer weights are 3-D
    tail = arrs[-2 * L_:] if all(a.ndim == 3 for a in arrs[-2 * L_::2]) else None
    bounds = (None, None)
    if tail is None:                           # NLL loss: (max_logvar, min_logvar) trail the layers
        tail = arrs[-2 * L_ - 2:-2]
        bounds = (arrs[-2], arrs[-1])
        if not all(a.ndim == 3 for a in tail[::2]):
            raise ValueError("%s.mat: cannot locate the layer weights" % stem)
        n_scal = n - 2 * L_ - 2
    else:
        n_scal = n - 2 * L_
    W = [np.ascontiguousarray(a) for a in tail[0::2]]
    b = [np.ascontiguousarray(a.reshape(a.shape[0], -1)) for a in tail[1::2]]
    acts = [l[2] for l in layers]
    E, in_dim, last = W[0].shape[0], W[0].shape[1], W[-1].shape[2]
    for (out, inp, _, ens), w in zip(layers[:-1], W[:-1]):
        if w.shape[2] != out or ens != E or (inp is not None and inp != w.shape[1]):
            raise ValueError("%s: .nns and .mat disagree on a layer shape" % stem)
    if last == 2 * layers[-1][0]:
        probabilistic = True
    elif last == layers[-1][0]:
        probabilistic = False
    else:
        raise ValueError("%s: last layer width %d vs described %d" % (stem, last, layers[-1][0]))
    d_out = last // 2 if probabilistic else last
    # The .nns last-layer activation is the reference's `end_act`, which a probabilistic net applies to the
    # MEAN half only, after unsetting the layer activation (pe.py:183-185, 817-818).  The kernels have no
    # mean-only output activation, so refuse it rather than apply it to the log-variance half as well.
    if probabilistic and acts[-1] not in (None, "None", "none", "linear"):
        raise ValueError("%s: output_activation %r on a probabilistic ensemble is not supported "
                         "(the reference applies it to the mean half only)" % (stem, acts[-1]))
    scal = [a.reshape(1, -1) for a in arrs[:n_scal]]
    mu_in = var_in = mu_out = var_out = None
    if n_scal == 4:
        mu_in, var_in, mu_out, var_out = scal
    elif n_scal == 2:                          # one scaler only: tell input from output by its width
        if scal[0].shape[1] == in_dim and in_dim != d_out:
            mu_in, var_in = scal
        elif scal[0].shape[1] == d_out and in_dim != d_out:
            mu_out, var_out = scal
        else:
            raise ValueError("%s: a single scaler of width %d is ambiguous (in %d, out %d)"
                             % (stem, scal[0].shape[1], in_dim, d_out))
    elif n_scal != 0:
        raise ValueError("%s.mat: %d leading arrays are not a set of scalers" % (stem, n_scal))
    return dict(W=W, b=b, acts=acts, probabilistic=probabilistic, mu_in=mu_in, var_in=var_in,
                mu_out=mu_out, var_out=var_out, max_logvar=bounds[0], min_logvar=bounds[1])


def _fc_repr(output_dim, input_dim, activation, weight_decay, ensemble_size):
    """FC.__repr__ (models/pens/fc.py:46-50)."""
    return "FC(output_dim=%r, input_dim=%r, activation=%r, weight_decay=%r, ensemble_size=%r)" % (
        output_dim, input_dim, activation, weight_decay, ensemble_size)


def write_pe_checkpoint(model_dir, name, timestep, pe):
    """`PE.save` (pe.py:736-764) of a B200PE (or of the dict its state_dict() returns), readable by the reference's
    `PE(load_model=True)` and by read_pe_checkpoint / load_pe: `<name>_<timestep>.nns` with one FC line per layer
    (weight decay from configure_training's `decay`, None when training was never configured) and
    `<name>_<timestep>.mat` with the scalers in use, then W [E,in,out] and b [E,1,out] per layer."""
    from scipy.io import savemat

    sd = pe.state_dict() if hasattr(pe, "state_dict") else pe
    layers = sd["layers"]
    n_l, E = len(layers), int(layers[0]["W"].shape[0])
    decays = layer_decays(sd["train"]["decay"], n_l) if sd.get("train") else [None] * n_l
    lines = []
    for l, (x, act, wd) in enumerate(zip(layers, sd["acts"], decays)):
        out = int(x["W"].shape[2])
        if l == n_l - 1 and sd["probabilistic"]:
            out //= 2                                  # pe.py:179-180: the layer was declared with the mean width
        lines.append(_fc_repr(out, int(x["W"].shape[1]), act, wd, E) + "\n")
    sc = sd["scalers"]
    arrs = [np.asarray(sc[k], np.float32).reshape(1, -1)
            for pair in (("mu_in", "var_in"), ("mu_out", "var_out")) if sc[pair[0]] is not None for k in pair]
    for x in layers:
        arrs += [np.asarray(x["W"], np.float32), np.asarray(x["b"], np.float32).reshape(E, 1, -1)]
    stem = os.path.join(model_dir, "%s_%s" % (name, timestep))
    with open(stem + ".nns", "w") as f:
        f.writelines(lines)
    savemat(stem + ".mat", {str(i): a for i, a in enumerate(arrs)})


def load_pe(engine, which, model_dir, name, timestep, elite_inds=None):
    """`PE(load_model=True)` (pe.py:87-96,121-160) for the B200 engine: reads the checkpoint and
    uploads it into ensemble slot `which`; returns the model object FakeEnv / CPOPolicy consume."""
    ck = read_pe_checkpoint(model_dir, name, timestep)
    E = ck["W"][0].shape[0]
    elites = list(range(E)) if elite_inds is None else [int(i) for i in elite_inds]
    return B200PE(engine, which, ck["W"], ck["b"], ck["acts"], ck["probabilistic"], elites,
                  ck["mu_in"], ck["var_in"], ck["mu_out"], ck["var_out"], name=name)


# ---- the policy's SavedModel (utilities/logx.py:202-259, policies/cpo_policy.py:890-894) ---------------------------
_DENSE = re.compile(r"(?P<scope>.*/)?pi/dense(?:_(?P<i>\d+))?/(?P<kind>kernel|bias)")
_FCVAR = re.compile(r"(?P<scope>.*/)?(?P<ens>[^/]+)/Layer(?P<i>\d+)/FC_(?P<kind>weights|biases)")


class _Ens:
    pass


def read_policy_savedmodel(export_dir, vf_activation="swish", vf_elites=None):
    """Variables of the SavedModel that `CPOPolicy.save` writes -> dict(actor_W, actor_b, log_std, v, vc).

    The builder stores every global variable of the session under its graph name (no TensorFlow needed to read
    them, see tf_bundle.py):
      * the actor: `AC/pi/dense{,_1,_2}/{kernel,bias}` ([in,out] / [out], tanh hidden, linear output) and
        `AC/pi/log_std` (network/ac_network.py:26-33, 99-123);
      * the value ensembles `AC/VEnsemble/...`, `AC/VCEnsemble/...` (policies/cpo_policy.py:467-468): per layer
        `Layer<i>/FC_weights` [E,in,out], `FC_biases` [E,1,out] (models/pens/fc.py:135-166), the scalers
        `scaler_in_mu`, `scaler_in_std` (which holds the VARIANCE, pens/utils.py:112-114), `scaler_out_*`, and
        `max_log_var` / `min_log_var` when trained with the NLL loss (pe.py:199-202).
    Optimizer slots (`.../Adam`, `.../Adam_1`) are ignored.  The hidden activation and the elite list are
    constructor arguments in the reference, not variables: pass them (`vf_activation`, `vf_elites`)."""
    from .tf_bundle import read_bundle, read_index

    prefix = os.path.join(export_dir, "variables", "variables")
    entries, _ = read_index(prefix + ".index")
    keys = ("scaler_in_mu", "scaler_in_std", "scaler_out_mu", "scaler_out_std", "max_log_var", "min_log_var")
    wanted = [n for n in entries
              if not n.endswith(("/Adam", "/Adam_1")) and (_DENSE.fullmatch(n) or n.endswith("pi/log_std") or
                  (n.split("/")[-2:-1] in (["VEnsemble"], ["VCEnsemble"]) and n.split("/")[-1] in keys) or
                  (_FCVAR.fullmatch(n) and _FCVAR.fullmatch(n).group("ens") in ("VEnsemble", "VCEnsemble")))]
    tens = read_bundle(prefix, names=wanted)        # the dynamics model and optimizer slots of the same graph stay on disk
    dense = {}
    log_std = None
    ens = {}
    for name, a in tens.items():
        if name.endswith("/Adam") or name.endswith("/Adam_1"):
            continue
        m = _DENSE.fullmatch(name)
        if m:
            dense.setdefault(int(m.group("i") or 0), {})[m.group("kind")] = a
            continue
        if name.endswith("pi/log_std"):
            log_std = np.asarray(a, np.float32).reshape(-1)
            continue
        m = _FCVAR.fullmatch(name)
        if m:
            ens.setdefault(m.group("ens"), {}).setdefault("layers", {}).setdefault(int(m.group("i")), {})[m.group("kind")] = a
            continue
        for key in ("scaler_in_mu", "scaler_in_std", "scaler_out_mu", "scaler_out_std", "max_log_var", "min_log_var"):
            if name.endswith("/" + key):
                ens.setdefault(name.split("/")[-2], {})[key] = a
    if not dense or log_std is None:
        raise ValueError("%s holds no Gaussian MLP actor (pi/dense*/kernel, pi/log_std)" % export_dir)
    idx = sorted(dense)
    if idx != list(range(len(idx))) or any(set(dense[i]) != {"kernel", "bias"} for i in idx):
        raise ValueError("%s: incomplete actor layers %s" % (export_dir, idx))
    out = dict(actor_W=[np.asarray(dense[i]["kernel"], np.float32) for i in idx],
               actor_b=[np.asarray(dense[i]["bias"], np.float32) for i in idx], log_std=log_std)
    for key, ens_name in (("v", "VEnsemble"), ("vc", "VCEnsemble")):
        e = ens.get(ens_name)
        if e is None or "layers" not in e:
            out[key] = None
            continue
        li = sorted(e["layers"])
        if li != list(range(len(li))) or any(set(e["layers"][i]) != {"weights", "biases"} for i in li):
            raise ValueError("%s: incomplete %s layers %s" % (export_dir, ens_name, li))
        o = _Ens()
        o.W = [np.ascontiguousarray(e["layers"][i]["weights"], np.float32) for i in li]
        o.b = [np.ascontiguousarray(np.asarray(e["layers"][i]["biases"], np.float32).reshape(o.W[0].shape[0], -1)) for i in li]
        o.acts = [vf_activation] * (len(li) - 1) + [None]
        o.probabilistic = "max_log_var" in e
        E = o.W[0].shape[0]
        o.elite_inds = list(range(E)) if vf_elites is None else [int(i) for i in vf_elites]
        for nm, src in (("mu_in", "scaler_in_mu"), ("var_in", "scaler_in_std"), ("mu_out", "scaler_out_mu"), ("var_out", "scaler_out_std")):
            setattr(o, nm, np.asarray(e[src], np.float32).reshape(1, -1) if src in e else None)
        o.max_logvar = e.get("max_log_var")
        o.min_logvar = e.get("min_log_var")
        out[key] = o
    return out


def load_policy(engine, export_dir, vf_activation="swish", vf_elites=None, seed=0):
    """A `B200Policy` driven by the variables of the reference's policy SavedModel."""
    from .policy import B200Policy

    ck = read_policy_savedmodel(export_dir, vf_activation, vf_elites)
    if ck["v"] is None or ck["vc"] is None:
        raise ValueError("%s holds no VEnsemble / VCEnsemble variables" % export_dir)
    pol = B200Policy(engine, seed=seed)
    pol.load_actor(ck["actor_W"], ck["actor_b"], ck["log_std"])
    pol.load_values(ck["v"], ck["vc"])
    return pol
