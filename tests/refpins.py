"""Answers of the original OpenSeq2Seq code, stored as data under tests/golden/reference/.

The tests that compare this project with the original ask `Pins(name)(key, compute)` for every value the original
produces.  Normally the stored answer is returned, so those tests run on any machine.  With OS2S_REFERENCE_ROOT set
to a checkout of NVIDIA/OpenSeq2Seq, `compute(root)` runs the original's own code from that checkout instead and the
stored answer is rewritten (`OS2S_REFERENCE_ROOT=<checkout> pytest -m "not gpu" tests` regenerates them all).

Arrays are stored small: shape, dtype, a digest of their values (for exact comparisons), their sum and largest
magnitude, and an evenly spread sample of their elements.  `equal` and `close` compare a computed array with such a
stored one; record and replay go through the same comparisons.
"""
import hashlib
import json
import os

import numpy as np

REFERENCE_ROOT = os.environ.get("OS2S_REFERENCE_ROOT") or None
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
SAMPLE = 32


def _np(x):
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    return np.asarray(x)


def _canonical(a):
    if a.dtype == np.bool_:
        return a.astype(np.uint8)
    if np.issubdtype(a.dtype, np.integer):
        return a.astype(np.int64)
    return a.astype(np.float64)


def digest(x):
    a = _np(x)
    h = hashlib.sha256(repr(tuple(a.shape)).encode())
    h.update(np.ascontiguousarray(_canonical(a)).tobytes())
    return h.hexdigest()[:24]


def sample_index(n, k):
    """k positions spread over [0, n): one per stripe of n / k elements, at a varying offset inside the stripe."""
    if n <= k:
        return np.arange(n)
    j = np.arange(k, dtype=np.int64)
    return (j * n) // k + (j * 7919) % (n // k)


class PinnedArray(object):
    def __init__(self, d):
        self.shape = tuple(d["shape"])
        self.dtype = d["dtype"]
        self.digest = d["digest"]
        self.sum = d["sum"]
        self.absmax = d["absmax"]
        self.values = np.asarray(d["values"], dtype=np.float64)
        self.size = int(np.prod(self.shape, dtype=np.int64))
        self.index = sample_index(self.size, len(self.values))

    def __len__(self):
        return self.shape[0]


def _encode(v, k):
    if hasattr(v, "detach") or isinstance(v, np.ndarray):
        a = _np(v)
        flat = _canonical(a).reshape(-1).astype(np.float64)
        idx = sample_index(flat.size, k)
        if a.dtype == np.float32:     # by their shortest float32 representation (within half a float32 ulp)
            values = [float(np.format_float_scientific(x, unique=True)) for x in a.reshape(-1)[idx]]
        else:
            values = [float(x) for x in flat[idx]]
        return {"__array__": {"shape": list(a.shape), "dtype": str(a.dtype), "digest": digest(a),
                              "sum": float(flat.sum()), "absmax": float(np.abs(flat).max()) if flat.size else 0.0,
                              "values": values}}
    if isinstance(v, np.generic):
        return v.item()
    if isinstance(v, dict):
        assert all(isinstance(key, str) for key in v), v.keys()
        return {key: _encode(x, k) for key, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [_encode(x, k) for x in v]
    assert v is None or isinstance(v, (bool, int, float, str)), type(v)
    return v


def _decode(v):
    if isinstance(v, dict):
        if "__array__" in v:
            return PinnedArray(v["__array__"])
        return {key: _decode(x) for key, x in v.items()}
    if isinstance(v, list):
        return [_decode(x) for x in v]
    return v


class Pins(object):
    """The stored answers of one test module (tests/golden/reference/<name>.json)."""

    def __init__(self, name):
        self.path = os.path.join(GOLDEN, name + ".json")
        self.data = json.load(open(self.path)) if os.path.exists(self.path) else {}

    def __call__(self, key, compute, sample=SAMPLE):
        if REFERENCE_ROOT:
            self.data[key] = _encode(compute(REFERENCE_ROOT), sample)
            os.makedirs(GOLDEN, exist_ok=True)
            with open(self.path, "w") as f:
                json.dump(self.data, f, sort_keys=True, separators=(",", ":"))
                f.write("\n")
        if key not in self.data:
            raise KeyError("%s: no stored answer for %r (regenerate with OS2S_REFERENCE_ROOT set)" % (self.path, key))
        return _decode(self.data[key])


def equal(got, want):
    """got (array / tensor) has exactly the values of the stored array `want`."""
    return tuple(_np(got).shape) == want.shape and digest(got) == want.digest


def max_dev(got, want):
    """Largest deviation of `got` from `want` over the stored sample, its sum (divided by the element count) and its
    largest magnitude."""
    g = _canonical(_np(got)).astype(np.float64)
    assert tuple(g.shape) == want.shape, (tuple(g.shape), want.shape)
    if not want.size:
        return 0.0
    dev = np.abs(g.reshape(-1)[want.index] - want.values)
    return float(max(dev.max() if dev.size else 0.0, abs(g.sum() - want.sum) / want.size,
                     abs(np.abs(g).max() - want.absmax)))


def close(got, want, atol=0.0, rtol=0.0):
    """np.allclose(got, want, rtol, atol) on the stored sample; the sum (per element) and the largest magnitude agree
    to within atol + rtol * largest magnitude."""
    g = _canonical(_np(got)).astype(np.float64)
    assert tuple(g.shape) == want.shape, (tuple(g.shape), want.shape)
    if not want.size:
        return True
    s = g.reshape(-1)[want.index]
    tol = atol + rtol * want.absmax
    return bool(np.all(np.abs(s - want.values) <= atol + rtol * np.abs(want.values))
                and abs(g.sum() - want.sum) / want.size <= tol and abs(np.abs(g).max() - want.absmax) <= tol)


# ------------------------------------------------------------------------------------------ configs
def encode_config(x):
    """A config value of the original's example configs (loaded through the drop-in `open_seq2seq` package) -> JSON:
    classes and functions by import path, activation lambdas by what they compute."""
    if isinstance(x, dict):
        return {k: encode_config(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [encode_config(v) for v in x]
    if x is None or isinstance(x, (bool, int, float, str)):
        return x
    import tensorflow as tf
    if isinstance(x, tf.DType):
        return {"__dtype__": x.name}
    if getattr(x, "__name__", "") == "<lambda>":
        return {"__activation__": list(tf.resolve_activation(x))}
    path = "%s:%s" % (x.__module__, x.__qualname__)
    assert _import(path) is x, path
    return {"__py__": path}


def _import(path):
    import importlib
    mod, qual = path.split(":")
    obj = importlib.import_module(mod)
    for part in qual.split("."):
        obj = getattr(obj, part)
    return obj


def decode_config(x):
    if isinstance(x, dict):
        if "__py__" in x:
            return _import(x["__py__"])
        if "__dtype__" in x:
            import tensorflow as tf
            return getattr(tf, x["__dtype__"])
        if "__activation__" in x:
            import tensorflow as tf
            kind, clip = x["__activation__"]
            assert kind == 1, kind
            if not clip:
                return tf.nn.relu
            return lambda t: tf.minimum(tf.nn.relu(t), clip)
        return {k: decode_config(v) for k, v in x.items()}
    if isinstance(x, list):
        return [decode_config(v) for v in x]
    return x


CONFIG_KEYS = ("base_model", "base_params", "train_params", "eval_params", "infer_params", "interactive_infer_params")


def config_imports(name):
    """What example_configs/speech2text/<name> of the original imports, as [module, name or None, alias or None]
    per imported name (read from the syntax tree of its import statements)."""
    def compute(root):
        import ast
        tree = ast.parse(open(os.path.join(root, "example_configs", "speech2text", name)).read())
        out = []
        for node in ast.walk(tree):
            if isinstance(node, ast.Import):
                out += [[a.name, None, a.asname] for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                assert node.level == 0, (name, node.module)
                out += [[node.module, a.name, a.asname] for a in node.names]
        return out
    return Pins("example_configs")(name + "/imports", compute)


def import_names(imports):
    """Runs the imports of config_imports() through the drop-in packages; returns the names they bind."""
    import importlib
    bound = {}
    for module, attr, alias in imports:
        mod = importlib.import_module(module)
        if attr is None:
            bound[alias or module.split(".")[0]] = mod if alias else importlib.import_module(module.split(".")[0])
        else:
            bound[alias or attr] = getattr(mod, attr)
    return bound


def example_config(name, tmp_dir):
    """example_configs/speech2text/<name> of the original as a config file in tmp_dir that get_base_config can load:
    it makes the original's imports through the drop-in packages, then defines the same base_model and params dicts,
    read from the stored answer."""
    pins = Pins("example_configs")
    config_imports(name)

    def compute(root):
        from open_seq2seq.utils.utils import get_base_config
        cwd = os.getcwd()
        os.chdir(root)  # (paths in the configs are relative to the original's repository root)
        try:
            _, _, _, mod = get_base_config(["--config_file=" + os.path.join(root, "example_configs", "speech2text",
                                                                           name)])
        finally:
            os.chdir(cwd)
        return {k: encode_config(mod[k]) for k in CONFIG_KEYS if k in mod}
    pins(name, compute)
    path = os.path.join(str(tmp_dir), name)
    with open(path, "w") as f:
        f.write("from tests import refpins\n\n"
                "globals().update(refpins.import_names(refpins.config_imports(%r)))\n"
                "globals().update(refpins.decode_config(refpins.Pins(%r).data[%r]))\n" % (name, "example_configs", name))
    return path
