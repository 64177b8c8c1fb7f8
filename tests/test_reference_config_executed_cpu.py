"""The reference's OWN config / params code against the drop-in package.

`open_seq2seq/utils/utils.py` of the reference is loaded BY PATH from a checkout of it (never copied); its only
TensorFlow import that matters at import time (`tensorflow.python.client.device_lib`) is replaced by an empty stand-in,
`tf` itself is the repo's minimal stand-in.  What runs is the reference's own get_base_config (argparse + runpy + the
nested command-line overrides), check_params, flatten_dict / nest_dict / nested_update and the id->text helpers; the
compat package's versions must return the same objects and raise on the same inputs.  The reference's answers are
stored under tests/golden/reference/reference_config.json (tests/refpins.py; OS2S_REFERENCE_ROOT re-runs the
reference and rewrites them).
"""
import copy
import hashlib
import importlib.util
import json
import os
import sys
import types

import pytest

import openseq2seq_b200.compat as compat

compat.install()
from open_seq2seq.utils import utils as OWN  # noqa: E402
from tests import refpins as RP  # noqa: E402

PINS = RP.Pins("reference_config")
_REF = {}


def ref_utils(root):
    """open_seq2seq/utils/utils.py of the reference checkout at `root`."""
    if root in _REF:
        return _REF[root]
    names = ("tensorflow.python", "tensorflow.python.client", "tensorflow.python.client.device_lib")
    fake = {n: types.ModuleType(n) for n in names}
    fake["tensorflow.python.client"].device_lib = fake["tensorflow.python.client.device_lib"]
    saved = {k: sys.modules.get(k) for k in fake}
    sys.modules.update(fake)
    try:
        spec = importlib.util.spec_from_file_location("_reference_utils",
                                                      os.path.join(root, "open_seq2seq", "utils", "utils.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    _REF[root] = mod
    return mod


def _digest(x):
    """Exact fingerprint of a JSON-able value (configs, dicts)."""
    return hashlib.sha256(json.dumps(x, sort_keys=True).encode()).hexdigest()[:16]


def _comparable(x):
    """Config values -> something == can compare (classes and functions by qualified name, activation lambdas by
    what they compute, dtypes by name)."""
    import tensorflow as tf
    if isinstance(x, dict):
        return {k: _comparable(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_comparable(v) for v in x]
    if isinstance(x, tf.DType):
        return repr(x)
    if getattr(x, "__name__", "") == "<lambda>":
        return "activation %r" % (tf.resolve_activation(x),)
    if isinstance(x, type) or callable(x):
        return getattr(x, "__module__", "") + "." + getattr(x, "__qualname__", repr(x))
    return x


OVERRIDES = [
    [],
    ["--batch_size_per_gpu=4", "--num_epochs=3"],
    ["--encoder_params/dropout_keep_prob=0.5", "--lr_policy_params/learning_rate=0.1", "--use_horovod=False"],
    ["--logdir=/tmp/x", "--data_layer_params/num_audio_features=80", "--optimizer_params/epsilon=1e-6",
     "--larc_params/larc_eta=0.002"],
]


@pytest.mark.parametrize("name", ["jasper10x5_LibriSpeech_nvgrad.py", "quartznet15x5_LibriSpeech.py",
                                  "w2lplus_large_8gpus_mp.py"])
@pytest.mark.parametrize("mode", ["train", "train_eval", "eval"])
def test_get_base_config_equals_the_executed_reference(name, mode, tmp_path):
    own_path = RP.example_config(name, tmp_path)      # the same config, loaded by the drop-in

    def reference(root, extra):
        ref = ref_utils(root)
        path = os.path.join(root, "example_configs", "speech2text", name)
        argv = ["--config_file=" + path, "--mode=" + mode] + extra
        keys = set(ref.flatten_dict(ref.get_base_config(["--config_file=" + path])[1]))
        usable = [a for a in argv if a.split("=")[0].lstrip("-") in keys or a.startswith(("--config_file", "--mode"))]
        r_args, r_base, r_model, r_mod = ref.get_base_config(list(usable))
        return {"usable": usable[1:], "base": _digest(_comparable(r_base)), "model": _comparable(r_model),
                "mod": {k: _digest(_comparable(r_mod.get(k))) for k in ("train_params", "eval_params", "infer_params")},
                "args": {k: v for k, v in vars(r_args).items() if k != "config_file"}}
    for i, extra in enumerate(OVERRIDES):
        want = PINS("get_base_config/%s/%s/%d" % (name, mode, i), lambda root: reference(root, extra))
        usable = ["--config_file=" + own_path] + want["usable"]
        o_args, o_base, o_model, o_mod = OWN.get_base_config(list(usable))
        assert want["base"] == _digest(_comparable(o_base)), (name, mode, usable)
        assert want["model"] == _comparable(o_model)
        for k in ("train_params", "eval_params", "infer_params"):
            assert want["mod"][k] == _digest(_comparable(o_mod.get(k))), k
        assert want["args"].keys() <= vars(o_args).keys()
        for k, v in want["args"].items():
            assert getattr(o_args, k) == v, k
        assert o_args.config_file == own_path

    def raises(root):
        try:
            ref_utils(root).get_base_config(["--config_file=" + os.path.join(root, "example_configs", "speech2text",
                                                                             name), "--mode=nonsense"])
        except ValueError:
            return True
        return False
    assert PINS("get_base_config/%s/nonsense_mode_raises" % name, raises)
    with pytest.raises(ValueError):
        OWN.get_base_config(["--config_file=" + own_path, "--mode=nonsense"])


def test_dict_helpers_equal_the_executed_reference():
    import random
    rnd = random.Random(0)

    def rand_dict(depth):
        d = {}
        for i in range(rnd.randint(1, 4)):
            k = "k%d_%d" % (depth, i)
            t = rnd.random()
            if t < 0.35 and depth < 3:
                d[k] = rand_dict(depth + 1)
            elif t < 0.5:
                d[k] = rnd.random()
            elif t < 0.65:
                d[k] = rnd.randint(-5, 5)
            elif t < 0.8:
                d[k] = rnd.choice([True, False])
            elif t < 0.9:
                d[k] = "s%d" % rnd.randint(0, 9)
            else:
                d[k] = [1, 2, 3]              # lists are dropped by flatten_dict
        return d

    cases = [(rand_dict(0), rand_dict(0)) for _ in range(200)]

    def helpers(lib, a, b):
        """(flatten_dict(a), nest_dict of it, a after nested_update(a, b) or None when that raised), as digests."""
        flat = lib.flatten_dict(a)
        ra = copy.deepcopy(a)
        try:
            lib.nested_update(ra, copy.deepcopy(b))
        except ValueError:
            ra = None
        return [_digest(flat), _digest(lib.nest_dict(flat)), None if ra is None else _digest(ra)]
    want = PINS("dict_helpers", lambda root: [helpers(ref_utils(root), a, b) for a, b in cases])
    for (a, b), w in zip(cases, want):
        got = helpers(OWN, a, b)
        assert got[:2] == w[:2], a
        assert (got[2] is None) == (w[2] is None)
        assert got[2] == w[2], (a, b)


def test_check_params_accepts_and_rejects_like_the_executed_reference():
    required = {"a": int, "mode": ["train", "eval"], "name": str, "fn": None}
    optional = {"x": float, "flag": bool, "kind": [None, "p", "q"], "anything": None}
    base = {"a": 1, "mode": "train", "name": "n", "fn": len}
    cases = [base, dict(base, x=0.5), dict(base, x=1), dict(base, flag=True), dict(base, flag=1), dict(base, kind="p"),
             dict(base, kind="z"), dict(base, kind=None), dict(base, anything=object()), dict(base, unknown=1),
             {k: v for k, v in base.items() if k != "a"}, dict(base, a="1"), dict(base, a=True), dict(base, mode="infer"),
             dict(base, name=3), dict(base, name=u"unicode")]
    def outcomes(lib):
        out = []
        for cfg in cases:
            try:
                lib.check_params(cfg, required, optional)
                out.append(None)
            except ValueError as e:
                out.append(str(e))
        return out
    want = PINS("check_params", lambda root: outcomes(ref_utils(root)))
    for cfg, r, o in zip(cases, want, outcomes(OWN)):
        assert (r is None) == (o is None), (cfg, r, o)
        if r is not None:
            assert r.split(" ")[0] == o.split(" ")[0] and r.split()[1:4] == o.split()[1:4], (r, o)
    assert PINS("check_params/no_rules", lambda root: ref_utils(root).check_params({"zzz": 1}, None, None) is None)
    assert OWN.check_params({"zzz": 1}, None, None) is None


def ast_parse(path):
    import ast
    return ast.parse(open(path).read())


def _reference_function(path, name):
    """Compile ONE top-level function of a reference module that cannot be imported as a whole (TensorFlow at import
    time) from its source in the reference checkout and return it; nothing is copied into the repository."""
    import ast
    tree = ast.parse(open(path).read())
    node = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == name)
    ns = {}
    exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    return ns[name]


def test_levenshtein_equals_the_executed_reference():
    """models/speech2text.py:51-71 (the distance behind the reference's WER) on random word and character
    sequences, next to the known answers of speech2text_test.py:229-256 that tests/test_compat_config.py holds."""
    import random
    from open_seq2seq.models.speech2text import levenshtein as own
    rnd = random.Random(1)
    words = ["the", "then", "seconds", "a", "cat", "sat", "on", "mat", ""]
    cases = []
    for _ in range(400):
        a = [rnd.choice(words) for _ in range(rnd.randint(0, 9))]
        b = [rnd.choice(words) for _ in range(rnd.randint(0, 9))]
        cases.append((a, b))

    def distances(fn):
        return [[fn(a, b), fn(" ".join(a), " ".join(b))] for a, b in cases]
    want = PINS("levenshtein", lambda root: distances(
        _reference_function(os.path.join(root, "open_seq2seq", "models", "speech2text.py"), "levenshtein")))
    for (a, b), w, o in zip(cases, want, distances(own)):
        assert w == o, (a, b)


def test_vocabulary_loader_equals_the_executed_reference(tmp_path, golden_dir):
    """data/utils.py:28-58 imported by path (it needs nothing beyond `six`): the toy vocabulary of the reference's
    tests and a word-level file with counts, empty lines and tabs."""
    from open_seq2seq.data.utils import load_pre_existing_vocabulary as own

    def reference(root):
        spec = importlib.util.spec_from_file_location("_reference_data_utils",
                                                      os.path.join(root, "open_seq2seq", "data", "utils.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod.load_pre_existing_vocabulary
    toy = os.path.join(golden_dir, "toy_speech_data", "vocab.txt")
    assert PINS("vocabulary/toy", lambda root: reference(root)(toy, read_chars=True)) == own(toy, read_chars=True)
    f = tmp_path / "words.txt"
    f.write_text(u"the\\t1234\\nof\\t99\\n\\nword with space\\t7\\nlast", encoding="utf-8")
    for kw in ({}, {"min_idx": 4}, {"read_chars": True}):
        want = PINS("vocabulary/words/%s" % sorted(kw.items()), lambda root: reference(root)(str(f), **kw))
        assert want == own(str(f), **kw), kw


@pytest.mark.parametrize("mode", ["train", "eval", "infer"])
def test_eval_shards_per_worker_equal_the_executed_reference(mode, golden_dir):
    """Speech2TextDataLayer.split_data (speech2text.py:200-210) compiled from the reference's source and run on a
    stand-in `self`: evaluation / inference shard the file list contiguously per worker, training does not."""
    import ast
    from open_seq2seq.data import Speech2TextDataLayer

    def split_data(root):
        src = open(os.path.join(root, "open_seq2seq", "data", "speech2text", "speech2text.py")).read()
        cls = next(n for n in ast.parse(src).body if isinstance(n, ast.ClassDef) and n.name == "Speech2TextDataLayer")
        fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "split_data")
        ns = {}
        exec(compile(ast.Module(body=[fn], type_ignores=[]), "speech2text.py", "exec"), ns)
        return ns["split_data"]
    toy = os.path.join(golden_dir, "toy_speech_data")
    for workers in (1, 2, 3, 4):
        seen = []
        for wid in range(workers):
            dl = Speech2TextDataLayer({"mode": mode, "batch_size": 1, "num_audio_features": 64, "input_type": "logfbank",
                                       "vocab_file": os.path.join(toy, "vocab.txt"), "shuffle": False,
                                       "dataset_files": [os.path.join(toy, "toy_data.csv")]}, None, workers, wid)
            all_rows = list(range(dl._all_size))
            me = types.SimpleNamespace(params={"mode": mode}, _num_workers=workers, _worker_id=wid)
            n_want = PINS("split_data/%s/%d/%d" % (mode, workers, wid), lambda root: len(split_data(root)(me, all_rows)))
            assert len(dl._files) == n_want, (mode, workers, wid)
            seen.append(n_want)
        if mode == "train":
            assert all(s == dl._all_size for s in seen)
        else:
            assert sum(seen) == dl._all_size


def _numpy_tf():
    """The five TensorFlow symbols optimizers/lr_policies.py touches, with TF 1.x's documented semantics on Python
    numbers (tf.train.polynomial_decay with cycle=False, exponential_decay, cosine_decay, cond, cast, maximum)."""
    import math
    tf = types.ModuleType("tensorflow")
    tf.float32 = "float32"
    tf.cast = lambda x, dtype: float(x)
    tf.cond = lambda pred, true_fn, false_fn, name=None: true_fn() if pred else false_fn()
    tf.maximum = max
    tf.train = types.SimpleNamespace()

    def polynomial_decay(learning_rate, global_step, decay_steps, end_learning_rate=0.0001, power=1.0, cycle=False):
        s = min(global_step, decay_steps)
        return (learning_rate - end_learning_rate) * (1.0 - s / float(decay_steps)) ** power + end_learning_rate

    def exponential_decay(learning_rate, global_step, decay_steps, decay_rate, staircase=False):
        p = global_step / float(decay_steps)
        return learning_rate * decay_rate ** (math.floor(p) if staircase else p)

    def cosine_decay(learning_rate, global_step, decay_steps, alpha=0.0):
        s = min(global_step, decay_steps)
        return learning_rate * ((1.0 - alpha) * 0.5 * (1.0 + math.cos(math.pi * s / float(decay_steps))) + alpha)
    tf.train.polynomial_decay, tf.train.exponential_decay, tf.train.cosine_decay = (
        polynomial_decay, exponential_decay, cosine_decay)
    return tf


def test_lr_policies_equal_the_executed_reference():
    """optimizers/lr_policies.py loaded by path over the stand-in above: the reference's own glue (warm-up, the
    begin_decay_at switch, how min_lr is handed to TF -- as `alpha`, a FRACTION, in cosine_decay) against the
    oracle's policies, which the device-side schedule of csrc/optim.cu is tested against."""
    from oracle import optimizer as OO

    def policies(root):
        tf = _numpy_tf()
        fake = {"tensorflow": tf, "tensorflow.python": types.ModuleType("tensorflow.python"),
            "tensorflow.python.framework": types.ModuleType("tensorflow.python.framework"),
            "tensorflow.python.framework.ops": types.ModuleType("tensorflow.python.framework.ops")}
        fake["tensorflow.python.framework"].ops = fake["tensorflow.python.framework.ops"]
        saved = {k: sys.modules.get(k) for k in fake}
        sys.modules.update(fake)
        try:
            spec = importlib.util.spec_from_file_location(
                "_reference_lr_policies", os.path.join(root, "open_seq2seq", "optimizers", "lr_policies.py"))
            ref = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(ref)
        finally:
            for k, v in saved.items():
                if v is None:
                    sys.modules.pop(k, None)
                else:
                    sys.modules[k] = v
        return ref
    steps = list(range(0, 40)) + [99, 100, 101, 499, 500, 501, 999, 1000, 1001, 5000]
    for kw in (dict(learning_rate=0.02, decay_steps=1000, power=2.0, min_lr=1e-5),                  # Jasper
               dict(learning_rate=0.05, decay_steps=1000, power=2.0),                               # w2l+
               dict(learning_rate=0.02, decay_steps=900, power=1.0, begin_decay_at=100, min_lr=1e-4, warmup_steps=30)):
        want = PINS("lr/poly_decay/%s" % sorted(kw.items()), lambda root: [policies(root).poly_decay(s, **kw) for s in steps])
        for s, w in zip(steps, want):
            assert abs(w - OO.poly_decay(s, **kw)) < 1e-12, (kw, s)
    for kw in (dict(learning_rate=0.01, decay_steps=1000, min_lr=0.0, warmup_steps=10),             # QuartzNet
               dict(learning_rate=0.01, decay_steps=800, min_lr=0.1, begin_decay_at=200, warmup_steps=20)):
        want = PINS("lr/cosine_decay/%s" % sorted(kw.items()),
                    lambda root: [policies(root).cosine_decay(s, **kw) for s in steps])
        for s, w in zip(steps, want):
            assert abs(w - OO.cosine_decay(s, **kw)) < 1e-12, (kw, s)
    for kw in (dict(learning_rate=0.1, decay_steps=100, decay_rate=0.5, use_staircase_decay=True, begin_decay_at=20,
                    min_lr=1e-3),
               dict(learning_rate=0.1, decay_steps=100, decay_rate=0.9, use_staircase_decay=False)):
        want = PINS("lr/exp_decay/%s" % sorted(kw.items()), lambda root: [policies(root).exp_decay(s, **kw) for s in steps])
        for s, w in zip(steps, want):
            assert abs(w - OO.exp_decay(s, **kw)) < 1e-12, (kw, s)
    assert PINS("lr/fixed_lr", lambda root: policies(root).fixed_lr(7, 0.3)) == OO.fixed_lr(7, 0.3)


def test_wer_accumulation_equals_the_executed_reference():
    """Speech2Text.evaluate / finalize_evaluation (models/speech2text.py:244-294) compiled from the reference's
    source and run on a stand-in `self` with tf.nn.ctc_greedy_decoder's SPARSE output; the drop-in model consumes the
    dense tokens + lengths that os2s_ctc_greedy writes.  Same per-batch (word errors, word count), same WER."""
    import ast
    import collections
    import random
    import numpy as np
    import torch
    from open_seq2seq.models.speech2text import Speech2Text

    def reference(root):
        path = os.path.join(root, "open_seq2seq", "models", "speech2text.py")
        tree = ast.parse(open(path).read())
        ns = {"deco_print": lambda *a, **k: None}
        for name in ("levenshtein", "sparse_tensor_to_chars"):
            ns[name] = _reference_function(path, name)
        cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "Speech2Text")
        for m in cls.body:
            if isinstance(m, ast.FunctionDef) and m.name in ("evaluate", "finalize_evaluation"):
                exec(compile(ast.Module(body=[m], type_ignores=[]), path, "exec"), ns)
        return ns
    chars = "abcdefghijklmnopqrstuvwxyz '"
    idx2char = dict(enumerate(chars))
    dl = types.SimpleNamespace(params={"idx2char": idx2char})
    own_self = types.SimpleNamespace(get_data_layer=lambda: dl)
    own_self._decode_batch = types.MethodType(Speech2Text._decode_batch, own_self)
    Sparse = collections.namedtuple("SparseTensorValue", "indices values dense_shape")
    rnd = random.Random(3)
    words = ["the", "then", "seconds", "a", "cat", "sat", "on", "mat"]
    r_inputs, o_batches = [], []
    for _ in range(12):
        B = rnd.randint(1, 5)
        truths = [" ".join(rnd.choice(words) for _ in range(rnd.randint(1, 8))) for _ in range(B)]
        preds = [" ".join(rnd.choice(words) for _ in range(rnd.randint(0, 8))) for _ in range(B)]
        enc = lambda s: [chars.index(c) for c in s]
        L = max(len(t) for t in truths)
        y = np.zeros((B, L), dtype=np.int32)
        ylen = np.array([len(t) for t in truths], dtype=np.int32)
        for b, t in enumerate(truths):
            y[b, :len(t)] = enc(t)
        P = max(1, max(len(p) for p in preds))
        toks = np.zeros((B, P), dtype=np.int32)
        tl = np.array([len(p) for p in preds], dtype=np.int32)
        idx, vals = [], []
        for b, p in enumerate(preds):
            toks[b, :len(p)] = enc(p)
            idx += [(b, t) for t in range(len(p))]
            vals += enc(p)
        iv = {"source_tensors": [np.zeros((B, 4, 2))], "target_tensors": [y, ylen]}
        r_inputs.append((iv, [Sparse(idx, vals, (B, P))]))
        o_iv = {"target_tensors": (torch.from_numpy(y), torch.from_numpy(ylen))}
        o_batches.append(Speech2Text.evaluate(own_self, o_iv, (torch.from_numpy(toks), torch.from_numpy(tl))))

    def evaluate(root):
        ns = reference(root)
        ref_self = types.SimpleNamespace(is_bpe=False, tensor_to_chars=ns["sparse_tensor_to_chars"],
                                         tensor_to_char_params={}, get_data_layer=lambda: dl)
        r_batches = [ns["evaluate"](ref_self, iv, out) for iv, out in r_inputs]
        return {"batches": r_batches, "final": ns["finalize_evaluation"](ref_self, r_batches)}
    want = PINS("wer", evaluate)
    for r, o in zip(want["batches"], o_batches):
        assert r == list(o)
    got = Speech2Text.finalize_evaluation(own_self, o_batches)
    assert want["final"].keys() == got.keys() and abs(want["final"]["Eval WER"] - got["Eval WER"]) < 1e-12


def test_larc_and_global_norm_clipping_equal_the_executed_reference(monkeypatch):
    """optimizers.py:289-480 (post_process_gradients: tf.clip_by_global_norm on the fp32 global norm, then LARC in
    'clip' or 'scale' mode) compiled from the reference's source over a NumPy stand-in for the dozen TF symbols it
    touches, vs oracle.optimizer.larc / clip_by_global_norm -- the functions the device optimizer is tested against."""
    import collections
    import collections.abc
    import contextlib
    import numpy as np
    import six
    from oracle import optimizer as OO
    monkeypatch.setattr(collections, "Sequence", collections.abc.Sequence, raising=False)   # (Python 2-era alias)

    class Var(np.ndarray):
        name = "v:0"
    tf = types.SimpleNamespace(
        float32=np.float32, int32=np.int32, IndexedSlices=type("IndexedSlices", (), {}),
        norm=lambda tensor=None, ord=2: np.float32(np.sqrt(np.sum(np.square(tensor, dtype=np.float32), dtype=np.float32))),
        cast=lambda x, dtype: np.asarray(x).astype(dtype), saturate_cast=lambda x, dtype: np.asarray(x).astype(dtype),
        maximum=np.maximum, minimum=np.minimum, less=np.less, identity=lambda x, name=None: x,
        convert_to_tensor=lambda x, name=None: np.asarray(x), ones=lambda shape, dtype=np.float32: np.ones(shape, dtype),
        global_norm=lambda ts: np.float32(np.sqrt(sum(np.sum(np.square(t, dtype=np.float32), dtype=np.float32)
                                                      for t in ts))),
        name_scope=lambda *a, **k: contextlib.nullcontext("clip"), colocate_with=lambda v: contextlib.nullcontext(),
        summary=types.SimpleNamespace(scalar=lambda *a, **k: None, histogram=lambda *a, **k: None))

    def post_process_gradients(root, *args):
        path = os.path.join(root, "open_seq2seq", "optimizers", "optimizers.py")
        tree = ast_parse(path)
        ns = {"tf": tf, "check_params": ref_utils(root).check_params, "mask_nans": None, "collections": collections,
              "six": six}
        for name in ("_global_norm_with_cast", "_clip_by_global_norm", "_clip_gradients_by_norm",
                     "post_process_gradients"):
            node = next(n for n in tree.body if getattr(n, "name", None) == name)
            exec(compile(__import__("ast").Module(body=[node], type_ignores=[]), path, "exec"), ns)
        return [np.asarray(g) for g, _ in ns["post_process_gradients"](*args)]
    rng = np.random.RandomState(0)
    shapes = [(11, 8, 16), (16,), (16,), (1, 8, 4), (40, 29), (29,)]
    for trial in range(6):
        ws = [(rng.standard_normal(s) * 0.1).astype(np.float32).view(Var) for s in shapes]
        gs = [(rng.standard_normal(s) * 10.0 ** rng.randint(-4, 2)).astype(np.float32) for s in shapes]
        lr = float(10.0 ** rng.uniform(-4, -1))
        for larc_params in ({"larc_eta": 0.001}, {"larc_eta": 0.002, "larc_mode": "scale", "min_update": 1e-6},
                            {"larc_eta": 0.001, "larc_mode": "clip", "epsilon": 1e-5}):
            want = PINS("larc/%d/%s" % (trial, sorted(larc_params.items())), lambda root: post_process_gradients(
                root, list(zip(gs, ws)), [], lr, None, dict(larc_params)), sample=8)
            kw = dict(larc_params)
            if "epsilon" in kw:
                kw["eps"] = kw.pop("epsilon")
            got = OO.larc(gs, [np.asarray(w) for w in ws], lr, **kw)
            for wg, g in zip(want, got):
                assert RP.close(g, wg, rtol=2e-6, atol=0), (trial, larc_params)
        for clip in (0.5, 5.0, 1e4):
            want = PINS("clip/%d/%s" % (trial, clip), lambda root: post_process_gradients(
                root, list(zip(gs, ws)), [], lr, clip, None), sample=8)
            got, gnorm = OO.clip_by_global_norm(gs, clip)
            for wg, g in zip(want, got):
                assert RP.close(g, wg, rtol=2e-6, atol=0), (trial, clip)
            if clip > gnorm:
                assert all(np.allclose(g, g0, rtol=1e-6) for g, g0 in zip(got, gs))       # below the threshold: untouched


def test_novograd_equals_the_executed_reference_class():
    """optimizers/novograd.py: the NovoGrad class body compiled from the reference's source on top of a stand-in
    tf.train.MomentumOptimizer with TensorFlow's documented update (accum <- momentum accum + grad; var <- var - lr
    accum).  In graph mode apply_gradients runs ONCE and the zero-initialised `nvgrad2_ema` variables are never
    assigned, so every step sees ema == 0 and normalises by the CURRENT ||g||^2 (the as-written behaviour the oracle
    and the device optimizer reproduce by default); the stand-in mirrors that by building the "graph" afresh per
    step.  Several steps, with and without weight decay / gradient averaging."""
    import ast
    import numpy as np
    from oracle import optimizer as OO

    class MomentumOptimizer(object):
        def __init__(self, learning_rate, momentum, use_locking=False, name="Momentum", use_nesterov=False):
            assert not use_nesterov
            self._lr, self._momentum, self.accum = learning_rate, momentum, {}

        def apply_gradients(self, grads_and_vars, global_step=None, name=None):
            for i, (g, v) in enumerate(grads_and_vars):
                a = self.accum.get(i)
                a = g.copy() if a is None else np.float32(self._momentum) * a + g
                self.accum[i] = a
                v -= np.float32(self._lr) * a

    tf = types.SimpleNamespace(
        float32=np.float32, get_variable=lambda name, shape, dtype, initializer, trainable: np.float32(0.0),
        keras=types.SimpleNamespace(initializers=types.SimpleNamespace(Zeros=lambda: None)),
        reduce_sum=lambda x: np.sum(x, dtype=np.float32), square=lambda x: np.square(x, dtype=np.float32),
        cast=lambda x, dtype: np.asarray(x).astype(dtype), equal=lambda a, b: a == b, sqrt=np.sqrt,
        cond=lambda pred, t, f: t() if pred else f())

    def novograd(root, w0, steps, lr, kw):
        path = os.path.join(root, "open_seq2seq", "optimizers", "novograd.py")
        cls = next(n for n in ast.parse(open(path).read()).body if isinstance(n, ast.ClassDef) and n.name == "NovoGrad")
        ns = {"tf": tf, "MomentumOptimizer": MomentumOptimizer}
        exec(compile(ast.Module(body=[cls], type_ignores=[]), path, "exec"), ns)
        w_ref = [w.copy() for w in w0]
        opt = ns["NovoGrad"](learning_rate=lr, **kw)
        out = []
        for gs in steps:
            opt._grads_ema = None                      # the graph is built once: ema reads as 0 on every run
            opt.apply_gradients([(g.copy(), w) for g, w in zip(gs, w_ref)])
            out.append([w.copy() for w in w_ref])
        return out
    rng = np.random.RandomState(2)
    shapes = [(5, 8, 16), (16,), (40, 29)]
    for kw in (dict(beta1=0.95, beta2=0.98, epsilon=1e-8, weight_decay=0.001),
               dict(beta1=0.9, beta2=0.5, epsilon=1e-6, weight_decay=0.0, grad_averaging=True)):
        lr = 0.02
        w0 = [(rng.standard_normal(s) * 0.1).astype(np.float32) for s in shapes]
        steps = [[(rng.standard_normal(s) * 0.05).astype(np.float32) for s in shapes] for _ in range(5)]
        want = PINS("novograd/%s" % sorted(kw.items()), lambda root: novograd(root, w0, steps, lr, kw), sample=8)
        w_own = [w.copy() for w in w0]
        state = OO.NovoGradState(len(shapes))
        for step, gs in enumerate(steps):
            OO.novograd_step(w_own, [g.copy() for g in gs], state, lr, **kw)
            for a, b in zip(want[step], w_own):
                assert RP.close(b, a, rtol=1e-5, atol=1e-7), (kw, step)


@pytest.mark.parametrize("dump", [False, True])
def test_inference_output_files_equal_the_executed_reference(tmp_path, dump):
    """Speech2Text.finalize_inference (models/speech2text.py:315-354) compiled from the reference's source: the CSV
    of predicted transcripts and, with `infer_logits_to_pickle`, the {logits, step_size, vocab} pickle that
    scripts/decode.py reads -- batches arrive in any order and are put back in dataset order."""
    import ast
    import pickle
    import numpy as np
    import pandas as pd
    from open_seq2seq.models.speech2text import Speech2Text
    files = ["a/%d.wav" % i for i in range(7)]
    idx2char = dict(enumerate("abcdefghijklmnopqrstuvwxyz '"))
    layers = [{"stride": [2]}, {"stride": [1]}, {"stride": [1]}]
    dl_ref = types.SimpleNamespace(all_files=np.array(files), params={"window_stride": 0.01, "idx2char": idx2char})
    dl_own = types.SimpleNamespace(_files=[(f, None) for f in files], params=dl_ref.params)
    enc = types.SimpleNamespace(params={"convnet_layers": layers})
    ref_self = types.SimpleNamespace(dump_outputs=dump, get_data_layer=lambda: dl_ref, encoder=enc)
    own_self = types.SimpleNamespace(dump_outputs=dump, get_data_layer=lambda: dl_own, encoder=enc)
    rng = np.random.RandomState(0)
    order = [np.array([4, 1]), np.array([6, 0, 3]), np.array([5, 2])]
    if dump:
        item = {i: rng.standard_normal((5 + i, 29)).astype(np.float32) for i in range(7)}
    else:
        item = {i: "text %d" % i for i in range(7)}
    batches = [([item[int(i)] for i in ids], [ids]) for ids in order]

    def summary(out):
        """The written file: the CSV text, or the pickle's keys, step size, vocabulary and logits (by digest)."""
        if not dump:
            return open(out).read()
        d = pickle.load(open(out, "rb"))
        return {"keys": sorted(d), "step_size": d["step_size"], "vocab": sorted(d["vocab"].items()),
                "files": list(d["logits"]), "logits": [RP.digest(d["logits"][f]) for f in d["logits"]]}

    def reference(root):
        path = os.path.join(root, "open_seq2seq", "models", "speech2text.py")
        cls = next(n for n in ast.parse(open(path).read()).body if isinstance(n, ast.ClassDef) and n.name == "Speech2Text")
        fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "finalize_inference")
        ns = {"np": np, "pd": pd, "pickle": pickle}
        exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
        if dump:
            # (the reference stacks equally long logits into one array; ragged lists need dtype=object in NumPy >= 1.24)
            orig = np.array
            ns["np"] = types.SimpleNamespace(array=lambda x: orig(x, dtype=object), hstack=np.hstack, argsort=np.argsort)
        a = str(tmp_path / "ref.out")
        ns["finalize_inference"](ref_self, batches, a)
        return summary(a)
    b = str(tmp_path / "own.out")
    Speech2Text.finalize_inference(own_self, batches, b)
    want, got = PINS("finalize_inference/dump=%s" % dump, reference), summary(b)
    if dump:
        assert want["keys"] == got["keys"] and abs(want["step_size"] - got["step_size"]) < 1e-12
        assert [list(kv) for kv in got["vocab"]] == want["vocab"]
        assert abs(want["step_size"] - 0.02) < 1e-12 and want["files"] == got["files"] == files
        assert want["logits"] == got["logits"]
    else:
        assert want == got
        assert pd.read_csv(b)["predicted_transcript"].tolist() == ["text %d" % i for i in range(7)]


def _reference_hooks(root):
    """RunEvaluationHook / PrintLossAndTimeHook / PrintSamplesHook (utils/hooks.py:57-245) compiled from the
    reference's source over a stand-in for the tf.train symbols they use; tf.train.SecondOrStepTimer is TensorFlow's
    (basic_session_run_hooks.py): first call fires, afterwards when step >= last_triggered + every_steps."""
    import ast
    import collections

    class SecondOrStepTimer(object):
        def __init__(self, every_secs=None, every_steps=None):
            self._every, self._last = every_steps, None

        def should_trigger_for_step(self, step):
            if self._last is None:
                return True
            if self._last == step:
                return False
            return step >= self._last + self._every

        def update_last_triggered_step(self, step):
            self._last = step
    train = types.SimpleNamespace(SessionRunHook=object, SecondOrStepTimer=SecondOrStepTimer,
                                  Saver=lambda **kw: types.SimpleNamespace(save=lambda *a, **k: None),
                                  get_global_step=lambda: "global_step",
                                  SessionRunArgs=lambda fetches: fetches)
    path = os.path.join(root, "open_seq2seq", "utils", "hooks.py")
    ns = {"tf": types.SimpleNamespace(train=train), "deco_print": lambda *a, **k: None, "time": __import__("time"),
          "math": __import__("math"), "os": os, "log_summaries_from_dict": lambda *a, **k: None}
    for node in ast.parse(open(path).read()).body:
        if isinstance(node, ast.ClassDef) and node.name in ("RunEvaluationHook", "PrintLossAndTimeHook",
                                                             "PrintSamplesHook"):
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    return ns, collections.namedtuple("RunValues", "results")


def _reference_hook_cadence(root, every, last_step, first, tmp_path):
    """The steps at which the reference's hooks evaluate, print the loss and print samples."""
    ns, RunValues = _reference_hooks(root)
    fired = {"eval": [], "loss": [], "samples": []}
    model = types.SimpleNamespace(
        params={"num_checkpoints": 2, "save_checkpoint_steps": None, "save_summaries_steps": None, "logdir": str(tmp_path)},
        on_horovod=False, loss="loss", steps_in_epoch=None, get_output_tensors=lambda i: "out",
        get_data_layer=lambda i=0: types.SimpleNamespace(input_tensors="in"),
        finalize_evaluation=lambda results, step: {},
        maybe_print_logs=lambda i, o, step: fired["samples"].append(int(step)))
    ns["get_results_for_epoch"] = lambda m, sess, mode, compute_loss: ([], 1.0)
    hooks = {"eval": ns["RunEvaluationHook"](every, model, last_step=last_step),
             "loss": ns["PrintLossAndTimeHook"](every, model), "samples": ns["PrintSamplesHook"](every, model)}
    for h in hooks.values():
        h.begin()
    ctx = types.SimpleNamespace(session=None)
    for k in range(first, last_step):
        req = {n: h.before_run(ctx) for n, h in hooks.items()}
        for n, h in hooks.items():
            wanted = req[n][0]
            res = [] if not wanted else ([1.0] if n == "loss" else ("in", "out"))
            before = len(fired["samples"])
            if n == "eval":
                calls = []
                ns["get_results_for_epoch"] = lambda m, sess, mode, compute_loss, c=calls: (c.append(1), ([], 1.0))[1]
                h.after_run(ctx, RunValues([res, k]))
                if calls:
                    fired["eval"].append(k)
            else:
                h.after_run(ctx, RunValues([res, k]))
                if n == "loss" and wanted:
                    fired["loss"].append(k)
            assert n != "samples" or len(fired["samples"]) - before == (1 if wanted else 0)
    return fired


@pytest.mark.parametrize("every,last_step,first", [(5, 12, 0), (4, 10, 0), (1, 3, 0), (7, 20, 0), (5, 23, 8)])
def test_hook_cadence_equals_the_executed_reference(every, last_step, first, tmp_path):
    """When evaluation, loss printing and sample printing fire: the reference's hooks driven the way
    MonitoredTrainingSession drives them (before_run -> run -> after_run with the global step the run started
    from) vs the drop-in's training loop on stub models, incl. a resumed run (first global step 8)."""
    import torch
    from open_seq2seq.utils import funcs as F
    fired = PINS("hooks/%d/%d/%d" % (every, last_step, first),
                 lambda root: _reference_hook_cadence(root, every, last_step, first, tmp_path))

    # the drop-in loop on stub models
    own = {"eval": [], "loss": [], "samples": []}

    class Eng(object):
        def __init__(self):
            self.istate = torch.zeros(8, dtype=torch.int64)
            self.istate[2] = first
            self.training = True

        def set_training(self, f):
            self.training = f

        def greedy_decode(self):
            return None
    eng = Eng()
    n_last = last_step

    class DL(object):
        def __init__(self, n):
            self.n, self.iterator = n, None
            self.build_graph()

        def build_graph(self):
            self.iterator = iter(range(10 ** 9)) if self.n is None else iter(range(self.n))

    class Train(object):
        on_horovod, hvd = False, None
        params = {"print_loss_steps": every, "print_samples_steps": every, "save_checkpoint_steps": None,
                  "eval_steps": every, "logdir": None, "bench_start": 0}
        last_step = n_last
        engine = eng
        _dl = DL(None)

        def get_data_layer(self):
            return self._dl

        def train_step(self, batch):
            self.engine.istate[2] += 1
            return torch.tensor(1.0), 1.0

        def maybe_print_logs(self, batch, toks, step):
            own["samples"].append(int(step))

    class Eval(object):
        on_horovod, hvd = False, None
        engine = eng
        _dl = DL(1)

        def get_data_layer(self):
            return self._dl

        def eval_step(self, batch):
            return torch.tensor(1.0), {"outputs": [None]}

        def evaluate(self, batch, out):
            return 0

        def finalize_evaluation(self, results):
            own["eval"].append(int(eng.istate[2]) - 1)       # the global step the triggering run started from
            return {}
    printed = []
    orig = F.deco_print
    F.deco_print = lambda line, *a, **k: printed.append(line)
    try:
        F.train(Train(), Eval())
    finally:
        F.deco_print = orig
    own["loss"] = [int(l.split()[2].rstrip(":")) for l in printed if l.startswith("Global step")]
    assert own == fired, (own, fired)
