"""The reference's OWN encoder code, executed and stored, against the oracle (CPU tests).

`TDNNEncoder._encode` (encoders/tdnn_encoder.py:87-265) and `conv_bn_actv / conv_bn_res_bn_actv`
(parts/cnns/conv_blocks.py:61-232) are graph BUILDERS: every number they produce comes from a handful of TensorFlow
symbols.  Here those symbols are an EAGER stand-in on torch-CPU tensors (class `EagerTF` below: `tf.layers.conv1d`,
`tf.layers.separable_conv1d`, `tf.layers.batch_normalization`, `tf.sequence_mask`, `expand_dims / squeeze /
transpose / reduce_max / mod / constant`, `tf.nn.dropout`) written from TensorFlow 1.x's documented semantics
(SAME padding `out = ceil(T / s)`, `pad = max((out - 1) s + (K - 1) d + 1 - T, 0)`, the smaller half on the left;
training-mode batch normalisation over every axis but the channel axis, biased variance; depth multiplier 1), with
the variables looked up BY THE NAME TensorFlow would give them.  The reference's own source, loaded by path / compiled
from a checkout of it (never copied), then builds the encoder: which layer is called with which input, in which
order, where the masks are applied and refreshed, how the lengths shrink, which residual sources feed which block
through which 1x1 convolution and batch norm, under which variable names.  The oracle (`oracle/torch_twin.py`
tdnn_encode -- what every GPU parity test compares with, and whose variable set the engine reproduces) must give the
same output, the same lengths, and use exactly the same variables.  The reference's outputs are stored under
tests/golden/reference/reference_encoder.json (tests/refpins.py; OS2S_REFERENCE_ROOT re-runs the reference and
rewrites them).
"""
import ast
import importlib.util
import math
import os
import sys
import types

import pytest
import torch
import torch.nn.functional as F

from oracle import torch_twin as TT
from tests import refpins as RP
from tests.common_cfg import MINI_JASPER, MINI_QUARTZ

PINS = RP.Pins("reference_encoder")


class EagerTF(object):
    """The TensorFlow symbols the TDNN encoder path touches, eager on torch tensors."""
    float32 = torch.float32

    def __init__(self, params):
        self.params = params
        self.used = []
        self.layers = types.SimpleNamespace(conv1d=self.conv1d, separable_conv1d=self.separable_conv1d,
                                            conv2d=None, batch_normalization=self.batch_normalization)
        self.nn = types.SimpleNamespace(dropout=self.dropout, relu=torch.relu)

    def var(self, name, shape):
        w = self.params[name]
        assert tuple(w.shape) == tuple(shape), (name, tuple(w.shape), tuple(shape))
        self.used.append(name)
        return w

    @staticmethod
    def _one(v):
        return int(v[0]) if isinstance(v, (list, tuple)) else int(v)

    @staticmethod
    def _same_pad(T, K, s, d):
        out = int(math.ceil(T / float(s)))
        total = max((out - 1) * s + (K - 1) * d + 1 - T, 0)
        return total // 2, total - total // 2

    def _pad(self, x, K, s, d, padding):
        if padding.upper() == "SAME":
            pl, pr = self._same_pad(x.shape[1], K, s, d)
            return F.pad(x.transpose(1, 2), (pl, pr))
        return x.transpose(1, 2)

    def conv1d(self, inputs, filters, kernel_size, strides=1, padding="valid", data_format="channels_last",
               dilation_rate=1, use_bias=True, kernel_regularizer=None, name=None):
        assert not use_bias and data_format == "channels_last" and name
        K, s, d = self._one(kernel_size), self._one(strides), self._one(dilation_rate)
        w = self.var(name + "/kernel", (K, inputs.shape[2], filters))
        y = F.conv1d(self._pad(inputs, K, s, d, padding), w.permute(2, 1, 0), stride=s, dilation=d)
        return y.transpose(1, 2)

    def separable_conv1d(self, inputs, filters, kernel_size, strides=1, padding="valid", data_format="channels_last",
                         dilation_rate=1, use_bias=True, depthwise_regularizer=None, pointwise_regularizer=None,
                         name=None):
        assert not use_bias and data_format == "channels_last" and name
        K, s, d = self._one(kernel_size), self._one(strides), self._one(dilation_rate)
        C = inputs.shape[2]
        dw = self.var(name + "/depthwise_kernel", (K, C, 1))
        pw = self.var(name + "/pointwise_kernel", (1, C, filters))
        z = F.conv1d(self._pad(inputs, K, s, d, padding), dw.permute(1, 2, 0), stride=s, dilation=d, groups=C)
        return F.conv1d(z, pw.permute(2, 1, 0)).transpose(1, 2)

    def batch_normalization(self, inputs, axis=-1, momentum=0.99, epsilon=1e-3, training=False, name=None,
                            gamma_regularizer=None):
        assert training and axis == -1 and name
        C = inputs.shape[-1]
        gamma, beta = self.var(name + "/gamma", (C,)), self.var(name + "/beta", (C,))
        dims = tuple(range(inputs.dim() - 1))
        mean = inputs.mean(dim=dims)
        var = inputs.var(dim=dims, unbiased=False)
        return (inputs - mean) * torch.rsqrt(var + epsilon) * gamma + beta

    @staticmethod
    def dropout(x, keep_prob):
        assert keep_prob == 1.0, "the comparison runs without dropout"
        return x

    @staticmethod
    def sequence_mask(lengths, maxlen, dtype):
        return (torch.arange(int(maxlen))[None, :] < lengths[:, None]).to(dtype)

    expand_dims = staticmethod(lambda x, axis: x.unsqueeze(axis))
    squeeze = staticmethod(lambda x, axis: x.squeeze(axis))
    transpose = staticmethod(lambda x, perm: x.permute(*perm))
    reduce_max = staticmethod(lambda x: int(x.max()))
    mod = staticmethod(lambda a, b: a % b)
    constant = staticmethod(lambda v: v)


def _reference_encoder(root, tf):
    """conv_blocks.py loaded by path with `tensorflow` = the eager stand-in, then TDNNEncoder._encode compiled from
    its source into a namespace that holds those block functions."""
    pk = {n: types.ModuleType(n) for n in ("_refpkg", "_refpkg.parts", "_refpkg.parts.cnns", "_refpkg.parts.cnns.tcn")}
    for m in pk.values():
        m.__path__ = []
    pk["_refpkg.parts.cnns.tcn"].tcn = None
    tfm = types.ModuleType("tensorflow")
    tfm.layers = tf.layers
    stand = dict(pk, tensorflow=tfm)
    saved = {k: sys.modules.get(k) for k in stand}
    sys.modules.update(stand)
    try:
        spec = importlib.util.spec_from_file_location("_refpkg.parts.cnns.conv_blocks",
                                                      os.path.join(root, "open_seq2seq/parts/cnns/conv_blocks.py"))
        blocks = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(blocks)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    blocks.tf = tf                       # expand_dims / squeeze / layers inside the block functions

    class Speech2TextDataLayer(object):
        def __init__(self, params):
            self.params = params
    path = os.path.join(root, "open_seq2seq/encoders/tdnn_encoder.py")
    cls = next(n for n in ast.parse(open(path).read()).body if isinstance(n, ast.ClassDef) and n.name == "TDNNEncoder")
    fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "_encode")
    ns = {"tf": tf, "Speech2TextDataLayer": Speech2TextDataLayer}
    for name in ("conv_actv", "conv_bn_actv", "conv_ln_actv", "conv_in_actv", "conv_bn_res_bn_actv"):
        ns[name] = getattr(blocks, name)
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
    return ns["_encode"], Speech2TextDataLayer


PLAIN_RESIDUAL = [
    {"type": "conv1d", "repeat": 1, "kernel_size": [11], "stride": [2], "num_channels": 32, "padding": "SAME",
     "dilation": [1]},
    {"type": "conv1d", "repeat": 3, "kernel_size": [7], "stride": [1], "num_channels": 48, "padding": "SAME",
     "dilation": [1], "residual": True},
    {"type": "conv1d", "repeat": 2, "kernel_size": [4], "stride": [1], "num_channels": 40, "padding": "SAME",
     "dilation": [3], "residual": True},
    {"type": "conv1d", "repeat": 1, "kernel_size": [1], "stride": [1], "num_channels": 24, "padding": "SAME",
     "dilation": [1]},
]


@pytest.mark.parametrize("name,layers", [("dense residual (Jasper DR)", MINI_JASPER),
                                         ("separable (QuartzNet)", MINI_QUARTZ),
                                         ("plain residual, even kernel, dilation 3", PLAIN_RESIDUAL)])
@pytest.mark.parametrize("use_conv_mask", [True, False])
def test_oracle_encoder_equals_the_executed_reference_encoder(name, layers, use_conv_mask):
    torch.manual_seed(0)
    F_in, V = 64, 29
    layers = [dict(l, dropout_keep_prob=1.0) for l in layers]      # (dropout is tested with given masks elsewhere)
    params = {k: v.double() for k, v in TT.init_params(layers, F_in, V, seed=3).items()}
    for k in params:                     # non-trivial affine parameters everywhere
        if k.endswith("/gamma"):
            params[k] = 1.0 + 0.3 * torch.randn_like(params[k])
        elif k.endswith("/beta"):
            params[k] = 0.2 * torch.randn_like(params[k])
    for lens in ([96, 77, 50, 9], [92, 92, 61, 33]):          # max length on / off the pad_to = 16 grid
        lens_t = torch.tensor(lens, dtype=torch.int64)
        T = -(-max(lens) // 16) * 16
        x = torch.randn(len(lens), T, F_in, dtype=torch.float64)
        x = x * TT.sequence_mask(lens_t, T, x.dtype)         # the data layer pads with zeros

        def reference(root):
            tf = EagerTF(params)
            encode, DataLayer = _reference_encoder(root, tf)
            me = types.SimpleNamespace(
                params={"convnet_layers": layers, "dropout_keep_prob": 1.0, "activation_fn": torch.relu,
                        "use_conv_mask": use_conv_mask, "data_format": "channels_last", "normalization": "batch_norm",
                        "bn_momentum": 0.9, "bn_epsilon": 1e-3},
                _mode="train",
                _model=types.SimpleNamespace(get_data_layer=lambda: DataLayer({"backend": "librosa", "pad_to": 16})))
            want = encode(me, {"source_tensors": [x, lens_t.clone()]})
            return {"src_length": want["src_length"], "outputs": want["outputs"], "used": sorted(tf.used)}
        want = PINS("encoder/%s/mask=%s/%s" % (name, use_conv_mask, lens), reference)
        got, got_len = TT.tdnn_encode(x, lens_t, layers, params, training=True, bn_eps=1e-3,
                                      use_conv_mask=use_conv_mask)
        assert RP.equal(got_len, want["src_length"]), name
        assert want["outputs"].shape == tuple(got.shape)
        err = RP.max_dev(got, want["outputs"]) / want["outputs"].absmax
        assert err < 1e-10, (name, lens, err)
        # exactly the encoder's variables were read, each once, under TensorFlow's names
        enc_vars = sorted(k for k in params if not k.startswith("fc/"))
        assert want["used"] == enc_vars, (set(enc_vars) ^ set(want["used"]))


def _compile_from(path, cls_name, fn_name, ns):
    tree = ast.parse(open(path).read())
    body = tree.body
    if cls_name:
        body = next(n for n in body if isinstance(n, ast.ClassDef) and n.name == cls_name).body
    fn = next(n for n in body if isinstance(n, ast.FunctionDef) and n.name == fn_name)
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
    return ns[fn_name]


class EagerTFHead(EagerTF):
    """+ the symbols of the FC decoder (decoders/fc_decoders.py:105-158) and of the CTC loss (losses/ctc_loss.py:
    12-89, utils/utils.py:366-370): tf.layers.dense, reshape, where / gather_nd / shape / SparseTensor, tf.nn.ctc_loss
    (blank = last class, softmax inside, per-utterance negative log-likelihood; TF 1.x documentation), zeros_like /
    is_finite / reduce_mean."""
    int64 = torch.int64

    def __init__(self, params, alias):
        super(EagerTFHead, self).__init__(params)
        self.alias = alias
        self.layers.dense = self.dense
        self.nn.ctc_loss = self.ctc_loss

    def dense(self, inputs, units, kernel_regularizer=None, name=None):
        base = self.alias.get(name, name)
        w = self.var(base + "/kernel", (inputs.shape[1], units))
        return inputs @ w + self.var(base + "/bias", (units,))

    reshape = staticmethod(lambda x, shape, name=None: x.reshape(*shape))
    zeros_like = staticmethod(torch.zeros_like)
    is_finite = staticmethod(torch.isfinite)
    reduce_mean = staticmethod(lambda x: x.mean())
    gather_nd = staticmethod(lambda t, idx: t[tuple(idx.t())])
    shape = staticmethod(lambda t, out_type=None: torch.tensor(t.shape))
    SparseTensor = staticmethod(lambda indices, values, shape: types.SimpleNamespace(indices=indices, values=values,
                                                                                   dense_shape=shape))

    @staticmethod
    def sequence_mask(lengths, maxlen=None, dtype=torch.bool):
        maxlen = int(lengths.max()) if maxlen is None else int(maxlen)
        return (torch.arange(maxlen)[None, :] < lengths[:, None]).to(dtype)

    @staticmethod
    def where(cond, x=None, y=None):
        return torch.nonzero(cond) if x is None else torch.where(cond, x, y)

    @staticmethod
    def ctc_loss(labels, inputs, sequence_length, ignore_longer_outputs_than_inputs=False):
        B = int(labels.dense_shape[0])
        lens = torch.bincount(labels.indices[:, 0], minlength=B)
        lp = F.log_softmax(inputs, dim=2)
        return F.ctc_loss(lp, labels.values, sequence_length, lens, blank=inputs.shape[2] - 1, reduction="none",
                          zero_infinity=ignore_longer_outputs_than_inputs)


@pytest.mark.parametrize("layers", [MINI_JASPER, MINI_QUARTZ], ids=["jasper", "quartznet"])
def test_oracle_forward_loss_equals_the_executed_reference_encoder_decoder_and_loss(layers, monkeypatch):
    """encoder -> FullyConnectedTimeDecoder._decode -> CTCLoss._compute_loss, all three compiled from the reference's
    source over the eager stand-in, vs oracle.torch_twin.forward_loss: logits (time-major) and the batch-mean loss,
    incl. an utterance whose transcript does not fit its input (ignore_longer_outputs_than_inputs + mask_nans)."""
    torch.manual_seed(1)
    F_in, V = 64, 29
    layers = [dict(l, dropout_keep_prob=1.0) for l in layers]
    params = {k: v.double() for k, v in TT.init_params(layers, F_in, V, seed=5).items()}
    lens_t = torch.tensor([96, 70, 41, 12], dtype=torch.int64)
    x = torch.randn(4, 96, F_in, dtype=torch.float64) * TT.sequence_mask(lens_t, 96, torch.float64)
    y_len = torch.tensor([11, 9, 5, 9], dtype=torch.int64)        # the last one does not fit 12 / 2 = 6 frames
    y = torch.zeros(4, 11, dtype=torch.int64)
    for b in range(4):
        y[b, :y_len[b]] = torch.randint(0, V - 1, (int(y_len[b]),))

    def reference(root):
        tf = EagerTFHead(params, {"fully_connected": "fc"})
        encode, DataLayer = _reference_encoder(root, tf)
        monkeypatch.setattr(torch.Tensor, "get_shape", lambda t: types.SimpleNamespace(as_list=lambda: list(t.shape)),
                            raising=False)
        me = types.SimpleNamespace(
            params={"convnet_layers": layers, "dropout_keep_prob": 1.0, "activation_fn": torch.relu,
                    "use_conv_mask": True, "data_format": "channels_last", "normalization": "batch_norm",
                    "bn_momentum": 0.9, "bn_epsilon": 1e-3, "tgt_vocab_size": V},
            _mode="train", _mask_nan=True,
            _model=types.SimpleNamespace(get_data_layer=lambda: DataLayer({"backend": "librosa", "pad_to": 16})))
        enc = encode(me, {"source_tensors": [x, lens_t.clone()]})
        src = os.path.join(root, "open_seq2seq")
        decode = _compile_from(os.path.join(src, "decoders/fc_decoders.py"), "FullyConnectedTimeDecoder", "_decode",
                               {"tf": tf})
        dec = decode(me, {"encoder_output": enc})
        ns = {"tf": tf}
        _compile_from(os.path.join(src, "utils/utils.py"), None, "mask_nans", ns)
        _compile_from(os.path.join(src, "losses/ctc_loss.py"), None, "dense_to_sparse", ns)
        compute = _compile_from(os.path.join(src, "losses/ctc_loss.py"), "CTCLoss", "_compute_loss", ns)
        loss = compute(me, {"decoder_output": dec, "target_tensors": [y, y_len]})
        return {"src_length": dec["src_length"], "logits": dec["logits"], "loss": float(loss), "used": sorted(tf.used)}
    want = PINS("forward_loss/%d_layers" % len(layers), reference)
    got, logits, out_len = TT.forward_loss(params, layers, x, lens_t, y, y_len, training=True)
    assert RP.equal(out_len, want["src_length"])
    assert want["logits"].shape == tuple(logits.shape)              # [T', B, V]
    assert RP.max_dev(logits, want["logits"]) / want["logits"].absmax < 1e-10
    assert abs(want["loss"] - float(got)) < 1e-4 * abs(want["loss"])  # (the twin evaluates the CTC lattice in fp32)
    assert want["used"] == sorted(params)
