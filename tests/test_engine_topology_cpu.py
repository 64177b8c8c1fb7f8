"""CPU tests of JasperEngine's host-side logic (no kernel runs: the 16-bit weight-copy launch is stubbed):
topology -> variables with the reference's names and shapes, zero-padded physical channel widths, the
folded stride-2 first layer, sep_conv1d split / composed modes, frozen pseudo-variables."""
import pytest
import torch

import openseq2seq_b200.engine as E
from tests.common_cfg import MINI_JASPER, MINI_QUARTZ


@pytest.fixture()
def cpu_engine(monkeypatch):
    monkeypatch.setattr(E.JasperEngine, "sync_half_copies", lambda self: None)

    def make(layers, F=64, V=29, **kw):
        return E.JasperEngine(layers, F, V, device="cpu", opt=kw.pop("opt", dict(loss_scaling=False)), **kw)
    return make


def test_variables_match_the_oracle_parameter_set(cpu_engine):
    from oracle import torch_twin as TT
    for layers in (MINI_JASPER, MINI_QUARTZ):
        eng = cpu_engine(layers)
        p = TT.init_params(layers, 64, 29, seed=0)
        names = dict(eng.named_parameters())
        assert set(names) == set(p)
        for n, v in names.items():
            assert tuple(v.shape) == tuple(p[n].shape), n
        eng.load_parameters(p)
        for n, v in eng.named_parameters():
            assert torch.equal(v, p[n].float()), n


def test_channel_widths_of_the_reference_toy_config_are_zero_padded(cpu_engine):
    """test_speech_configs/w2l_test_config.py: 40 features, 200 / 400 channels -> physical 128 / 256 / 512 with
    exact-zero pad channels (kernel rows / columns, BN gamma and beta), logical views for everything the
    reference names."""
    from oracle import torch_twin as TT
    layers = [{"type": "conv1d", "repeat": 3, "kernel_size": [7], "stride": [1], "num_channels": 200, "padding": "SAME",
               "dilation": [1]},
              {"type": "conv1d", "repeat": 1, "kernel_size": [1], "stride": [1], "num_channels": 400, "padding": "SAME",
               "dilation": [1]}]
    eng = cpu_engine(layers, F=40)
    assert (eng.Fp, eng.H, eng.Hl) == (128, 512, 400)
    assert [(l.lc_in, l.lc_out, l.c_in, l.c_out) for l in eng.layers] == [(40, 200, 128, 256), (200, 200, 256, 256),
                                                                        (200, 200, 256, 256), (200, 400, 256, 512)]
    p = TT.init_params(layers, 40, 29, seed=0)
    eng.load_parameters(p)
    assert sum(s["size"] for s in eng.specs) == sum(v.numel() for v in p.values())
    k = eng.by_name["conv11/kernel"]
    full = eng.master[k["offset"]:k["offset"] + k["store_size"]].view(*k["store_shape"])
    assert full.shape == (7, 128, 256) and float(full[:, 40:].abs().sum()) == 0 and float(full[:, :, 200:].abs().sum()) == 0
    g = eng.by_name["conv11/bn/gamma"]
    assert float(eng.master[g["offset"]:g["offset"] + g["store_size"]].sum()) == 200.0     # pad gammas are 0
    assert eng.moving["conv11/bn"].shape == (2, 256)


def test_jasper10x5_parameter_count_and_folded_first_layer(cpu_engine):
    import os
    import openseq2seq_b200.compat as compat
    compat.install()
    from open_seq2seq.utils.utils import get_base_config
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    _, cfg, _, _ = get_base_config(["--config_file=" + os.path.join(root, "configs", "jasper10x5_dr.py")])
    eng = cpu_engine(cfg["encoder_params"]["convnet_layers"])
    assert sum(s["size"] for s in eng.specs) == 332632349 and len(eng.named_parameters()) == 326
    l0 = eng.layers[0]
    assert l0.fold and (l0.kK, l0.kC_in, eng.Fp) == (6, 128, 64)
    v = eng.param_view("conv11/kernel")
    assert tuple(v.shape) == (11, 64, 256)
    # regularised variables: main conv kernels, BN gammas, the FC kernel -- not the 1x1 residual kernels
    eng.set_optimizer(l2_regularizer_scale=0.5, loss_scaling=False)
    reg = dict(zip([s["name"] for s in eng.specs], eng._reg.tolist()))
    assert reg["conv11/kernel"] == 0.5 and reg["conv25/res_bn_0/gamma"] == 0.5 and reg["fc/kernel"] == 0.5
    assert reg["conv25/res_0/kernel"] == 0.0 and reg["conv11/bn/beta"] == 0.0


def test_sep_conv_modes_and_frozen_pseudo_variables(cpu_engine):
    eng = cpu_engine(MINI_QUARTZ, opt=dict(loss_scaling=False, freeze_variables_regex="ForwardPass/w2l_encoder/conv2.*"))
    assert [(l.sep, l.sep_mode) for l in eng.layers][:2] == [(True, "compose"), (True, "split")]
    assert eng.layers[-2].sep_mode == "compose" and not eng.layers[-1].sep
    composed = [s["name"] for s in eng.specs if s["name"].endswith("@composed")]
    assert "conv11/kernel@composed" in composed and "conv22/res/kernel@composed" in composed
    frozen = {s["name"] for s, f in zip(eng.specs, eng._frozen.tolist()) if f}
    assert set(composed) <= frozen
    assert "conv21/depthwise_kernel" in frozen and "conv31/depthwise_kernel" not in frozen
    assert eng.frozen_names and all(n.startswith("conv2") for n in eng.frozen_names)
    assert eng.layers[1].wname == "conv21/pointwise_kernel" and eng.res_wname(eng.layers[2], 0) == "conv22/res/kernel@composed"
    with pytest.raises(AttributeError):
        cpu_engine(MINI_JASPER, opt=dict(max_grad_norm=1.0, larc_eta=0.001))


def test_gradient_buckets_tile_the_flat_buffer_and_split_into_aligned_rank_slices(cpu_engine):
    """Host side of the peer-memory gradient exchange (csrc/peer.cu): the buckets are cut at layer boundaries,
    last layer first, and cover the flat gradient buffer exactly once; the rank slices of a bucket are 16-byte
    aligned, disjoint and cover it (empty slices for tiny buckets)."""
    from openseq2seq_b200.dist import split_bucket
    for layers in (MINI_JASPER, MINI_QUARTZ):
        eng = cpu_engine(layers)
        eng.bucket_bytes = 64 << 10
        b = eng.grad_buckets()
        assert len(b) > 1 and b[0][1] == eng._total and b[-1][0] == 0
        for (s0, e0), (s1, e1) in zip(b[:-1], b[1:]):
            assert e1 == s0 and s1 < e1
        assert all(s % 4 == 0 for s, _ in b)
        firsts = {eng.layer_first_offset(li) for li in range(len(eng.layers))}
        assert all(s in firsts for s, _ in b)
    for world in (2, 3, 4, 8, 16):
        for (s, e) in ((0, 67), (128, 128 + 4 * (4 * world + 3)), (1000, 1000 + 33554432), (64, 64)):
            sl = split_bucket(s, e, world)
            assert len(sl) == world and sl[0][0] == s and sl[-1][1] == e
            for r in range(world):
                lo, hi = sl[r]
                assert lo <= hi and (lo == hi or (lo - s) % 4 == 0)
                if r:
                    assert lo == sl[r - 1][1]


@pytest.mark.parametrize("name,layers,params,sep", [
    ("jasper10x5_LibriSpeech_nvgrad_masks.py", 53, 332632349, False),   # (same encoder as ..._nvgrad.py)
    ("jasper-Mini-for-Jetson.py", 33, 8192733, True),
    ("quartznet15x5_LibriSpeech.py", 78, 19193949, True),
    ("w2l_large_8gpus.py", 17, 105774877, False),
    ("w2l_large_8gpus_mp.py", 17, 105774877, False),
    ("w2lplus_large_8gpus.py", 18, 106496285, False),
    ("w2lplus_large_8gpus_mp.py", 18, 106496285, False),
])
def test_every_tdnn_example_config_of_the_reference_builds_an_engine(cpu_engine, name, layers, params, sep, tmp_path):
    """All TDNNEncoder configs under example_configs/speech2text load unchanged through the compat package and
    their encoder params (activation, normalisation, initializer, conv / sep_conv layers, residual topologies,
    channel widths) map onto a JasperEngine: number of trainable variables as a regression value."""
    from open_seq2seq.encoders import TDNNEncoder
    from open_seq2seq.utils.utils import get_base_config
    from tests.refpins import example_config
    _, cfg, model, _ = get_base_config(["--config_file=" + example_config(name, tmp_path), "--mode=train"])
    assert model.__name__ == "Speech2Text" and cfg["encoder"] is TDNNEncoder
    kw = TDNNEncoder(dict(cfg["encoder_params"]), None, mode="train").engine_kwargs()
    nf = cfg.get("data_layer_params", {}).get("num_audio_features", 64)
    eng = E.JasperEngine(num_features=nf, vocab_size=29, device="cpu", opt=dict(loss_scaling=False), **kw)
    assert len(eng.layers) == layers and any(l.sep for l in eng.layers) == sep
    # (QuartzNet 15x5: 19.2 M variables incl. BN -- the paper quotes 18.9 M)
    assert sum(v.numel() for _, v in eng.named_parameters()) == params
