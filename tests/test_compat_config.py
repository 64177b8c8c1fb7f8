"""CPU tests of the drop-in boundary at the Python level: reference-style configs load through the
`open_seq2seq` / `tensorflow` compat surface, params dicts are validated with the reference's rules,
and the plugin classes can be constructed (no GPU work happens before compile())."""
import copy
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
import openseq2seq_b200.compat as compat  # noqa: E402

compat.install()

from open_seq2seq.utils.utils import (check_params, flatten_dict, get_base_config, nest_dict,  # noqa: E402
                                      nested_update)
from tests.refpins import example_config  # noqa: E402

OWN_CFG = os.path.join(ROOT, "configs", "jasper10x5_dr.py")


def test_own_jasper_config_loads_with_cli_overrides():
    args, cfg, model_cls, module = get_base_config([
        "--config_file=" + OWN_CFG, "--mode=train", "--batch_size_per_gpu=4",
        "--lr_policy_params/learning_rate=0.5", "--data_layer_params/dither=0.0", "--use_horovod=False"])
    assert model_cls.__name__ == "Speech2Text"
    assert cfg["batch_size_per_gpu"] == 4 and cfg["lr_policy_params"]["learning_rate"] == 0.5
    assert cfg["data_layer_params"]["dither"] == 0.0 and cfg["use_horovod"] is False
    layers = cfg["encoder_params"]["convnet_layers"]
    assert len(layers) == 13 and sum(l["repeat"] for l in layers) == 53
    assert args.mode == "train"


def test_reference_jasper_config_loads_unchanged_and_matches_own_config(tmp_path):
    ref_cfg = example_config("jasper10x5_LibriSpeech_nvgrad.py", tmp_path)
    _, ref, ref_model, ref_mod = get_base_config(["--config_file=" + ref_cfg, "--mode=train"])
    _, own, own_model, own_mod = get_base_config(["--config_file=" + OWN_CFG, "--mode=train"])
    assert ref_model.__name__ == own_model.__name__ == "Speech2Text"
    assert ref["encoder_params"]["convnet_layers"] == own["encoder_params"]["convnet_layers"]
    for key in ("optimizer_params", "lr_policy_params", "larc_params", "dtype", "loss_scaling",
                "batch_size_per_gpu", "num_epochs", "iter_size"):
        assert ref[key] == own[key], key
    assert ref["optimizer"].__name__ == own["optimizer"].__name__ == "NovoGrad"
    skip = {"vocab_file"}
    for k, v in ref["data_layer_params"].items():
        if k not in skip:
            assert own["data_layer_params"][k] == v, k
    for k in ("dropout_keep_prob", "normalization", "data_format", "use_conv_mask", "initializer_params"):
        assert ref["encoder_params"][k] == own["encoder_params"][k]
    assert ref_mod["train_params"]["data_layer_params"]["max_duration"] == 16.7


@pytest.mark.parametrize("name", ["jasper10x5_LibriSpeech_nvgrad.py", "jasper10x5_LibriSpeech_nvgrad_masks.py",
                                  "w2lplus_large_8gpus_mp.py", "jasper-Mini-for-Jetson.py"])
def test_other_reference_speech_configs_import_through_the_shim(name, tmp_path):
    from tests.refpins import config_imports, import_names
    imports = config_imports(name)
    bound = import_names(imports)          # every name the config imports resolves through the drop-in packages
    assert "Speech2Text" in bound and len(bound) == len(imports)
    path = example_config(name, tmp_path)
    _, cfg, model, mod = get_base_config(["--config_file=" + path, "--mode=train"])
    assert model.__name__ == "Speech2Text" and "convnet_layers" in cfg["encoder_params"]
    assert all(mod[k] is v for k, v in bound.items())


def test_check_params_rules_and_errors():
    check_params({"a": 1, "b": "x"}, {"a": int}, {"b": str})
    with pytest.raises(ValueError, match="has to be specified"):
        check_params({}, {"a": int}, {})
    with pytest.raises(ValueError, match="has to be of type"):
        check_params({"a": "1"}, {"a": int}, {})
    with pytest.raises(ValueError, match="has to be one of"):
        check_params({"a": 3}, {"a": [1, 2]}, {})
    with pytest.raises(ValueError, match="Unknown parameter"):
        check_params({"a": 1, "zz": 2}, {"a": int}, {})
    check_params({"a": object()}, {"a": None}, {})  # None = any value


def test_flatten_nest_update_roundtrip():
    d = {"x": 1, "y": {"z": 2.5, "w": {"q": "s"}}, "skip": [1, 2]}
    flat = flatten_dict(d)
    assert flat == {"x": 1, "y/z": 2.5, "y/w/q": "s"}
    assert nest_dict(flat) == {"x": 1, "y": {"z": 2.5, "w": {"q": "s"}}}
    nested_update(d, {"y": {"z": 3.0}, "new": {"k": 1}})
    assert d["y"]["z"] == 3.0 and d["y"]["w"]["q"] == "s" and d["new"] == {"k": 1}
    with pytest.raises(ValueError):
        nested_update({"a": 1}, {"a": {"b": 2}})


def test_model_and_plugins_construct_without_gpu_and_validate_params():
    import copy
    _, cfg, model_cls, module = get_base_config(["--config_file=" + OWN_CFG, "--mode=train",
                                                 "--use_horovod=False"])
    cfg = copy.deepcopy(cfg)
    nested_update(cfg, copy.deepcopy(module["train_params"]))
    model = model_cls(params=cfg, mode="train", hvd=None)
    assert model.get_data_layer().params["tgt_vocab_size"] == 29
    assert model.decoder.params["tgt_vocab_size"] == 29
    assert model.last_step == 400 * (64 // 32)
    assert type(model.encoder).__name__ == "TDNNEncoder" and model.encoder.name == "w2l_encoder"
    kw = model.encoder.engine_kwargs()
    assert kw["use_conv_mask"] and kw["bn_momentum"] == 0.90 and kw["relu_clip"] == 0.0
    bad = copy.deepcopy(cfg)
    bad["encoder_params"]["no_such_param"] = 1
    with pytest.raises(ValueError, match="Unknown parameter"):
        model_cls(params=bad, mode="train", hvd=None)
    bad = copy.deepcopy(cfg)
    del bad["batch_size_per_gpu"]
    with pytest.raises(ValueError, match="has to be specified"):
        model_cls(params=bad, mode="train", hvd=None)


def test_activation_tracing_of_config_lambdas():
    import tensorflow as tf
    assert tf.resolve_activation(tf.nn.relu) == (1, 0.0)
    assert tf.resolve_activation(lambda x: tf.minimum(tf.nn.relu(x), 20.0)) == (1, 20.0)
    assert tf.resolve_activation(None) == (0, 0.0)


def test_optimizer_kwargs_from_jasper_params():
    from open_seq2seq.optimizers.optimizers import optimizer_engine_kwargs
    _, cfg, _, _ = get_base_config(["--config_file=" + OWN_CFG, "--mode=train"])
    kw = optimizer_engine_kwargs(cfg, last_step=1000)
    assert kw["algo"] == "novograd" and kw["beta1"] == 0.95 and kw["weight_decay"] == 0.001
    assert kw["larc_eta"] == 0.001 and kw["larc_mode"] == "clip"
    assert kw["decay_steps"] == 1000 and kw["power"] == 2.0 and kw["min_lr"] == 1e-5
    assert kw["loss_scaling"] is True


def test_optimizer_and_data_layer_kwargs_from_reference_w2lplus_config(tmp_path):
    """example_configs/speech2text/w2lplus_large_8gpus_mp.py unchanged: Momentum + poly_decay + LARC + an L2
    regulariser + the default (python_speech_features) feature backend all map onto built pieces."""
    from open_seq2seq.optimizers.optimizers import optimizer_engine_kwargs
    path = example_config("w2lplus_large_8gpus_mp.py", tmp_path)
    _, cfg, _, mod = get_base_config(["--config_file=" + path, "--mode=train"])
    kw = optimizer_engine_kwargs(cfg, last_step=2000)
    assert kw["algo"] == "momentum" and kw["momentum"] == 0.9
    assert kw["l2_regularizer_scale"] == cfg["regularizer_params"]["scale"] > 0
    assert kw["larc_eta"] == cfg["larc_params"]["larc_eta"] and kw["loss_scaling"] is True
    assert kw["iter_size"] == 1 and kw["decay_steps"] == 2000
    dl = mod["train_params"]["data_layer_params"]
    assert dl.get("backend", "psf") == "psf" and dl["input_type"] == "logfbank"
    widths = {l["num_channels"] for l in cfg["encoder_params"]["convnet_layers"]}
    assert all(w % 64 == 0 for w in widths)   # every layer is covered by the tensor-core tiles


def test_levenshtein_and_wer_known_answers():
    # known answers of the reference's own test (models/speech2text_test.py:229-256)
    from open_seq2seq.models.speech2text import levenshtein
    assert levenshtein("kitten", "sitting") == 3
    assert levenshtein("", "abc") == 3 and levenshtein("abc", "abc") == 0
    assert levenshtein("this is a test".split(), "this is test".split()) == 1
    assert levenshtein("hello world".split(), "world hello".split()) == 2


def test_benchmark_flag_rewrites_the_train_config_like_the_reference():
    """utils.py:846-865: --benchmark empties logdir (a str, so Model's params check still passes), drops
    num_epochs for max_steps = bench_steps and silences samples / summaries / checkpoints."""
    import argparse
    from open_seq2seq.models import Speech2Text
    from open_seq2seq.utils.utils import adjust_for_benchmark
    _, cfg, _, mod = get_base_config(["--config_file=" + OWN_CFG, "--mode=train"])
    train_cfg = copy.deepcopy(cfg)
    nested_update(train_cfg, copy.deepcopy(mod["train_params"]))
    adjust_for_benchmark(train_cfg, argparse.Namespace(bench_steps=30, bench_start=None))
    assert train_cfg["logdir"] == "" and train_cfg["max_steps"] == 30 and "num_epochs" not in train_cfg
    assert train_cfg["bench_start"] == 10 and train_cfg["save_checkpoint_steps"] is None
    assert train_cfg["data_layer_params"]["shuffle"] is False
    check_params(train_cfg, Speech2Text.get_required_params(), Speech2Text.get_optional_params())


def test_nothing_in_the_headline_config_is_silently_ignored(tmp_path):
    """The reference's jasper10x5_LibriSpeech_nvgrad.py trains with speed perturbation (train_params
    augmentation :199-201); accepted-but-unimplemented options must raise, implemented ones must reach the
    engine / data layer."""
    import numpy as np
    from open_seq2seq.data import Speech2TextDataLayer
    from open_seq2seq.optimizers.optimizers import optimizer_engine_kwargs
    from open_seq2seq.utils.utils import resolve_initializer
    import tensorflow as tf
    _, cfg, _, mod = get_base_config(["--config_file=" + OWN_CFG])
    aug = mod["train_params"]["data_layer_params"]["augmentation"]
    assert aug == {"speed_perturbation_ratio": [0.9, 1.0, 1.1]}
    _, _, _, ref_mod = get_base_config(["--config_file=" + example_config("jasper10x5_LibriSpeech_nvgrad.py", tmp_path)])
    assert ref_mod["train_params"]["data_layer_params"]["augmentation"] == aug
    base = dict(cfg["data_layer_params"], mode="train", batch_size=2, dataset_files=["synthetic:4:1.0"])
    dl = Speech2TextDataLayer(dict(base, augmentation=dict(aug, noise_level_min=-90, noise_level_max=-46)), None, 1, 0)
    rs = np.random.RandomState(0)
    sr_new, noise, n_out = dl._draw_augmentation([16000] * 64, rs)
    assert set(sr_new.tolist()) == {14400, 16000, 17600}
    assert all(int(n) == int(16000 * (s / 16000.0)) for n, s in zip(n_out, sr_new))
    assert (noise >= 10 ** (-90 / 20.0)).all() and (noise < 10 ** (-46 / 20.0)).all()
    # the draws of the reference's own augment_audio_signal, executed in the build container (fixture written by
    # tools/make_golden_reference_draws.py): the data layer's host-side draws reproduce them seed by seed
    import json
    fx = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                                     "reference_augmentation_draws.json")))
    for case in fx["cases"]:
        dlc = Speech2TextDataLayer(dict(base, augmentation=case["augmentation"]), None, 1, 0)
        sr_c, noise_c, n_c = dlc._draw_one(fx["n_samples"], np.random.RandomState(case["seed"]))
        assert n_c == case["n_out"], case
        want = 0.0 if case["noise_level_db"] is None else 10.0 ** (case["noise_level_db"] / 20.0)
        assert abs(noise_c - want) <= 1e-7 * max(want, 1.0), case
    eval_dl = Speech2TextDataLayer(dict(base, mode="eval", augmentation=aug, shuffle=False), None, 1, 0)
    assert eval_dl._aug is None                       # training-time transform only
    with pytest.raises(ValueError):
        Speech2TextDataLayer(dict(base, augmentation={"pitch_shift": 2}), None, 1, 0)
    # speech2text.py:184-197: a frequency mask wider than the feature axis raises; the legacy key is an alias
    with pytest.raises(ValueError, match="width_freq_mask"):
        Speech2TextDataLayer(dict(base, augmentation={"n_freq_mask": 1, "width_freq_mask": 65}), None, 1, 0)
    legacy = Speech2TextDataLayer(dict(base, augmentation={"time_stretch_ratio": 0.05}), None, 1, 0)
    assert legacy._aug == {"speed_perturbation_ratio": 0.05}
    s_l, _, n_l = legacy._draw_augmentation([16000] * 200, np.random.RandomState(1))
    assert s_l.min() >= int(16000 * 0.95) and s_l.max() <= int(16000 * 1.05) and len(set(s_l.tolist())) > 50
    with pytest.raises(NotImplementedError):
        Speech2TextDataLayer(dict(base, backend="psf", augmentation=aug), None, 1, 0)
    with pytest.raises(NotImplementedError):
        Speech2TextDataLayer(dict(base, backend="psf", gain=0.5), None, 1, 0)
    # optimizer options that used to be dropped
    p = dict(cfg, max_grad_norm=5.0, freeze_variables_regex="ForwardPass/w2l_encoder/conv1.*")
    p.pop("larc_params")
    kw = optimizer_engine_kwargs(p, 1000)
    assert kw["max_grad_norm"] == 5.0 and kw["freeze_variables_regex"].startswith("ForwardPass")
    with pytest.raises(AttributeError):
        optimizer_engine_kwargs(dict(cfg, max_grad_norm=5.0), 1000)     # LARC + clipping (optimizers.py:161-164)
    # initializers: Xavier in both flavours is built, anything else raises
    assert resolve_initializer(cfg["encoder_params"], cfg, "enc") == "xavier_truncnorm"
    assert resolve_initializer(cfg["decoder_params"], cfg, "dec") == "xavier_uniform"
    assert resolve_initializer({}, {}, "x") == "xavier_uniform"
    with pytest.raises(NotImplementedError):
        resolve_initializer({"initializer": lambda **kw: None}, {}, "x")


def test_quartznet_config_matches_the_reference_and_sep_conv_topology_builds_on_paper(tmp_path):
    """configs/quartznet15x5.py == example_configs/speech2text/quartznet15x5_LibriSpeech.py (layers, optimizer,
    lr policy, spec-augment); sep_conv1d layers map to variables with tf.layers.separable_conv1d's names."""
    ref_path = example_config("quartznet15x5_LibriSpeech.py", tmp_path)
    _, ref, _, rmod = get_base_config(["--config_file=" + ref_path, "--mode=train"])
    _, own, _, omod = get_base_config(["--config_file=" + os.path.join(ROOT, "configs", "quartznet15x5.py"), "--mode=train"])
    assert ref["encoder_params"]["convnet_layers"] == own["encoder_params"]["convnet_layers"]
    for key in ("optimizer_params", "lr_policy_params", "dtype", "batch_size_per_gpu", "num_epochs"):
        assert ref[key] == own[key], key
    assert ref["lr_policy"].__name__ == own["lr_policy"].__name__ == "cosine_decay"
    assert rmod["train_params"]["data_layer_params"]["augmentation"] == omod["train_params"]["data_layer_params"]["augmentation"]
    # the oracle's variable set for this topology: separable main convs AND separable residual convs
    from oracle import torch_twin as TT
    p = TT.init_params(own["encoder_params"]["convnet_layers"][:3], 64, 29, seed=0)
    assert p["conv11/depthwise_kernel"].shape == (33, 64, 1) and p["conv11/pointwise_kernel"].shape == (1, 64, 256)
    assert p["conv25/res/depthwise_kernel"].shape == (1, 256, 1) and p["conv25/res/pointwise_kernel"].shape == (1, 256, 256)
    assert "conv25/res_bn/gamma" in p and "conv21/kernel" not in p


@pytest.mark.parametrize("name,optimizer,policy,larc,aug", [
    ("jasper10x5_LibriSpeech_nvgrad_masks.py", "NovoGrad", "poly_decay", True, True),
    ("jasper-Mini-for-Jetson.py", "NovoGrad", "poly_decay", True, True),
    ("quartznet15x5_LibriSpeech.py", "NovoGrad", "cosine_decay", False, True),
    ("w2l_large_8gpus_mp.py", "Momentum", "poly_decay", True, False),
    ("w2lplus_large_8gpus.py", "Momentum", "poly_decay", True, False),
])  # (w2l_large_8gpus.py / w2lplus_large_8gpus_mp.py differ from these two in `dtype` only; jasper10x5_..._nvgrad.py
    # from its _masks variant in the spec-augment keys only -- each 333 M-parameter dry run holds ~9 GB of host memory)
def test_create_model_dry_run_of_every_tdnn_example_config(monkeypatch, golden_dir, tmp_path, name, optimizer, policy,
                                                           larc, aug):
    """run.py's path for `--mode=train_eval` on every TDNNEncoder config under example_configs/speech2text, unchanged
    except for the dataset paths and the batch size (the reference's toy speech set): get_base_config -> create_model
    -> Speech2Text(train) + Speech2Text(eval) with their data layers, encoder / decoder / loss plugins, the engine
    (on the CPU, kernels stubbed) and the optimizer arguments.  Nothing on that path may raise or be dropped."""
    import copy
    import openseq2seq_b200.engine as E
    from open_seq2seq.utils.utils import create_model
    monkeypatch.setattr(E.JasperEngine, "sync_half_copies", lambda self: None)
    orig = E.JasperEngine.__init__

    def on_cpu(self, *a, **kw):
        kw.setdefault("device", "cpu")
        return orig(self, *a, **kw)
    monkeypatch.setattr(E.JasperEngine, "__init__", on_cpu)
    toy = os.path.join(golden_dir, "toy_speech_data")
    path = example_config(name, tmp_path)
    args, cfg, model, module = get_base_config(["--config_file=" + path, "--mode=train_eval"])
    module = dict(module)
    for k in ("train_params", "eval_params"):
        module[k] = copy.deepcopy(module[k])
        module[k]["data_layer_params"]["dataset_files"] = [os.path.join(toy, "toy_data.csv")]
        if "vocab_file" in module[k]["data_layer_params"]:
            module[k]["data_layer_params"]["vocab_file"] = os.path.join(toy, "vocab.txt")
        module[k]["batch_size_per_gpu"] = 2
    cfg = copy.deepcopy(cfg)
    cfg.setdefault("data_layer_params", {})["vocab_file"] = os.path.join(toy, "vocab.txt")
    cfg.update(logdir=str(tmp_path), batch_size_per_gpu=2, use_horovod=False, num_gpus=1)
    train_model, eval_model = create_model(args, cfg, module, model, None)
    assert train_model.engine is not None and eval_model.engine is not None
    opt = train_model.params["optimizer"]
    assert (opt if isinstance(opt, str) else opt.__name__) == optimizer
    assert train_model.params["lr_policy"].__name__ == policy
    assert bool(train_model.params.get("larc_params")) == larc
    assert bool(train_model.get_data_layer().params.get("augmentation")) == aug
    assert not eval_model.get_data_layer().params.get("augmentation")
    assert train_model.engine.hp is not None          # the optimizer arguments reached the engine
