"""bench.py -- Jasper 10x5 bf16 training throughput (audio-seconds/sec) on N B200s.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # CPU reference arm (oracle port, TF1 is
                                                           # not installable offline; see DESIGN.md)

One "step" = one pass of the hot path over one batch of 32 synthetic 16 kHz / 15 s utterances per
rank: log-mel featurizer -> Jasper 10x5 DR encoder -> FC -> CTC loss fwd/bwd -> gradient all-reduce
(NCCL, N > 1) -> loss-scaled LARC + NovoGrad step.  `value` times K steps with the int16 waveforms
already resident in HBM (CUDA events, barrier + synchronize on both sides, max over ranks); `e2e`
times the same steps driven through the public plugin API with pinned HOST waveforms copied to the
device and the loss read back every step.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

AUDIO_SECONDS = 15.0
BATCH = 32
SR = 16000
TRAIN_GFLOP_PER_AUDIO_S = 100.02  # SURVEY.md section 8d (fwd+dgrad+wgrad conv/GEMM FLOPs)
NOMINAL_BF16_TFLOPS = 2250.0   # dense bf16, B200 data sheet (at the 1965 MHz boost clock)
METRIC = "audio-seconds/sec Jasper-10x5 bf16 train"
WORKLOAD = ("Jasper 10x5 DR (configs/jasper10x5_dr.py = reference jasper10x5_LibriSpeech_nvgrad): "
            "featurizer + encoder + FC + CTC fwd/bwd + LARC/NovoGrad, 16 kHz x 15 s utterances")


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1380.3), d.get("hbm_gbs", 6566.7), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "samples": len(rows), "power_w_max": max(float(r[2]) for r in rows)}


def nvlink_counters(index):
    """(tx_bytes, rx_bytes) moved over all NVLinks of GPU `index` so far (NVML throughput counters, KiB), or
    None when NVML / the counters are not available."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        v = pynvml.nvmlDeviceGetFieldValues(h, [(pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, 0xFFFFFFFF),
                                                (pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX, 0xFFFFFFFF)])
        if any(x.nvmlReturn != 0 for x in v):
            return None
        return tuple(int(x.value.ullVal) * 1024 for x in v)
    except Exception:
        return None


def _cgroup_cpu_limit():
    """CPU quota of this container in cores (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return float(q) / float(per)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return q / per
    except Exception:
        pass
    return None


_THREADS = {}


def _host_threads():
    """Threads of the CPU arm.  BASELINE.md section 3 asks for every host core (`torch.set_num_threads(
    os.cpu_count())`); on the GPU boxes that is 128 logical CPUs and measured 9x SLOWER than 32 threads for this
    graph (profiles/r01_bench_first.jsonl vs the later round-1 lines; the final round-2 run repeated it), so the
    count is calibrated instead: the cores this process may use (affinity, cgroup quota), halved while a short
    fp32 conv forward + backward of a Jasper-sized layer runs faster with fewer threads.  The JSON line states the
    count that was used.  OS2S_CPU_THREADS overrides."""
    if os.environ.get("OS2S_CPU_THREADS"):
        return max(1, int(os.environ["OS2S_CPU_THREADS"]))
    if "n" in _THREADS:
        return _THREADS["n"]
    import math
    import torch
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    lim = _cgroup_cpu_limit()
    if lim:
        n = min(n, max(1, int(math.ceil(lim))))
    x = torch.randn(2, 512, 600)
    w = torch.randn(512, 512, 11, requires_grad=True)

    def probe(k):
        torch.set_num_threads(k)
        best = 1e30
        for _ in range(3):
            t0 = time.time()
            y = torch.nn.functional.conv1d(x, w, padding=5)
            y.sum().backward()
            best = min(best, time.time() - t0)
        return best

    best_k, best_t = n, probe(n)
    k = n // 2
    while k >= 4:
        t = probe(k)
        if t < 0.9 * best_t:
            best_k, best_t = k, t
        elif t > 1.3 * best_t:
            break
        k //= 2
    _THREADS["n"] = max(1, best_k)
    _THREADS["of"] = n
    torch.set_num_threads(_THREADS["n"])
    return _THREADS["n"]


def synth_waveforms(rank, n_utts, seconds):
    """SURVEY.md section 8d: int16(clip(3000*N(0,1))) per rank, fixed seed."""
    import numpy as np
    g = np.random.default_rng(1234 + rank * 1000)
    n = int(seconds * SR)
    return [np.clip(3000.0 * g.standard_normal(n), -32768, 32767).astype(np.int16) for _ in range(n_utts)]


def synth_labels(rank, n_utts):
    import numpy as np
    g = np.random.default_rng(4321 + rank)
    lens = g.integers(180, 261, size=n_utts)
    y = np.zeros((n_utts, int(lens.max())), dtype=np.int32)
    for i, L in enumerate(lens):
        y[i, :L] = g.integers(0, 28, size=L)
    return y, lens.astype(np.int32)


# --------------------------------------------------------------------------- reference arm
def _own_config(batch, world, augmentation=True):
    """`config` of the JSON line: the SAME dict for the own arm and the reference arm (the reference arm
    times bounded samples of this workload, described in its cpu_baseline.sample)."""
    return {"workload": WORKLOAD,
            "batch_per_gpu": batch, "global_batch": batch * world, "audio_seconds_per_utt": AUDIO_SECONDS,
            "parallelism": "dp%d" % world,
            "augmentation": ("speed_perturbation_ratio [0.9, 1.0, 1.1] (train_params of the headline config), on: the "
                             "padded batch is 16.5 s long, audio-seconds count the resampled signals"
                             if augmentation else "off (--no_augmentation A/B run)"),
            "l2_policy": "working set per step (activations ~6 GB, params/grads ~5 GB) >> 126 MB L2; no flush needed",
            "train_gflop_per_audio_s": TRAIN_GFLOP_PER_AUDIO_S}


class _CpuPort(object):
    """The reference's CPU path restated (oracle/torch_twin.py + oracle/featurizer.py + oracle/augment.py): fp32
    PyTorch-CPU port of the identical graph -- featurizer (with the recipe's speed perturbation), Jasper 10x5
    DR forward, CTC, backward, LARC + NovoGrad.  TF1 / librosa / resampy are not installable offline."""

    def __init__(self, n_utts, secs, cores):
        import numpy as np
        import torch
        from oracle import torch_twin as TT
        import openseq2seq_b200.compat as compat
        compat.install()
        from open_seq2seq.utils.utils import get_base_config
        _, cfg, _, _ = get_base_config(["--config_file=" + os.path.join(ROOT, "configs", "jasper10x5_dr.py")])
        self.layers = cfg["encoder_params"]["convnet_layers"]
        torch.set_num_threads(cores)
        self.params = TT.init_params(self.layers, 64, 29, seed=0)
        for v in self.params.values():
            v.requires_grad_(True)
        self.mom = {}
        self.waves = synth_waveforms(0, n_utts, secs)
        # the same label generator as the own arm (synth_labels), scaled to the sample's duration
        g = np.random.default_rng(4321)
        lens = g.integers(int(12 * secs), int(17.3 * secs) + 1, size=n_utts)
        y = np.zeros((n_utts, int(lens.max())), dtype=np.int64)
        for i, L in enumerate(lens):
            y[i, :L] = g.integers(0, 28, size=L)
        self.y, self.ylen = torch.tensor(y), torch.tensor(lens, dtype=torch.long)
        self.rng = np.random.RandomState(1)
        self.n_utts, self.secs = n_utts, secs

    def step(self):
        import numpy as np
        import torch
        from oracle import augment as AU
        from oracle import featurizer as FZ
        from oracle import torch_twin as TT
        aug = {"speed_perturbation_ratio": [0.9, 1.0, 1.1]}
        sigs = []
        for w in self.waves:
            x = FZ.normalize_signal(w.astype(np.float32))
            sigs.append(AU.augment_audio_signal(x, SR, aug, self.rng))
        feats, lens = FZ.batch_features(sigs, pad_to=16)
        x = torch.tensor(feats, dtype=torch.float32)
        loss, _, _ = TT.forward_loss(self.params, self.layers, x, torch.tensor(lens, dtype=torch.long), self.y, self.ylen)
        grads = torch.autograd.grad(loss, list(self.params.values()))
        TT.larc_novograd_step(self.params, dict(zip(self.params.keys(), grads)), self.mom, lr=0.02)
        return float(loss.detach())


def run_reference(args):
    """`--impl reference`: the reference's CPU path (restated port, see _CpuPort) on the host cores, same metric /
    unit / config as the own arm; each of the K steps is BASELINE.md section 3's batch -- 2 utterances x 15 s -- and
    the run stops early after ~200 s of timed steps.  If the single warm-up step shows that one such step takes
    over a minute, the samples are shortened to 2 x 4 s and the line says so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _host_threads()
    secs, B = AUDIO_SECONDS, 2
    port = _CpuPort(B, secs, cores)
    t0 = time.time()
    port.step()
    if time.time() - t0 > 60.0:
        secs = 4.0
        port = _CpuPort(B, secs, cores)
        port.step()
    t0 = time.time()
    n = 0
    budget = 200.0
    for _ in range(args.steps):
        port.step()
        n += 1
        if time.time() - t0 > budget:
            break
    dt = time.time() - t0
    val = n * B * secs / dt
    sample = ("1 warm-up + %d training steps of %d utterances x %.0f s each, %d threads (fastest count for an fp32 conv probe among "
              "the %d usable host CPUs); fp32 torch-CPU port of the reference graph incl. the speed-perturbation "
              "resampler; TF1 not installable offline" % (n, B, secs, cores, _THREADS.get("of", cores)))
    out = {"impl": "reference", "metric": METRIC, "value": round(val, 4),
           "unit": "audio-s/s", "n_gpus": args.gpus, "steps": n, "warmup": args.warmup,
           "ms_per_step": round(1000 * dt / n, 2), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": _own_config(args.batch, max(1, args.gpus)),
           "cpu_baseline": {"value": round(val, 4), "unit": "audio-s/s", "cores": cores, "kind": "port",
                            "sample": sample},
           "e2e": {"value": round(val, 4), "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def cpu_baseline_quick():
    """BASELINE.md section 3 protocol, timed inside the default run (rank 0, N = 1): B = 2 utterances x 15 s of
    the same synthetic waveforms, 1 warm-up + 3 timed training steps (featurizer + fwd + bwd + optimizer), all
    host cores, fp32.  If the warm-up step shows that 3 more steps would take over ~75 s, fewer steps are
    timed and the line says so."""
    cores = _host_threads()
    B, secs = 2, AUDIO_SECONDS
    port = _CpuPort(B, secs, cores)
    t0 = time.time()
    port.step()
    warm = time.time() - t0
    n_timed = 3 if warm * 3 <= 75.0 else (2 if warm * 2 <= 75.0 else 1)
    t0 = time.time()
    for _ in range(n_timed):
        port.step()
    dt = time.time() - t0
    return {"value": round(n_timed * B * secs / dt, 4), "unit": "audio-s/s", "cores": cores, "kind": "port",
            "sample": "BASELINE.md section 3: 1 warm-up + %d timed training steps of 2 utterances x 15 s, %d threads "
                      "(fastest count for an fp32 conv probe among the %d usable host CPUs), fp32 torch-CPU port of the "
                      "reference graph (oracle/); TF1 not installable offline"
                      % (n_timed, cores, _THREADS.get("of", cores))}


# --------------------------------------------------------------------------- CUDA arm
PARAM_SAMPLE = 1 << 20   # fp32 master weights written by --dump-outputs (4 MB + 8 MB of float64 indices)
DUMP_BUDGET = 64 << 20   # bytes --dump-outputs writes at most


def dump_outputs(out_dir, eng, last):
    """--dump-outputs: what the last timed step computed, as float32 / float64 .npy files (~28 MB at the default
    batch, never more than DUMP_BUDGET), so two builds can be compared output for output.  The inputs are seeded, so the same arguments give the
    same inputs on every run.  Written: the features and their lengths, the batch-mean loss and the input frame count
    (what Speech2Text.train_step returns), the per-utterance CTC loss and the logits of that step's forward pass, and
    a fixed, seeded sample of the parameters after its optimizer update (with the flat indices of the sample).
    Features and logits are written for the first U utterances of the batch, U as large as the budget allows (all
    32 at the default batch).  That step starts from the seeded initial training state (see run_own), so the features repeat bit for bit and
    the rest differs between runs only by that one step's float-atomic reductions, amplified through the 53 bf16
    layers (two runs of --steps 10 on a B200 at 1000 W: loss 5e-5 apart relative, sampled parameters 8e-4 absolute,
    logits 1.6 % in relative L2 norm)."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    ws = eng._last_ws
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(eng.master.numel(), min(PARAM_SAMPLE, eng.master.numel()),
                                                  replace=False))
    arrays = {
        "feature_lengths": last["feature_lengths"].double(),
        "loss": last["loss"].float().reshape(1),
        "frames": last["frames"].double().reshape(1),
        "loss_per_utterance": ws.loss.float(),
        "params_sample": eng.master[torch.from_numpy(idx).to(eng.master.device)].float(),
        "params_sample_index": torch.from_numpy(idx.astype(np.float64)),
    }
    feats, logits = last["features"], ws.logits
    per_utt = 4 * (feats[0].numel() + logits[0].numel())
    fixed = sum(t.numel() * t.element_size() for t in arrays.values())
    n_utt = min(feats.shape[0], (DUMP_BUDGET - fixed - 4096) // per_utt)   # (4 KB for the .npy headers)
    arrays.update(features=feats[:n_utt].float(), logits=logits[:n_utt].float())
    assert sum(t.numel() * t.element_size() for t in arrays.values()) <= DUMP_BUDGET
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


def training_state(eng):
    """Every device buffer a training step reads and then updates: fp32 masters, gradients and optimizer slots, the
    16-bit weight copies, the merged residual kernels, BN moving statistics, the loss-scaler / step / dropout counters."""
    ts = [eng.master, eng.grad, eng.mom, eng.wb, eng.fstate, eng.istate] + list(eng.wcat) + list(eng.dwcat)
    ts += list(eng.moving.values()) + [eng._opt[k] for k in ("ema", "norms", "nonfinite", "coef")]
    return ts + [t for t in (eng.mom2, eng.grad_acc) if t is not None]


def run_own(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import openseq2seq_b200.compat as compat
    compat.install()
    from open_seq2seq.utils.utils import get_base_config, nested_update
    from openseq2seq_b200.dist import TorchDistHvd
    import copy

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        hvd = TorchDistHvd.init()
    else:
        torch.cuda.set_device(0)
        hvd = TorchDistHvd.single()
    rank, local = hvd.rank(), hvd.local_rank()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device -- the product path has no CPU fallback")

    _, cfg, model_cls, module = get_base_config([
        "--config_file=" + os.path.join(ROOT, "configs", "jasper10x5_dr.py"), "--mode=train"])
    cfg = copy.deepcopy(cfg)
    nested_update(cfg, copy.deepcopy(module["train_params"]))
    cfg.pop("num_epochs", None)
    cfg["max_steps"] = 100000  # lr schedule horizon; the bench runs K + W steps of it
    cfg["batch_size_per_gpu"] = args.batch
    if args.no_augmentation:
        cfg["data_layer_params"].pop("augmentation", None)   # A/B only: the headline recipe trains with it
    model = model_cls(params=cfg, mode="train", hvd=hvd if world > 1 else None)
    model.compile()
    eng = model.engine
    dl = model.get_data_layer()
    # the seeded initial training state; the last timed step starts from it again (see below).  One device copy made
    # before any step, on every run so that the timed path is the same with and without --dump-outputs: ~4.7 GB of
    # HBM per rank for Jasper 10x5 (fp32 masters, gradients and momenta, 3 x 1.33 GB, + the 0.67 GB 16-bit weights)
    initial_state = [(t, t.clone()) for t in training_state(eng)]

    # the synthetic utterances come from the data layer's own in-memory generator ("synthetic:<n>:<seconds>" in
    # configs/jasper10x5_dr.py: int16 Gaussian-noise waveforms + random transcripts, SURVEY.md section 8d)
    res_targets = None
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()

    last = {}

    def step_resident():
        # waveforms already in HBM (dl keeps a device staging buffer): featurizer + train step
        feats, flens = dl.featurize_resident(seed=eng.step_count)
        loss, frames = model.train_step({"source_tensors": [feats, flens], "target_tensors": res_targets})
        last.update(features=feats, feature_lengths=flens, loss=loss, frames=frames)

    # end to end = the call sequence a user of the plugin API makes (utils/funcs.py train loop): next(iterator) --
    # the data layer's producer thread stages the batch's HOST waveforms in pinned memory, copies them to the
    # device and runs augmentation + featurizer on a side stream one batch ahead -- then model.train_step, then
    # a device->host read of the step's loss.
    it = dl.iterator
    h2d = {"bytes": 0}

    def step_e2e():
        batch = next(it)
        h2d["bytes"] = int(dl.h2d_bytes + batch["target_tensors"][0].numel() * 4 + batch["target_tensors"][1].numel() * 4)
        loss, _ = model.train_step(batch)
        loss_host.copy_(loss.reshape(1), non_blocking=False)              # D2H read of the step's loss
        return float(loss_host[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms

    # warm-up (also builds the launch plans and the device staging buffers)
    last_loss = None
    for _ in range(max(args.warmup, 3)):
        last_loss = step_e2e()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_e2e = timed(step_e2e, args.steps)
    # device-resident leg: stop the producer thread, stage ONE batch through the same collate path on this stream
    # (length-sorted, its draws of the speed perturbation stay fixed), then time featurizer + train step on the
    # waveforms that are now resident in HBM
    dl._stop_producer()
    torch.cuda.synchronize()
    res_batch = next(dl._batches_sync())
    res_targets = res_batch["target_tensors"]
    for _ in range(3):
        step_resident()
    barrier()
    nv0 = nvlink_counters(local) if (world > 1 and rank == 0) else None
    # The reductions of a step sum with float atomics, so two runs' training states drift apart step by step.  The
    # last of the K timed steps therefore starts from the seeded initial state, restored between two timed windows:
    # what it computes (--dump-outputs) depends only on the arguments, up to that one step's rounding.  That step
    # runs at the initial weights, loss scale, scaler iteration and global step (the learning rate of step 0).  The
    # running count of skipped (non-finite) steps, istate[4], is not part of that state: it carries over, so
    # `skipped_steps` counts every step of the run.
    ms = timed(step_resident, args.steps - 1) if args.steps > 1 else 0.0
    if args.steps > 0:
        skipped_so_far = int(eng.istate[4])
        for t, t0 in initial_state:
            t.copy_(t0)
        eng.istate[4] = skipped_so_far
        ms += timed(step_resident, 1)
    nv1 = nvlink_counters(local) if nv0 is not None else None
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, last)

    # roofline of the dominant kernel family (tcgen05 implicit-GEMM conv): per-launch CUDA-event
    # timing of every conv launch of instrumented steps run right after the timed region
    roof = eng.profile_conv_launches(lambda: step_resident(), steps=2)
    skipped = int(eng.istate[4])
    total_audio = world * args.batch * AUDIO_SECONDS
    value = total_audio * args.steps / (ms / 1000.0)
    e2e = total_audio * args.steps / (ms_e2e / 1000.0)
    if rank != 0:
        return
    peak_tf, peak_hbm, peak_src = _peaks()
    # roofline.traffic: DRAM bytes per launch of the dominant conv kernel from the committed `ncu --set full`
    # capture (a profiler run of an earlier build of the same kernel, not this run: say so in the line)
    traffic, traffic_src = None, None
    for name in ("r02_ncu_conv_halo_summary.json", "ncu_conv_summary.json"):
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
                traffic_src = "profiles/" + name + " (ncu --set full capture of this kernel, committed; not measured in this run)"
                break
            except Exception:
                traffic = None
    out = {
        "metric": METRIC,
        "value": round(value, 2), "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": _own_config(args.batch, world, not args.no_augmentation),
        "storage": {"half": eng.act_dtype, "conv_out": eng.conv_dtype,
                    "note": "format of the 16-bit tensors (activations, weight copies, gradients) / of the conv outputs; "
                            "fp32 masters and fp32 accumulation in every mode"},
        "e2e": {"value": round(e2e, 2), "unit": "audio-s/s", "ms_per_step": round(ms_e2e / args.steps, 3),
                "h2d_bytes_per_step": h2d["bytes"],
                "api": "next(Speech2TextDataLayer.iterator) [pinned host waveforms -> H2D + augmentation + featurizer on a "
                       "side stream] + Speech2Text.train_step + loss read",
                "d2h_bytes_per_step": 4},
        "gpu_launches": int(eng.kernel_launches_per_step() * args.steps),
        "clocks": clocks,
        "roofline": {"bound": "tensor",
                     "kernel": "tapgemm_kmajor_pair_halo / tapgemm_mnmajor_pair (+ single-CTA variants on the narrow layers): "
                               "tcgen05 cta_group::2 implicit-GEMM conv fwd + dgrad + wgrad",
                     "achieved": roof["tflops"], "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": round(roof["tflops"] / peak_tf, 4), "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src,
                     # the measured peak is cuBLAS bf16 run back to back under the same 1000 W cap; a frac
                     # above 1 means these kernels sustain more than cuBLAS does, not more than the silicon
                     "peak_nominal": NOMINAL_BF16_TFLOPS,
                     "frac_nominal": round(roof["tflops"] / NOMINAL_BF16_TFLOPS, 4),
                     "launches_per_step": roof["launches"],
                     "conv_ms_per_step": roof["ms"], "share_of_step": round(roof["ms"] / (ms / args.steps), 4),
                     "algorithmic_tflop_per_step": roof["tflop"],
                     "how": "CUDA events around every conv launch of 2 instrumented steps after the timed region",
                     "by_kind": roof["by_kind"],
                     # the HBM-bound family (BN forward / backward, optimizer, depthwise): algorithmic bytes / CUDA-event
                     # time of the same instrumented steps, against the measured copy bandwidth
                     "hbm_family": dict(roof["hbm"], peak=peak_hbm, unit="GB/s",
                                        frac=round(roof["hbm"]["gbs"] / peak_hbm, 4)),
                     "step_frac_of_peak": round(value / world * TRAIN_GFLOP_PER_AUDIO_S / 1000.0 / peak_tf, 4)},
        "loss": last_loss, "skipped_steps": skipped,
    }
    if world > 1 and nv0 is not None and nv1 is not None:
        # algorithmic volume of a two-phase sum of the 1.33 GB flat fp32 gradient: 2 (N-1)/N x 1.33 GB each way
        out["nvlink"] = {"tx_bytes_per_step": (nv1[0] - nv0[0]) // args.steps,
                         "rx_bytes_per_step": (nv1[1] - nv0[1]) // args.steps,
                         "algorithmic_bytes_per_step_each_way": int(2 * (world - 1) / world * eng._total * 4),
                         "how": "NVML NVLink data throughput counters of rank 0's GPU around the timed region"}
    if world > 1:
        out["grad_exchange"] = ("peer memory: copy engines over NVLink + slice-sum kernel (csrc/peer.cu)"
                                if getattr(eng, "peer", None) is not None else "nccl all_reduce")
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_quick()
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_augmentation", action="store_true",
                    help="A/B measurement without the recipe's speed perturbation (fixed 15 s utterances)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
