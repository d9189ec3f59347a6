#!/usr/bin/env python
"""bench.py -- MERLOT pretraining-step throughput on B200 (BASELINE.json metric: frame-caption segments/sec, fwd+bwd+AdamW).

  python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path (N>1: launched under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  # the reference math on the box's host cores (oracle port;
                                                           # TF 1.15 cannot be installed here, see DESIGN.md)

Workload (configs[1]): 4-segment pretrain step, model/configs/merlot.yaml sizes with the 16x16 patch-embed ViT-B/16
(resnet_layers: []), bf16, batch 8 per GPU (32 segments/step/GPU), synthetic frames + captions, random-init weights,
hidden dropout 0.1 as in the reference's training graph.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T00 = time.time()


def log(msg):
    print(f"[bench +{time.time() - T00:7.1f}s] {msg}", file=sys.stderr, flush=True)


METRIC = "frame-caption segments/sec (fwd+bwd+AdamW)"
UNIT = "segments/s"
PER_GPU_BATCH = 8
STEM = "patch"  # --stem hybrid: merlot.yaml exactly as shipped (resnet_layers [3, 4, 9]) -- reported beside the headline, never instead of it


def load_config():
    """merlot.yaml's model/optimizer sections (restated here because /root/reference does not travel to the GPU box),
    with the patch-embed stem the north star names (SURVEY.md discrepancy 1)."""
    from merlot_b200.config import NeatConfig
    model = dict(transpose_input=True, num_chunks_in_group=4, masking_use_attn=True, masking_rate=0.2, masking_do_spanbert=True,
                 masking_choose_topk_prob=0.5, image_shuffle_prob=0.4, masking_spanbert_len_probs=[0.625, 0.25, 0.125],
                 resnet_layers=[], do_projection=True, do_bias=True, image_size=[192, 352], patch_size=16, spatial_pool_size=2,
                 use_bfloat16=True, vocab_size=50370, hidden_size=768, contrastive_size=768, contrast_coef=0.25,
                 contrast_temp=0.05, attention_probs_dropout_prob=0.0, hidden_dropout_prob=0.1, hidden_act="gelu",
                 initializer_range=0.02, intermediate_size=3072, max_position_embeddings=1024, num_attention_heads=12,
                 num_hidden_layers=12, num_vision_transformer_hidden_layers=12, num_lang_transformer_hidden_layers=12,
                 share_params=True)
    optimizer = dict(type="adam_optimizer", learning_rate=0.0003, num_train_steps=460000, num_warmup_steps=10000,
                     weight_decay_rate=0.1, beta_2=0.98, clip_norm=0.0, adafactor=False, use_bfloat16_adam=True, verbose=False,
                     param_overrides=[[["LayerNorm", "layer_norm", "GroupNorm", "bias"], {"weight_decay_rate": 0}]])
    if STEM == "hybrid":
        model["resnet_layers"] = [3, 4, 9]  # model/configs/merlot.yaml:33
    return NeatConfig.from_dict({"data": {"num_chunks": 16, "chunk_text_len": 32}, "model": model, "optimizer": optimizer,
                                 "device": {"use_tpu": False, "output_dir": "/tmp/merlot_b200"}})


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler:
    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                                       str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        sm = sorted(int(r[0]) for r in rows if r[0].isdigit())
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        mx = max((int(r[1]) for r in rows if r[1].isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(rows)}


# ---------------------------------------------------------------------------------------------------------------------
def usable_cores():
    """Host threads this process can really use: CPU affinity, capped by a cgroup CPU quota if one is set."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


def cpu_threads():
    # The oracle is ~2000 small-to-medium torch ops per step; beyond ~32 OpenMP threads the per-op fork/join cost on a
    # shared 128-thread host outweighs the extra cores (measured: >100 s/step with 128 threads vs ~5 s with 8).
    return int(os.environ.get("MERLOT_CPU_THREADS", min(usable_cores(), 32)))


def cpu_reference_step_fn(config, batch):
    """One fwd + bwd + AdamW step of the restated reference math (oracle) on the host cores. Returns (fn, segments)."""
    from oracle import merlot_oracle as O
    torch.set_num_threads(cpu_threads())
    cfg = dict(config.model)
    params = O.init_params(cfg, seed=0)
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    adam = O.AdamOracle(leaf, dict(config.optimizer))
    n = cfg["num_chunks_in_group"]
    g = torch.Generator().manual_seed(0)
    Hh, Ww = cfg["image_size"]
    image = torch.rand(batch * n, Hh, Ww, 3, generator=g)
    ids = torch.randint(100, 50357, (batch, n, 32), generator=g, dtype=torch.int32)
    ids[:, :, 0] = O.START
    ids[:, :, 24:] = 0
    shuf = torch.arange(n, dtype=torch.int32).repeat(batch)
    vid = torch.zeros(batch, n, dtype=torch.int32)
    draws = O.make_mask_draws(batch, n * 32, int(n * 32 * 0.2), cfg["vocab_size"], seed=1)

    def step():
        for v in leaf.values():
            v.grad = None
        m = O.MerlotOracle(cfg, leaf, image, ids, mask_input=True, shuffled_idx_img=shuf, mask_draws=draws,
                           log_attention_probs=False)
        total, _ = O.pretrain_losses(m, shuf, vid)
        total.backward()
        adam.apply_gradients(leaf, {k: v.grad for k, v in leaf.items()})
        return float(total)

    return step, batch * n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    config = load_config()
    step, segs = cpu_reference_step_fn(config, batch=1)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = segs * args.steps / dt
    cores = cpu_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: 4-segment pretrain step, merlot.yaml sizes, ViT-B/16 patch-embed + 12-layer joint "
                               "encoder; reference math restated in torch fp32 on host cores (TF 1.15 not installable)",
                   "global_batch": 1, "segments_per_step": segs},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} steps of batch=1 (4 segments) fwd+bwd+AdamW, dropout 0"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
DUMP_PARAM_SAMPLE = 1 << 22  # parameters --dump-outputs writes: a fixed, seeded sample (16 MB as float32) of the 223 M
DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir, spec, store):
    """--dump-outputs: what a caller of the timed step receives from its last run, as DIR/<name>.npy in float32/float64 --
    the three losses, every logged metric, the joint encoder's hidden states, and the updated parameters sampled at fixed
    seeded positions of their reference-named, name-sorted concatenation -- so that two builds run with the same arguments
    (hence the same inputs) can be compared output for output.  Reads buffers the next step overwrites: call it first."""
    import re
    import numpy as np
    arrays = {"loss_parts": np.array([float(x) for x in spec.loss_parts], dtype=np.float64)}
    for k, v in spec.metrics.items():
        arrays["metric_" + re.sub(r"[^0-9A-Za-z]+", "_", k).strip("_")] = torch.as_tensor(v).detach().double().cpu().numpy()
    for k, v in spec.model.encoder_hidden_states.items():
        arrays[f"hidden_{k}"] = v.detach().float().cpu().numpy()
    params = store.to_tf_dict("p")
    names = sorted(params)
    offs = np.cumsum([0] + [params[n].numel() for n in names])
    idx = np.unique(np.random.default_rng(0).integers(0, offs[-1], DUMP_PARAM_SAMPLE))
    owner = np.searchsorted(offs, idx, side="right") - 1
    sample = np.empty(idx.size, dtype=np.float32)
    for i in np.unique(owner):
        sel = owner == i
        sample[sel] = params[names[i]].reshape(-1).numpy()[idx[sel] - offs[i]]
    arrays["params_sample"] = sample
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def run_ours(args):
    from merlot_b200 import _lib as L
    from merlot_b200.train import DataParallel, model_fn_builder, synthetic_batch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (merlot_b200 has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = DataParallel("nccl") if world > 1 else None
    lib = L.lib()
    config = load_config()
    log("building parameter store")
    model_fn = model_fn_builder(config, dist=dist, device=dev)
    store = model_fn.store
    log(f"store ready: {store.num_params() / 1e6:.1f} M params")
    segs_per_rank = PER_GPU_BATCH * config.model["num_chunks_in_group"]

    def sync_all():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident inputs: `value` ----
    feats = synthetic_batch(config, PER_GPU_BATCH, seed=rank, device=dev)

    def one_step(f):
        spec = model_fn(f, None, "train", None)
        spec.train_op()
        return spec

    for i in range(max(args.warmup, 3)):
        one_step(feats)
        torch.cuda.synchronize()
        log(f"warmup step {i} done")
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    lib.merlot_reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        spec = one_step(feats)
    e1.record()
    sync_all()
    launches = int(lib.merlot_launch_count())
    log("timed region done")
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, spec, store)
        log(f"outputs of the last timed step written to {args.dump_outputs}")
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if dist is not None:
        dist.dist.all_reduce(ms, op=dist.dist.ReduceOp.MAX)
    ms_total = float(ms)
    loss_val = spec.loss

    # ---- end to end: pinned host inputs, H2D inside the timed region, loss read back every step ----
    # Every step copies ITS OWN inputs host->device (two device-side buffers; the copy of step i+1 runs on a copy stream while
    # step i computes) and copies its three loss scalars device->pinned host memory; nothing blocks the host in between, all
    # of it is inside the timed region and is drained before the clock stops.
    host = synthetic_batch(config, PER_GPU_BATCH, seed=rank + 1000, pin=True)
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    copy_stream = torch.cuda.Stream(device=dev)
    dev_bufs = [{k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in host.items()} for _ in range(2)]
    copied = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    host_loss = torch.zeros(args.steps + 2, 3, dtype=torch.float32).pin_memory()

    def start_copy(i):
        j = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[j])  # the step that last read this buffer has finished with it
            for k, v in host.items():
                dev_bufs[j][k].copy_(v, non_blocking=True)
            copied[j].record(copy_stream)

    def e2e_step(i, slot):
        j = i & 1
        torch.cuda.current_stream().wait_event(copied[j])
        spec = one_step(dev_bufs[j])
        consumed[j].record(torch.cuda.current_stream())
        host_loss[slot].copy_(torch.stack([x.reshape(()) for x in spec.loss_parts]), non_blocking=True)  # 12 bytes D2H

    for j in range(2):
        consumed[j].record(torch.cuda.current_stream())
    start_copy(0)
    for i in range(2):  # warm-up of this path
        start_copy(i + 1)
        e2e_step(i, args.steps + i)
    sync_all()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    start_copy(0)
    for i in range(args.steps):
        if i + 1 < args.steps:
            start_copy(i + 1)
        e2e_step(i, i)
    t1.record()
    sync_all()
    loss_e2e = float(host_loss[args.steps - 1].sum())
    ms_e = torch.tensor([t0.elapsed_time(t1)], device=dev)
    if dist is not None:
        dist.dist.all_reduce(ms_e, op=dist.dist.ReduceOp.MAX)
    clocks = sampler.stop() if sampler else None
    log("e2e region done")

    # ---- data-parallel diagnostics: per-rank device time of the timed region, and the step time WITHOUT the gradient
    # all-reduce (same kernels, collective skipped) = what the collective costs after overlap ----
    dp_info = None
    if dist is not None:
        mine = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
        allms = [torch.empty_like(mine) for _ in range(world)]
        dist.dist.all_gather(allms, mine)
        dist.skip_grad_allreduce = True
        one_step(feats)
        sync_all()
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0.record()
        for _ in range(5):
            one_step(feats)
        n1.record()
        sync_all()
        dist.skip_grad_allreduce = False
        nc = torch.tensor([n0.elapsed_time(n1) / 5], device=dev)
        dist.dist.all_reduce(nc, op=dist.dist.ReduceOp.MAX)
        dp_info = {"per_rank_ms_per_step": [round(float(x), 3) for x in allms], "ms_per_step_without_grad_allreduce": float(nc),
                   "grad_allreduce_exposed_ms": ms_total / args.steps - float(nc), "grad_bytes_fp32": int(store.g.numel() * 4),
                   "buckets": "1 (everything outside the ViT, under the ViT backward) + 4 ViT layer groups top-down",
                   "note": "runs after both timed regions; the replicas parameters differ afterwards (only the single-rank roofline step follows)"}

    # ---- roofline of the dominant kernel (K1 GEMM), one extra step with per-launch CUDA events ----
    roof = None
    # the profiled step runs with the language-only stack serialised on the main stream: with two streams sharing the SMs a
    # per-launch event duration is no longer that kernel's own execution time
    os.environ["MERLOT_NO_SIDE_STREAM"] = "1"
    one_step(feats)
    torch.cuda.synchronize()
    if rank == 0:
        lib.merlot_gemm_profile_begin()
    one_step(feats)  # every rank takes part (the step contains the NCCL collectives); only rank 0 records events
    os.environ["MERLOT_NO_SIDE_STREAM"] = "0"
    if rank == 0:
        tm, fl, nl = ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
        L.check(lib.merlot_gemm_profile_end(ctypes.byref(tm), ctypes.byref(fl), ctypes.byref(nl)))
        sustained, burst, hbm, how = peaks()
        ach = fl.value / (tm.value * 1e-3) / 1e12
        dom = dominant_k1_instance(dev, sustained)
        roof = {"bound": "tensor", "kernel": "gemm_bf16_kernel / gemm2_bf16_kernel (K1, tcgen05), all launches of a step", "achieved": ach,
                "peak": sustained, "unit": "TFLOP/s", "frac": ach / sustained, "traffic": dom.get("traffic"),
                "traffic_of": dom.get("traffic_of"), "dominant_instance": dom, "peak_source": f"{how} bf16_tflops_sustained",
                "launches_per_step": nl.value, "gemm_ms_per_step": tm.value, "gemm_share_of_step": tm.value / (ms_total / args.steps),
                "note": "sum over all K1 launches (1-CTA and CTA-pair variants) of one single-stream step: sum(2MNK) / sum(CUDA-event "
                        "duration on the launch stream). The event pairs switch off the PDL overlap between consecutive kernels and "
                        "add ~2 us per launch, so this is a lower bound (CUPTI kernel times give ~9.5 ms of K1 per step); isolated "
                        "per-shape rates are in profiles/r01_k1_epilogue_timings.txt"}
    torch.cuda.synchronize()
    # ---- attention TFLOP/s as a share of the peak (second half of BASELINE.json's metric), rank 0, after the timed regions ----
    attn = attention_rates(dev) if rank == 0 else None
    if dist is not None:
        dist.barrier()

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            log("cpu baseline: running `bench.py --impl reference` as a bounded subprocess")
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                                   capture_output=True, text=True, timeout=240)
                ref = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
                cpu = ref["cpu_baseline"]
            except Exception as e:  # the baseline is reported, never fatal
                cpu = {"value": None, "unit": UNIT, "cores": cpu_threads(), "kind": "port", "sample": f"failed/timeout: {e!r}"[:200]}
            log("cpu baseline done")
        val = segs_per_rank * world * args.steps / (ms_total * 1e-3)
        e2e_val = segs_per_rank * world * args.steps / (float(ms_e) * 1e-3)
        line = {
            "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": ("configs[1]: 4-segment pretrain step (ViT-B/16 patch-embed frames 192x352 + 12-layer "
                                    "language-only + 12-layer joint encoder, merlot.yaml sizes), fwd+bwd+AdamW, hidden dropout 0.1")
                       if STEM == "patch" else
                       ("merlot.yaml AS SHIPPED: hybrid ResNet-lite stem (resnet_layers [3, 4, 9]) in front of the ViT, otherwise "
                        "configs[1]'s 4-segment pretrain step, fwd+bwd+AdamW, hidden dropout 0.1 -- not the north-star workload"),
                       "global_batch": PER_GPU_BATCH * world, "segments_per_step": segs_per_rank * world,
                       "parallelism": f"dp{world}", "l2": "per-step working set (~6 GB activations + 2.7 GB parameter state) "
                                                          "is far larger than the 126 MB L2; no explicit flush",
                       "params": store.num_params()},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 12,
                    "ms_per_step": float(ms_e) / args.steps},
            "gpu_launches": launches,
            "roofline": roof,
            "attention": attn,
            "data_parallel": dp_info,
            "cpu_baseline": cpu,
            "loss": loss_val, "loss_e2e_last_step": loss_e2e,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()


def run_other_config(args):
    """`--config 1|4|5`: the other BASELINE.json configs as single-GPU (or per-rank) timed loops -- parity-test shapes, reported
    beside the headline, never instead of it.  1: MerlotModel forward, 1 frame 192x320 + 32 tokens, batch 1 (2-D ids);
    4: sort_story zero-shot forward, 32 rows x 5 frames 384x384 + all-pairs temporal softmax
    (downstream/sort_story/get_zero_shot_logits.py:55-90); 5: stress pretrain step, 8 segments x 384-token captions, batch 16
    per GPU, joint sequence 3608 (needs max_position_embeddings >= 3072: stated override, utils/model_utils.py:282)."""
    from merlot_b200 import _lib as L
    from merlot_b200.modeling import MerlotModel
    from merlot_b200.train import DataParallel, model_fn_builder, synthetic_batch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = DataParallel("nccl") if world > 1 else None
    config = load_config()
    m = config.model
    g = torch.Generator().manual_seed(rank)
    sustained, _, _, how = peaks()
    if args.config == 5:
        m.update(num_chunks_in_group=8, max_position_embeddings=3072)
        config.data.update(num_chunks=8, chunk_text_len=384)
        batch = args.batch or 16
        model_fn = model_fn_builder(config, dist=dist, device=dev)
        feats = synthetic_batch(config, batch, seed=rank, device=dev, num_chunks=8, chunk_text_len=384)
        segs = batch * 8
        flops_step = 115.0e12 * batch / 16  # SURVEY 8(d): 38.33 TFLOP fwd, x3 per step at batch 16

        def step():
            spec = model_fn(feats, None, "train", None)
            spec.train_op()
        what = ("configs[4] stress: 8 segments x 384-token captions, 192x352 frames, joint sequence 3608, pretrain step "
                "fwd+bwd+AdamW, hidden dropout 0.1; max_position_embeddings overridden 1024 -> 3072")
        metric = METRIC
    else:
        from merlot_b200.params import ParamStore
        m["hidden_dropout_prob"] = 0.0
        if args.config == 4:
            m.update(num_chunks_in_group=5, image_size=[384, 384])
            batch, n, hw = args.batch or 32, 5, (384, 384)
            flops_step = 23.52e12 * batch / 32
        else:
            batch, n, hw = args.batch or 1, 1, (192, 320)
            flops_step = 0.060e12 * batch
        store = ParamStore(m, device=dev, with_optimizer_state=False)
        store.init_reference(seed=0)
        image = torch.rand(batch * n, hw[0], hw[1], 3, generator=g).to(torch.bfloat16).to(dev)
        ids = torch.randint(100, 50357, (batch, n, 32), generator=g, dtype=torch.int32)
        ids[:, :, 0] = 2
        ids[:, :, 24:] = 0
        ids = ids.to(dev)
        shuf = (torch.stack([torch.randperm(n, generator=g) for _ in range(batch)]) + 64).int().reshape(-1).to(dev)
        segs = batch * n

        def step():
            if args.config == 1:
                mm = MerlotModel(m, is_training=False, use_tpu=False, image=image, input_ids=ids[:, 0], params=store)
                return mm.encoder_hidden_states["lang"]
            mm = MerlotModel(m, is_training=False, use_tpu=False, image=image, input_ids=ids, mask_input=False,
                             shuffled_idx_img=shuf, params=store)
            H = m["hidden_size"]
            hl = mm.encoder_hidden_states["lang"].reshape(mm.B, n, mm.lang_chunk_length, H)[:, :, 0]
            hv = mm.encoder_hidden_states["viz"].reshape(mm.B, n, mm.viz_chunk_length, H)[:, :, 0]
            return torch.softmax(mm.allpairs_temporal_logits(hl, hv, scope_name="lang_viz_temporal"), -1)
        what = ("configs[3]: sort_story zero-shot forward, 5 x 384x384 frames per story + all-pairs temporal softmax, eval mode"
                if args.config == 4 else "configs[0]: MerlotModel forward, 1 frame 192x320 + 32 text tokens (2-D ids), eval mode")
        metric = "frame-caption segments/sec (forward)"
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    L.lib().merlot_reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if dist is not None:
        dist.dist.all_reduce(ms, op=dist.dist.ReduceOp.MAX)
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        t = float(ms) / args.steps
        tf = flops_step / (t * 1e-3) / 1e12
        print(json.dumps({
            "metric": metric, "value": segs * world / (t * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": what, "global_batch": batch * world, "segments_per_step": segs * world, "parallelism": f"dp{world}",
                       "l2": "working set far larger than the 126 MB L2; no explicit flush"},
            "clocks": clocks, "gpu_launches": int(L.lib().merlot_launch_count()),
            "roofline": {"bound": "tensor", "kernel": "whole step (algorithmic FLOPs of SURVEY 8(d) / step time)", "achieved": tf,
                         "peak": sustained, "unit": "TFLOP/s", "frac": tf / sustained, "traffic": None,
                         "peak_source": f"{how} bf16_tflops_sustained"},
            "e2e": None, "cpu_baseline": None}), flush=True)
    if dist is not None:
        dist.barrier()


def dominant_k1_instance(dev, sustained):
    """The K1 instance with the largest share of the step (profiles/r02_launch_summary_final.txt: the split-K wgrad pair kernel,
    15 %): its ViT FFN2 shape timed live with CUDA events, and its DRAM traffic per launch from the committed `ncu --set full`
    capture (profiles/r02_ncu_kernels_final.json; algorithmic bytes: A 52.3 MB + B 13.1 MB + fp32 red.add output 9.4 MB)."""
    from merlot_b200 import ops
    M, H, I = 8512, 768, 3072
    g = torch.Generator().manual_seed(0)
    xi = (torch.randn(M, I, generator=g) * 0.5).to(torch.bfloat16).to(dev)
    dy = (torch.randn(M, H, generator=g) * 0.5).to(torch.bfloat16).to(dev)
    gw = torch.zeros(I, H, dtype=torch.float32, device=dev)
    fn = lambda: ops.gemm(xi, dy, a_mn_major=True, b_mn_major=True, out=gw, atomic=True, M=I, N=H, K=M)
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(20):
        fn()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / 20 * 1e3
    tf = 2.0 * M * H * I / (us * 1e-6) / 1e12
    out = {"kernel": "gemm2_bf16_kernel<256, A MN-major, B MN-major, split-K red.add f32> (ViT FFN2 wgrad 3072x768x8512)",
           "us_per_launch": us, "achieved": tf, "frac": tf / sustained, "algorithmic_bytes": M * I * 2 + M * H * 2 + I * H * 4,
           "inputs": "104 MB working set per launch pair alternates with nothing else: L2-resident repeats (the ncu capture is the cold figure)"}
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_kernels_final.json")))
        ls = [x for x in d["launches"] if "gemm2_bf16_kernel<256, 1, 1, 2, 1>" in x["kernel"]]
        top = max(ls, key=lambda x: x.get("dram_read_bytes", 0))
        out["traffic"] = top["dram_read_bytes"] + top["dram_write_bytes"]
        out["traffic_of"] = "dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant instance, ncu --set full (profiles/r02_ncu_kernels_final.json)"
        out["ncu_tensor_pipe_pct"] = top.get("tensor_pipe_pct")
    except Exception as e:  # the capture is evidence, never fatal
        out["traffic"] = None
        out["traffic_of"] = f"profiles/r02_ncu_kernels_final.json not readable: {e!r}"[:160]
    return out


def attention_rates(dev):
    """K2 (forward) and K3 (backward incl. dsum / dq finish) alone, CUDA-event timed, at the ViT shape of configs[1]
    (32 frames x 266 tokens) and the joint-encoder shape of SURVEY 8(d) cfg5 (16 x 3608 tokens, key mask off); algorithmic
    FLOPs 4 B h S^2 d forward, 10 B h S^2 d backward (all S keys, no mask discount)."""
    from merlot_b200 import ops
    sustained, _, _, how = peaks()
    out = {"peak": sustained, "peak_source": f"{how} bf16_tflops_sustained", "unit": "TFLOP/s", "shapes": {}}
    g = torch.Generator().manual_seed(0)
    for name, (B, S, it) in {"cfg2_vit_B32_S266": (32, 266, 10), "cfg5_joint_B16_S3608": (16, 3608, 3)}.items():
        heads, H = 12, 768
        qkv = (torch.randn(B * S, 3 * H, generator=g) * 0.5).to(torch.bfloat16).to(dev)
        dctx = (torch.randn(B * S, H, generator=g) * 0.5).to(torch.bfloat16).to(dev)
        ctx, lse = ops.attention_fwd(qkv, B, S, heads)
        dqkv = torch.empty(B * S, 3 * H, dtype=torch.bfloat16, device=dev)
        dq_acc = ops.attention_bwd_workspace(B, S, heads, dev)  # K3 hands it back zeroed
        dsum = torch.empty(B, heads, S, dtype=torch.float32, device=dev)
        ops.attention_bwd(qkv, ctx, dctx, lse, B, S, heads, dqkv=dqkv, dq_accum=dq_acc, dsum=dsum)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        torch.cuda.synchronize()
        ev[0].record()
        for _ in range(it):
            ops.attention_fwd(qkv, B, S, heads, ctx=ctx, lse=lse)
        ev[1].record()
        for _ in range(it):
            ops.attention_bwd(qkv, ctx, dctx, lse, B, S, heads, dqkv=dqkv, dq_accum=dq_acc, dsum=dsum)
        ev[2].record()
        torch.cuda.synchronize()
        f = 4.0 * B * heads * S * S * 64
        tf_f = f / (ev[0].elapsed_time(ev[1]) / it * 1e-3) / 1e12
        tf_b = 2.5 * f / (ev[1].elapsed_time(ev[2]) / it * 1e-3) / 1e12
        out["shapes"][name] = {"fwd_tflops": tf_f, "bwd_tflops": tf_b, "fwd_frac": tf_f / sustained, "bwd_frac": tf_b / sustained}
        del qkv, dctx, ctx, lse, dqkv, dq_acc, dsum
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 4, 5],
                    help="BASELINE.json configs, 1-based as SURVEY 8 numbers them: 2 (default) = the headline 4-segment pretrain step")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override for --config 1/4/5")
    ap.add_argument("--stem", default="patch", choices=["patch", "hybrid"],
                    help="hybrid: merlot.yaml as shipped (ResNet-lite stem before the ViT); default = the north star's patch embedding")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (headline workload only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != 2):
        ap.error("--dump-outputs applies to the headline workload (--impl ours, --config 2)")
    global STEM
    STEM = args.stem
    if args.impl == "reference":
        run_reference(args)
    elif args.config != 2:
        run_other_config(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
