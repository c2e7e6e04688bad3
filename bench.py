#!/usr/bin/env python
"""bench.py — images/sec of the LSeg forward path (480x480, ADE20K-150) on 1..8 B200.

One "step" = one LSegNet.forward over one batch of synthetic images (BASELINE.json configs[1]: batch 8 per GPU, K=150,
480x480, ViT-L/16 DPT); at N > 1 the step is BASELINE.json configs[2]: the batch shards over the ranks and the logits of
all shards are gathered on rank 0 INSIDE the timed region (lang-seg_b200/parallel.py::LogitsGather). Contract: see the
task prompt / DESIGN.md section "Measurement". Prints ONE JSON line on rank 0.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # B200 arm
  python bench.py --impl reference [--steps K] [--warmup W]      # the reference's own CPU path on the host cores
  python bench.py --config 5                                     # BASELINE.json configs[4]: 736^2 (720 padded), K=512, B=4/GPU
  python bench.py --dump-outputs DIR                             # also write the last timed step's logits (sample) to DIR
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NET_KW = dict(backbone="clip_vitl16_384", features=256, crop_size=480, arch_option=0, block_depth=0,
              activation="lrelu")
METRIC = "images/sec at 480x480 ADE20K-150 forward"


DUMP_SAMPLE = 1 << 21  # logit values --dump-outputs writes when the step's logits are larger than that


def sample_outputs(logits):
    """The logits of one step as {name: float32/float64 array}: all of them up to DUMP_SAMPLE values, else DUMP_SAMPLE
    values at flat indices drawn from a fixed seed (the same indices for the same shape in every run, so that two builds
    can be compared value for value). Runs on the device; only the sample is copied to the host."""
    import numpy as np
    flat = logits.detach().reshape(-1)
    out = {"logits_shape": np.array(logits.shape, dtype=np.float64)}
    if flat.numel() <= DUMP_SAMPLE:
        out["logits"] = flat.float().cpu().numpy()
        return out
    idx = np.sort(np.random.Generator(np.random.PCG64(0)).integers(0, flat.numel(), size=DUMP_SAMPLE))
    out["logits"] = flat[torch.from_numpy(idx).to(flat.device)].float().cpu().numpy()
    out["logits_index"] = idx.astype(np.float64)  # exact: numel < 2**53
    return out


def write_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def ade_labels():
    labels = []
    with open(os.path.join(ROOT, "tests", "golden", "ade20k_objectInfo150.txt")) as f:
        for line in f.readlines():
            labels.append(line.strip().split(",")[-1].split(";")[0])
    return labels[1:]


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return (p.get("bf16_tflops_sustained", 1428.7), p.get("bf16_tflops", 1692.4), p.get("hbm_gbs", 6564.2), "measured")
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                parts = [p.strip() for p in out.stdout.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[3:7]) if v.lower().startswith("active")})
        pw = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": reasons, "samples": len(self.samples)}


def bind_to_gpu_numa(index):
    """Pin this process (and the pinned host buffers it allocates afterwards) to the NUMA node the GPU hangs off."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return {"node": None}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus)}
    except Exception as e:  # best effort
        return {"node": None, "error": str(e)[:80]}


# ---------------------------------------------------------------------------------------------------------------------
# the reference's CPU path
# ---------------------------------------------------------------------------------------------------------------------
def _calibrate_threads(fn):
    """torch's CPU kernels do not scale to very wide hosts on these matrix sizes: try a few thread counts on a reduced
    problem and keep the fastest ("all the host threads it can use")."""
    cores = len(os.sched_getaffinity(0))
    best, best_t = cores, None
    for n in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16)}, reverse=True):
        torch.set_num_threads(n)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_reference_rate(steps, warmup, labels, size):
    """images/sec of the reference's CPU path, one image of the workload per step.

    kind "reference": the UNMODIFIED reference `LSegModule.evaluate_random` (modules/lsegmentation_module.py:54-59 ->
    modules/models/lseg_net.py:160-205) from the checkout named by LSEG_REFERENCE_ROOT, with the stand-ins of
    oracle/ref_standins.py for the absent third-party packages; kind "port": the oracle restatement when the reference
    tree is not installed. The reference re-runs the text tower on every call (lseg_net.py:183); `text_cached` subtracts
    a separately timed encode_text so that both accountings are visible."""
    from oracle import ref_standins as R
    from oracle import synth
    sd = synth.make_state_dict(0)
    x_small = synth.make_image(1, 160, 160, seed=0)
    x = synth.make_image(1, size, size, seed=0)
    if R.reference_available():
        module = R.build_reference_module(sd, drop_in=False)
        kind = "reference"

        def fwd(img, lab):
            with torch.no_grad():
                return module.evaluate_random(img, lab)

        def text_only(lab):
            with torch.no_grad():
                return module.net.clip_pretrained.encode_text(synth.tokenize(lab))
    else:
        from oracle import lseg_oracle as O
        tw = O.clip_text_weights_fp16(sd)
        kind = "port"

        def fwd(img, lab):
            return O.lseg_forward(img, synth.tokenize(lab), sd, tw)

        def text_only(lab):
            return O.clip_encode_text(synth.tokenize(lab), tw)
    cores = _calibrate_threads(lambda: fwd(x_small, labels[:8]))
    for _ in range(warmup):
        fwd(x, labels)
    t0 = time.perf_counter()
    for _ in range(steps):
        fwd(x, labels)
    dt = (time.perf_counter() - t0) / steps
    t0 = time.perf_counter()
    text_only(labels)
    t_text = time.perf_counter() - t0
    return {"rate": 1.0 / dt, "sec": dt, "cores": cores, "kind": kind, "text_sec": t_text,
            "rate_text_cached": 1.0 / max(dt - t_text, 1e-9)}


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    labels = cfg["labels"]
    steps = args.steps
    r = cpu_reference_rate(steps, max(1, min(args.warmup, 2)), labels, cfg["size"])
    sample = (f"one {cfg['size']}x{cfg['size']} image of the batch-{cfg['batch']} workload per step (K={len(labels)} labels), "
              f"{steps} steps; the reference re-runs the text tower on every call")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["rate"], "unit": "images/sec", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": r["sec"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32 trunk / fp16 text+corr", "data": "synthetic",
        "config": line_config(cfg, args, int(os.environ.get("WORLD_SIZE", "1"))),
        "cpu_baseline": {"value": r["rate"], "unit": "images/sec", "cores": r["cores"], "kind": r["kind"], "sample": sample,
                         "value_text_cached": r["rate_text_cached"], "text_tower_sec_per_call": r["text_sec"]},
        "e2e": {"value": r["rate"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def line_config(cfg, args, world):
    """The `config` object of the JSON line — the SAME dict in both arms (`--impl b200` and `--impl reference` describe one
    workload; what differs between the arms is said per arm inside the values, and the reference arm's bounded sample is
    in its `cpu_baseline.sample`)."""
    par = f"B200 arm: dp{world}, batch shard per rank, no collective on the image path"
    if world > 1:
        par += f"; all shards' logits gathered on rank 0 inside the timed step ({args.gather})"
    par += "; reference arm: the host cores of rank 0"
    return dict(cfg["config"], backbone=args.backbone, global_batch=cfg["batch"] * world, parallelism=par,
                weights="random init of the architecture",
                text_features="B200 arm: cached per label set; reference arm: re-run on every call as the reference does "
                              "(cpu_baseline.value_text_cached = the same run with the text tower subtracted)",
                l2="B200 arm, N=1: 256 MiB flush (untimed) between timed steps; N>1: back-to-back steps, per-step working "
                   "set ~3.7 GB >> 126 MB L2")


def make_config(args):
    """Workload of this run. config 2 (default): BASELINE.json configs[1] (configs[2] at N > 1); 5: configs[4]."""
    if args.config == 5:
        import numpy as np
        size, batch, K = 736, (args.batch or 4), (args.labels or 512)
        # synthetic prompts as SURVEY.md 8(d) config 5 defines them: [SOT, t_1..t_L, EOT, 0...], L ~ U{1..6}, t ~ U{1000..40000}
        rng = np.random.Generator(np.random.PCG64(0))
        tokens = torch.zeros((K, 77), dtype=torch.int64)
        for i in range(K):
            n = int(rng.integers(1, 7))
            ids = [49406] + [int(v) for v in rng.integers(1000, 40001, size=n)] + [49407]
            tokens[i, : len(ids)] = torch.tensor(ids, dtype=torch.int64)
        labels = [f"prompt{i}" for i in range(K)]
        name = (f"open-vocab stress (BASELINE.json configs[4]): 720x720 padded to {size}x{size} with -1 (720 is not "
                f"runnable: odd token grid), K={K} synthetic prompts, ViT-L/16 DPT")
        return {"size": size, "batch": batch, "labels": labels, "tokens": tokens,
                "config": {"workload": name, "batch_per_gpu": batch}}
    size, batch = args.size, (args.batch or 8)
    labels = ade_labels()[: (args.labels or 150)]
    name = f"ADE20K-150 (K={len(labels)}), ViT-L/16 DPT, {size}x{size}"
    return {"size": size, "batch": batch, "labels": labels, "tokens": None,
            "config": {"workload": name, "batch_per_gpu": batch}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 5])
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default 8; config 5: 4)")
    ap.add_argument("--labels", type=int, default=0)
    ap.add_argument("--size", type=int, default=480)
    ap.add_argument("--gather", default=os.environ.get("LSEG_GATHER_MODE", "p2p_copy"),
                    choices=["p2p_copy", "p2p_store", "nccl"])
    ap.add_argument("--backbone", default="clip_vitl16_384",
                    choices=["clip_vitl16_384", "clipRN50x16_vitl16_384", "clip_vitb32_384"],
                    help="BASELINE.json's metric is quoted on the default; the others are extra lines (config.backbone)")
    ap.add_argument("--gather-sidestream", action="store_true",
                    help="rank 0 expands step s on a side stream during step s+1 instead of on its main stream after it "
                         "(LogitsGather pipelined=False; measured slower, kept for A/B)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-eval", action="store_true", help="skip the multi-scale evaluator line (SURVEY 8(f) row 1)")
    ap.add_argument("--dump-profile", default=None, help="write the per-launch profile of one step to this JSON file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the logits of the last timed step (rank 0; a seeded sample, see sample_outputs) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 arm computes")
    cfg = make_config(args)
    if args.impl == "reference":
        return run_reference(args, cfg)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    import lseg_b200  # noqa: F401
    from lseg_b200 import ops, tokenizer
    from lseg_b200.lseg_net import LSegNet
    from lseg_b200.parallel import LogitsGather
    tokenizer.enable_stand_in()  # random-init weights of the architecture: no CLIP vocabulary offline either

    labels = cfg["labels"]
    K = len(labels)
    B, S = cfg["batch"], cfg["size"]
    torch.manual_seed(1234 + rank)
    net = LSegNet(labels=labels if cfg["tokens"] is None else ["x"], **{**NET_KW, "backbone": args.backbone}).eval().to(dev)
    tokens = cfg["tokens"] if cfg["tokens"] is not None else tokenizer.tokenize(labels)
    if cfg["tokens"] is not None:
        net.text = tokens  # the constructor's label set, pre-tokenised (the public call `net(x)` uses it)
    x_host = torch.randn(B, 3, S, S).clamp_(-1, 1).pin_memory()
    x = x_host.to(dev)
    eng = net._engine_for(dev)
    text = net._text_features(eng, tokens)  # encoded once, cached (steady state of a fixed label set)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    W, Ksteps = max(3, args.warmup), args.steps
    out = torch.empty((B, K, S, S), dtype=torch.float32, device=dev)
    for _ in range(W):
        eng.forward(x, text, K, out=out)
    barrier()
    launches_per_step = eng.last_launch_count()

    # ---- compute only: K steps, L2 flushed (untimed) between steps, CUDA events per step, max over ranks ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(Ksteps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(Ksteps)]
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(Ksteps):
        flush.zero_()
        starts[i].record()
        eng.forward(x, text, K, out=out)
        ends[i].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and dist is None:
        write_outputs(args.dump_outputs, sample_outputs(out))
    clocks = sampler.summary() if world == 1 else None
    compute_ms = max_over_ranks(sum(s.elapsed_time(e) for s, e in zip(starts, ends)))
    compute_value = world * B * Ksteps / (compute_ms / 1e3)

    # ---- N > 1: the step of BASELINE.json configs[2] — forward + gather of all shards' logits on rank 0, timed as a whole.
    # The steps run back to back (the gather of step i overlaps the compute of step i+1 on a side stream), one event pair
    # around all K steps including the drain of the last gather; no flush kernel in between: a step streams ~3 GB of
    # activations and 0.7 GB of weights through the 126 MB L2, nothing of step i survives into step i+1.
    gather_info = None
    value, total_ms = compute_value, compute_ms
    if dist is not None:
        del out
        def run_gather(materialize, root_batch=None):
            g = LogitsGather(eng, B, K, S, S, root=0, mode=args.gather, materialize=materialize,
                             pipelined=not args.gather_sidestream)
            xg = x
            if root_batch is not None and g.mode.startswith("p2p"):
                g.root_batch = root_batch
                if rank == 0:
                    xg = x[:root_batch].contiguous()
            for _ in range(W):
                g.forward(xg, text)
            g.flush()
            barrier()
            smp = ClockSampler(local_rank)
            smp.start()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            t0 = time.perf_counter()
            e0.record()
            for i in range(Ksteps):
                g.forward(xg, text)
            full = g.flush()  # pipelined gather: the expansion of the last step; side-stream gather: its drain
            e1.record()
            barrier()
            wall = time.perf_counter() - t0
            return g, full, max_over_ranks(e0.elapsed_time(e1)), wall, smp.summary()

        # Load-balanced variant: rank 0 also expands every shard to fp32 (t_up per image, serialised with its trunk), so it
        # computes fewer images itself: the largest root batch whose step fits the other ranks' (which skip the expansion).
        t_up = 0.0285 * (K * S * S) / (150.0 * 480 * 480)             # ms per image, measured (profiles/r02_upsample*)
        t_img = max(1e-3, compute_ms / Ksteps / B - t_up)              # ms per image of the trunk
        root_batch = B
        while root_batch > 1 and root_batch * t_img + (root_batch + (world - 1) * B) * t_up > B * t_img:
            root_batch -= 1
        if os.environ.get("LSEG_BENCH_ROOT_BATCH"):  # exercise the path at small N
            root_batch = max(1, min(B, int(os.environ["LSEG_BENCH_ROOT_BATCH"])))
        balanced = None
        if root_batch < B and args.gather.startswith("p2p"):
            gb, _, bal_ms, _, _ = run_gather(True, root_batch)
            n_img = (world - 1) * B + root_batch
            if gb.mode.startswith("p2p"):
                balanced = {"value": n_img * Ksteps / (bal_ms / 1e3), "ms_per_step": bal_ms / Ksteps,
                            "images_per_step": n_img, "root_batch": root_batch,
                            "what": "same gather, rank 0 computes root_batch images instead of %d because it alone expands "
                                    "all shards to fp32; the other ranks keep %d (NOT the configuration of `value`)" % (B, B)}
            gb.close()
            del gb

        g0, _, lowres_ms, _, _ = run_gather(False)   # exchange only: root keeps the fp16 low-res logits of all shards
        g0.close()
        del g0
        g, full, total_ms, t_wall, clocks = run_gather(True)
        if args.dump_outputs and rank == 0:
            write_outputs(args.dump_outputs, sample_outputs(full))
        value = world * B * Ksteps / (total_ms / 1e3)
        wd = ops.read_watchdog()
        check = None
        if rank == 0:  # the gathered tensor is what N independent forwards would have produced: rank 0's own shard bit for bit
            own = eng.forward(x, text, K)
            check = bool(torch.equal(full[:B], own))
            del own
        gather_info = {"mode": g.mode, "fallback_reason": g.fallback_reason, "watchdog": wd[0],
                       "bytes_per_rank_per_step": g.slot_bytes, "gathered_shape": [world * B, K, S, S],
                       "root_shard_bit_identical_to_plain_forward": check,
                       "what": "fp16 low-res logits (the reference's fp16 matmul result, 1/8 of the fp32 bytes it determines) "
                               "pushed into rank 0's buffer over NVLink by the copy engines, release/acquire flags, rank 0 "
                               "expands all shards to fp32 [N*B,K,H,W] (x2 upsample, bit-identical to each rank's own); "
                               + ("on a side stream during its next step" if args.gather_sidestream else
                                  "pipelined: step s-1 is expanded on its main stream after its forward of step s, the last "
                                  "step inside the timed region too"),
                       "pipelined": not args.gather_sidestream,
                       "lowres_only": {"value": world * B * Ksteps / (lowres_ms / 1e3), "ms_per_step": lowres_ms / Ksteps,
                                       "what": "the same steps with the exchange but without rank 0's fp32 expansion: all "
                                               "shards' fp16 low-res logits resident on rank 0 (the difference to `value` is "
                                               "rank 0 writing N*B*K*H*W*4 bytes of fp32 logits per step, which cannot "
                                               "overlap kernels that own every SM's shared memory)"},
                       "balanced": balanced,
                       "compute_only": {"value": compute_value, "ms_per_step": compute_ms / Ksteps,
                                        "what": "the same K steps without the gather (round-1 definition of value)"}}
        g.close()
        out = torch.empty((B, K, S, S), dtype=torch.float32, device=dev)

    # ---- roofline of the dominant kernel family (tcgen05 GEMM) + MHSA: per-launch CUDA events, one step ----
    peak_tf, peak_burst, peak_gbs, peak_src = measured_peaks()
    roofline, mhsa_roof, breakdown = None, None, None
    if rank == 0:
        eng.forward_profiled(x, text, K, out=out)
        _, prof = eng.forward_profiled(x, text, K, out=out)
        if args.dump_profile:
            with open(args.dump_profile, "w") as f:
                json.dump([{"ms": m, "kind": k, "gflop": fl / 1e9} for m, k, fl in prof], f)
        by = {k: [0.0, 0.0, 0] for k in range(5)}  # 0 elementwise, 1 GEMM, 2 MHSA, 3 LayerNorm, 4 memset
        for ms, kind, fl in prof:
            by[kind][0] += ms
            by[kind][1] += fl
            by[kind][2] += 1
        tot = sum(v[0] for v in by.values())
        g_ms_, g_fl, g_n = by[1]
        m_ms, m_fl, m_n = by[2]
        ach = g_fl / (g_ms_ / 1e3) / 1e12 if g_ms_ > 0 else 0.0
        traffic, traffic_m = None, None  # DRAM bytes per launch from this round's committed ncu capture, if present
        try:
            with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
                tj = json.load(f)
            traffic, traffic_m = tj["gemm"]["dram_bytes_per_launch"], tj["mhsa"]["dram_bytes_per_launch"]
        except (OSError, KeyError, ValueError):
            pass
        roofline = {"kernel": "gemm_tc2_kernel (tcgen05 GEMM / implicit conv, all launches of one step)",
                    "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                    "frac_of_burst_peak": ach / peak_burst,
                    "peak_source": f"{peak_src} bf16 sustained (kernel timed inside a long step); burst peak {peak_burst}",
                    "launches": g_n, "avg_launch_ms": g_ms_ / max(g_n, 1), "share_of_step": g_ms_ / tot,
                    "traffic": traffic,
                    "traffic_note": "dram__bytes_read+write per launch (mean over the family) from the ncu capture "
                                    "profiles/r02_traffic.md; per-shape table in profiles/r02_gemm_shapes.md",
                    "timing_note": "per-launch events serialise the programmatic-dependent-launch overlap of consecutive "
                                   "kernels: the breakdown sums to more than ms_per_step"}
        ach_m = m_fl / (m_ms / 1e3) / 1e12 if m_ms > 0 else 0.0
        mhsa_roof = {"kernel": "mhsa2_kernel (lseg_mhsa_variant %s)" % os.environ.get("LSEG_MHSA_VARIANT", "0"),
                     "bound": "tensor", "achieved": ach_m, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_m / peak_tf,
                     "frac_of_burst_peak": ach_m / peak_burst, "launches": m_n, "traffic": traffic_m,
                     "avg_launch_ms": m_ms / max(m_n, 1), "share_of_step": m_ms / tot}
        breakdown = {"gemm_ms": g_ms_, "mhsa_ms": m_ms, "layernorm_ms": by[3][0], "elementwise_ms": by[0][0],
                     "sum_ms": tot}

    # ---- end to end through the public API with HOST buffers (pinned), H2D + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        out_host = [torch.empty((B, K, S, S), dtype=torch.float32).pin_memory() for _ in range(2)]
        copy = torch.cuda.Stream(device=dev)

        def e2e_steps(n):
            for i in range(n):
                xd = x_host.to(dev, non_blocking=True)
                y = net(xd)  # public API: LSegNet.forward(x) with the constructor's labels
                ready = torch.cuda.Event()
                ready.record()
                with torch.cuda.stream(copy):
                    copy.wait_event(ready)
                    out_host[i & 1].copy_(y, non_blocking=True)
                    y.record_stream(copy)
            torch.cuda.current_stream().wait_stream(copy)

        e2e_steps(2)
        barrier()
        t0 = time.perf_counter()
        e2e_steps(Ksteps)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": world * B * Ksteps / dt, "unit": "images/sec", "h2d_bytes_per_step": x_host.numel() * 4,
               "d2h_bytes_per_step": B * K * S * S * 4, "numa": numa,
               "what": "LSegNet.forward from pinned host images to pinned host fp32 logits (each rank its own shard); D2H of "
                       "step i overlaps step i+1; bound by PCIe Gen5 / host memory for the 4*K bytes per pixel"}
        del out_host

    # ---- SURVEY 8(f) row 2, reported beside (not instead of) the contract's e2e: the fused argmax path returns the
    # int64 class mask every caller of the reference derives from the logits, so 8 B/pixel cross PCIe, not 4*K ----
    e2e_argmax = None
    if not args.no_e2e:
        mask_host = [torch.empty((B, S, S), dtype=torch.int64).pin_memory() for _ in range(2)]
        copy2 = torch.cuda.Stream(device=dev)

        def argmax_steps(n):
            for i in range(n):
                xd = x_host.to(dev, non_blocking=True)
                m = net.predict(xd)
                ready = torch.cuda.Event()
                ready.record()
                with torch.cuda.stream(copy2):
                    copy2.wait_event(ready)
                    mask_host[i & 1].copy_(m, non_blocking=True)
                    m.record_stream(copy2)
            torch.cuda.current_stream().wait_stream(copy2)

        argmax_steps(2)
        barrier()
        t0 = time.perf_counter()
        argmax_steps(Ksteps)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        e2e_argmax = {"value": world * B * Ksteps / dt, "unit": "images/sec", "h2d_bytes_per_step": x_host.numel() * 4,
                      "d2h_bytes_per_step": B * S * S * 8,
                      "what": "LSegNet.predict (forward fused with torch.max(.,1)[1]) from pinned host images to a pinned "
                              "host int64 mask"}

    # ---- SURVEY 8(f) row 1: the ADE20K evaluation workload — one 512x683 image, 6 scales, flip, sliding 480x480 windows
    # (test_lseg.py:308-317,383; additional_utils/models.py:55-140): the reference issues one batch-1 forward per window
    # and flip; here the fused evaluator batches every network input of a scale and keeps the glue in three gather kernels.
    evaluator = None
    if rank == 0 and world == 1 and not args.no_eval and cfg["tokens"] is None:
        from lseg_b200.evaluator import MultiScaleEvaluator
        ev = MultiScaleEvaluator(net, base_size=520, crop_size=480, max_batch=16)
        img = torch.randn(1, 3, 512, 683, device=dev).clamp_(-1, 1)
        n_fwd = ev.num_forwards(img)[0]

        def run_eval(fused):
            ev.fused = fused
            ev(img, labels)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                ev(img, labels)
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / 3

        t_fused, t_glue = run_eval(True), run_eval(False)
        evaluator = {"value": 1.0 / t_fused, "unit": "images/sec", "ms_per_image": t_fused * 1e3,
                     "ms_per_image_torch_glue": t_glue * 1e3, "network_inputs_per_image": n_fwd,
                     "workload": "one 512x683 image, scales 0.5..1.75, flip, 480x480 windows with stride 320, K=%d" % K,
                     "reference_forwards_per_image": n_fwd,
                     "what": "MultiScaleEvaluator (fused gather kernels + batched LSegNet.forward), wall clock incl. host "
                             "planning; the reference runs the same %d crops as batch-1 forwards" % n_fwd}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_rate(3, 1, labels if cfg["tokens"] is None else labels[:K], S) if cfg["tokens"] is None else None
        if r is not None:
            cpu_baseline = {"value": r["rate"], "unit": "images/sec", "cores": r["cores"], "kind": r["kind"],
                            "value_text_cached": r["rate_text_cached"], "text_tower_sec_per_call": r["text_sec"],
                            "sample": f"3 timed forwards of one {S}x{S} image (K={K}) after 1 warm-up ({r['sec']:.2f} s each) "
                                      f"through the reference's LSegModule.evaluate_random on the host cores; fp32 trunk, "
                                      f"fp16 text tower re-run per call as the reference does"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "images/sec", "n_gpus": world, "steps": Ksteps, "warmup": W,
            "ms_per_step": total_ms / Ksteps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 operands, fp32 accumulate (fp32 residual stream)", "data": "synthetic",
            "config": line_config(cfg, args, world),
            "wall_s": t_wall, "clocks": clocks, "gpu_launches": launches_per_step * Ksteps,
            "launches_per_step": launches_per_step,
            "roofline": roofline, "roofline_mhsa": mhsa_roof, "step_breakdown_ms": breakdown,
            "cpu_baseline": cpu_baseline, "e2e": e2e, "e2e_argmax": e2e_argmax, "evaluator": evaluator,
        }
        if evaluator is not None and cpu_baseline is not None:
            evaluator["reference_cpu_estimate"] = {
                "value": 1.0 / (evaluator["reference_forwards_per_image"] / cpu_baseline["value"]), "unit": "images/sec",
                "what": "forwards per image x the measured per-forward time of the reference CPU path above (not run: "
                        "%d forwards of ~%.1f s)" % (evaluator["reference_forwards_per_image"], 1.0 / cpu_baseline["value"])}
        if gather_info is not None:
            line["gather"] = gather_info
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
