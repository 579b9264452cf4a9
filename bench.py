#!/usr/bin/env python
"""Benchmark of the descriptor-extraction + retrieval hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W              # configs[1] + configs[3]: the headline line
    python bench.py --config c3|c4|c5 ...                      # the other BASELINE configurations (one JSON line each)
    python bench.py --impl reference --gpus N ...              # the reference's CPU path (oracle port), rank 0 only
    python bench.py ... --dump-outputs DIR                     # also write the last timed step's outputs as DIR/<name>.npy

Default (config c2): a "step" = one pass of the extraction path over one batch: ResNet101-GeM descriptors of 64
synthetic 1024x1024 RGB images per GPU (random-init weights of that architecture, inputs resident in HBM).  `value` is
device-timed images/s (CUDA events, max over ranks); `e2e` is the same metric through the C-ABI host entry point (pinned
host images -> H2D -> forward -> D2H descriptors) with the copies inside the timed region.  `roofline` is computed from
launches timed INSIDE a sustained region of the same K steps (CUDA events on the launch stream around every kernel),
`roofline.traffic` is the measured DRAM traffic per launch of the same kernels (ncu, profiles/r2_traffic.json).  The
second half of BASELINE's metric (configs[3]: 1000 queries x 1M x 2048, k = 100, rows sharded over the GPUs, one
all-reduce of thresholds + one all-gather of per-shard top-k) is reported under "search" and, compactly, under
roofline.search.

  c3: 70 queries x 100k x 2048, PCA-whitening (p = 0.25) of the queries + similarity + top-k per step (HBM-bound).
  c4: the search half alone (1000 x 1M, sharded).
  c5: multi-scale extraction (scales 0.7 / 1.0 / 1.4 of 1024^2, resized on the GPU) and alpha-QE (k=2, alpha=0.5)
      search on the sharded 1M database.
Every GPU measurement on the line times --steps steps.  The inputs (images, weights, databases, queries) come from fixed
seeds, so two builds run with the same arguments can be compared output for output with --dump-outputs.
Prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

ARCH = "resnet101_rmac"
BATCH, SIZE = 64, 1024
SEARCH_N, SEARCH_Q, SEARCH_D, SEARCH_K = 1_000_000, 1000, 2048, 100
C3_N, C3_Q = 100_000, 70
CPU_THREADS = 16          # measured on the GPU host: torch CPU conv is fastest at 16 threads (128 logical cores)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--size", type=int, default=SIZE)
    ap.add_argument("--no-search", action="store_true", help="c2: skip the 1M-row search measurement")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="c2: skip the small-batch latency table")
    ap.add_argument("--no-peer", action="store_true", help="N > 1: exchange thresholds / lists with NCCL collectives instead of peer memory")
    ap.add_argument("--fuse-c23", type=int, default=-1, help="override the library default of option fuse_c23 (A/B runs)")
    ap.add_argument("--opt", action="append", default=[], help="library option KEY=VALUE for the network handle (A/B runs)")
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--host-chunk", type=int, default=0)
    ap.add_argument("--search-n", type=int, default=SEARCH_N)
    ap.add_argument("--search-q", type=int, default=SEARCH_Q)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what each timed path returned in its last step as DIR/<name>.npy "
                         "(float32 / float64, rank 0, at most 64 MB in all: larger outputs are cut to a seeded row sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    return args


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU while the timed region runs: NVML (a few ms per sample) when
    the bindings are importable, else nvidia-smi (tens of ms per sample)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    BITS = [0x8, 0x40, 0x20, 0x4]     # nvmlClocksEventReason{HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.source = index, [], False, "nvidia-smi"
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml, self.source = pynvml, "nvml"
        except Exception:
            self.nvml = None

    def _reasons_mask(self):
        for fn in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
            f = getattr(self.nvml, fn, None)
            if f is not None:
                try:
                    return int(f(self.handle))
                except Exception:
                    pass
        return 0

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    mhz = float(self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
                    mask = self._reasons_mask()
                    self.rows.append([mhz, self.max_mhz] + [bool(mask & b) for b in self.BITS])
                    time.sleep(0.02)      # (NVML queries contend with kernel launches: 4 ms polling slowed 1 ms search steps)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) == 6:
                    self.rows.append([float(parts[0]), float(parts[1])] + [p.lower().startswith("active") for p in parts[2:]])
            except Exception:
                pass
            time.sleep(0.05)

    def finish(self):
        self.stop_flag = True
        self.join(timeout=2)
        return self.summary()

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        sm = sorted(r[0] for r in self.rows)
        reasons = [n for j, n in enumerate(self.NAMES) if any(r[2 + j] for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.rows[0][1], "reasons": reasons,
                "samples": len(self.rows), "source": self.source}


# --------------------------------------------------------------------------------------------- CPU reference arm
def cpu_extract_rate(n_img, size, repeats):
    """The reference's CPU path for extraction = oracle port of net(imgs) (torch CPU fp32)."""
    import torch
    import synthdata as synth
    from oracle import dir_oracle as O
    torch.set_num_threads(min(CPU_THREADS, os.cpu_count() or 1))
    sd = synth.make_state_dict(ARCH, seed=0)
    x = synth.make_images(n_img, size, size, seed=1234, smooth=False)
    O.extract(x[:1, :, :256, :256], sd, ARCH)                 # warm-up (thread pool, oneDNN primitives)
    t0 = time.perf_counter()
    for _ in range(repeats):
        O.extract(x, sd, ARCH)
    dt = time.perf_counter() - t0
    return n_img * repeats / dt, dt / repeats, torch.get_num_threads()


def cpu_search_rate(n_db, n_q, dim, k, whiten=False, aqe=False):
    """The reference's CPU path for retrieval: (whiten_features, common.py:221-239) + np.dot scores (common.py:33) +
    per-query argsort (generic.py:207) (+ expand_descriptors and a second ranking, test_dir.py:24-44)."""
    import numpy as np
    from oracle import dir_oracle as O
    r = np.random.RandomState(0)
    db = r.standard_normal((n_db, dim)).astype(np.float32)
    db /= np.linalg.norm(db, axis=1, keepdims=True)
    q = r.standard_normal((n_q, dim)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    pca = None
    if whiten:
        import synthdata as synth
        pca = synth.make_pca(dim, seed=11)
    t0 = time.perf_counter()
    if whiten:
        q = O.whiten_features(q, pca, whitenp=0.25).astype(np.float32)
    if aqe:
        q = O.expand_descriptors(q, db=db, k=2, alpha=0.5).astype(np.float32)
    sc = np.dot(q, db.T)
    for i in range(n_q):
        np.argsort(sc[i])[::-1][:k]
    dt = time.perf_counter() - t0
    return n_q / dt, dt


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    steps = max(1, min(args.steps, 3))
    base = {"impl": "reference", "n_gpus": args.gpus, "steps": steps, "warmup": 1, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "gpu_launches": 0}
    if args.config in ("c3", "c4"):
        n, q = (C3_N, C3_Q) if args.config == "c3" else (100_000, 16)
        full_n = C3_N if args.config == "c3" else args.search_n
        rates = [cpu_search_rate(n, q, SEARCH_D, SEARCH_K, whiten=args.config == "c3") for _ in range(steps)]
        rate, dt = max(r[0] for r in rates) * n / full_n, min(r[1] for r in rates)
        sample = ("%d queries x %d x %d: %snp.dot + argsort (%.2f s)%s" %
                  (q, n, SEARCH_D, "whiten_features + " if args.config == "c3" else "", dt,
                   "" if n == full_n else ", scaled linearly to %d rows" % full_n))
        line = dict(base, metric="queries/sec", value=rate, unit="queries/s", ms_per_step=dt * 1e3,
                    config={"workload": workload_name(args.config, args), "queries_per_step": q},
                    cpu_baseline={"value": rate, "unit": "queries/s", "cores": os.cpu_count(), "kind": "port", "sample": sample},
                    e2e={"value": rate, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        print(json.dumps(line))
        return
    sample = 2
    n_scales = 3 if args.config == "c5" else 1
    if args.config == "c5":
        t0 = time.perf_counter()
        for sc in (0.7, 1.0, 1.4):
            cpu_extract_rate(1, int(0.5 + sc * args.size), 1)
        per_step = time.perf_counter() - t0
        rate, threads, sample = 1.0 / per_step, min(CPU_THREADS, os.cpu_count() or 1), 1
    else:
        rate, per_step, threads = cpu_extract_rate(sample, args.size, steps)
    qrate, qdt = cpu_search_rate(100_000, 16, SEARCH_D, SEARCH_K, aqe=args.config == "c5")
    line = dict(base, metric="descriptor images/sec", value=rate, unit="images/s", ms_per_step=per_step * 1e3,
                config={"workload": workload_name(args.config, args), "arch": ARCH, "images_per_step": sample, "scales": n_scales},
                cpu_baseline={"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
                              "sample": "%d image(s) of %dx%d%s per step through oracle/dir_oracle.py (torch CPU fp32, %d threads of %d logical cores)"
                                        % (sample, args.size, args.size, " at 3 scales" if n_scales == 3 else "", threads, os.cpu_count())},
                e2e={"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                search={"metric": "queries/sec", "value": qrate * 100_000 / SEARCH_N, "unit": "queries/s",
                        "sample": "16 queries x 100k x 2048 %snp.dot + argsort (%.2f s), scaled linearly to the 1M-row database"
                                  % ("alpha-QE + " if args.config == "c5" else "", qdt)})
    print(json.dumps(line))


def workload_name(config, args):
    return {
        "c2": "Resnet101-GeM descriptor extraction, batch %d x %dx%d synthetic RGB per GPU (BASELINE configs[1])" % (args.batch, args.size, args.size),
        "c3": "Resnet101-AP-GeM descriptors: %d queries x %d x %d database, whitening p=0.25 of the queries + similarity + top-%d (BASELINE configs[2])" % (C3_Q, C3_N, SEARCH_D, SEARCH_K),
        "c4": "%d queries x %d x %d database sharded row-wise over the GPUs, top-%d (BASELINE configs[3])" % (args.search_q, args.search_n, SEARCH_D, SEARCH_K),
        "c5": "multi-scale {0.7,1.0,1.4} Resnet101-GeM extraction of %dx%d images + alpha-QE (k=2, alpha=0.5) search on the sharded %d x %d database (BASELINE configs[4])" % (args.size, args.size, args.search_n, SEARCH_D),
    }[config]


# --------------------------------------------------------------------------------------------- our arm
class Ctx:
    """Distributed plumbing + measured peaks."""

    def __init__(self):
        import torch
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dist = None
        self.last = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        self.peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        self.peak_tf_burst = peaks.get("bf16_tflops", 1590.0)
        self.peak_gbs = peaks.get("hbm_gbs", 6650.0)
        self.peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        self.traffic = {}
        try:
            self.traffic = json.load(open(os.path.join(REPO, "profiles", "r2_traffic.json")))
        except Exception:
            pass

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.dist is None:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps):
        """K calls of fn bracketed by barrier + synchronize, CUDA events on the current stream, max over ranks -> ms/step.
        What the last call returned is left in self.last."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.last = fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def wall(self, fn, steps):
        """As timed(), on the host clock -> s/step."""
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.last = fn()
        self.barrier()
        return self.max_over_ranks(time.perf_counter() - t0) / steps


DUMP_BYTES = 64_000_000


def keep(dump, name, value):
    """Record an output of a timed path for --dump-outputs (dump is None when it was not asked for)."""
    if dump is not None:
        dump[name] = value


def write_outputs(path, arrays):
    """{name: tensor or array} -> path/<name>.npy: float64 for float64 and integer data (indices are exact below 2^53),
    float32 otherwise.  An array over its share of DUMP_BYTES keeps a fixed, seeded sample of its rows, taken on the
    device before the copy."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    budget = DUMP_BYTES // max(1, len(arrays)) - 4096          # 4 KB per file for the .npy header
    for name, a in arrays.items():
        a = torch.as_tensor(a)
        a = a.double() if a.dtype == torch.float64 or not a.is_floating_point() else a.float()
        if a.numel() * a.element_size() > budget:
            rows = budget // (a[0].numel() * a.element_size())
            pick = np.sort(np.random.RandomState(0).choice(a.shape[0], rows, replace=False))
            a = a[torch.from_numpy(pick).to(a.device)]
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy())


def make_net(args, ctx):
    import synthdata as synth
    from dirb200 import nets
    net = nets.create_model(ARCH)
    net.load_state_dict(synth.make_state_dict(ARCH, seed=0))
    net.eval()
    if args.chunk:
        net.set_backend_option("chunk", args.chunk)
    if args.host_chunk:
        net.set_backend_option("host_chunk", args.host_chunk)
    if args.fuse_c23 >= 0:
        net.set_backend_option("fuse_c23", args.fuse_c23)
    for kv in args.opt:
        k_, v_ = kv.split("=")
        net.set_backend_option(k_, float(v_))
    return net


def conv_roofline(net, ctx, steps, fwd):
    """Per launch-type CUDA-event timing accumulated over a sustained region of `steps` forwards."""
    torch = ctx.torch
    net.set_backend_option_live("profile", 2)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    p0.record()
    for _ in range(steps):
        fwd()
    p1.record()
    torch.cuda.synchronize()
    region_ms = p0.elapsed_time(p1) / steps
    table = net.profile_table()
    net.set_backend_option_live("profile", 0)
    conv = [r for r in table if r["cls"] == 0]
    ms = sum(r["ms"] for r in conv)
    fl = sum(r["flops"] for r in conv)
    by = sum(r["bytes"] for r in conv)
    n_l = sum(r["launches"] for r in conv)
    tot_ms = sum(r["ms"] for r in table)
    tf = fl / (ms * 1e-3) / 1e12 if ms else 0.0
    dom = max(conv, key=lambda r: r["ms"]) if conv else None
    tr = ctx.traffic.get("conv_stack", {})
    roof = {"bound": "tensor",
            "kernel": "conv_pers_kernel / conv_halo_kernel: all %d Bottleneck convolution launches of a step" % (n_l // max(1, steps)),
            "achieved": tf, "peak": ctx.peak_tf, "unit": "TFLOP/s", "frac": tf / ctx.peak_tf,
            "traffic": tr.get("dram_bytes_per_launch"), "traffic_source": tr.get("source"),
            "peak_source": ctx.peak_src + ", sustained dense 16-bit",
            "timed": "CUDA events around every launch, accumulated over %d consecutive steps (%.2f ms/step with the events)" % (steps, region_ms),
            "launches_per_step": n_l / max(1, steps), "avg_launch_ms": ms / max(1, n_l), "flops_per_launch": fl / max(1, n_l), "algorithmic_bytes_per_launch": by / max(1, n_l),
            "share_of_step": ms / tot_ms if tot_ms else None,
            "hbm_view": {"achieved_gbs": by / (ms * 1e-3) / 1e9 if ms else 0.0, "peak_gbs": ctx.peak_gbs,
                         "note": "algorithmic activation+weight bytes of the same launches / same time"}}
    if dom:
        d_tr = ctx.traffic.get("dominant", {})
        roof["dominant_launch_type"] = {
            "tag": dom["tag"], "launches_per_step": dom["launches"] / steps, "avg_ms": dom["ms"] / dom["launches"],
            "share_of_step": dom["ms"] / tot_ms, "tflops": dom["flops"] / (dom["ms"] * 1e-3) / 1e12,
            "algorithmic_gbs": dom["bytes"] / (dom["ms"] * 1e-3) / 1e9,
            "frac_of_bound": max(dom["flops"] / (dom["ms"] * 1e-3) / 1e12 / ctx.peak_tf, dom["bytes"] / (dom["ms"] * 1e-3) / 1e9 / ctx.peak_gbs),
            "traffic": d_tr.get("dram_bytes_per_launch"), "algorithmic_bytes": dom["bytes"] / dom["launches"]}
    roof["classes_ms_per_step"] = {}
    for r in table:
        key = ["conv_tcgen05", "stem_conv", "layout_maxpool", "head"][r["cls"]]
        roof["classes_ms_per_step"][key] = round(roof["classes_ms_per_step"].get(key, 0.0) + r["ms"] / steps, 4)
    layer_table = [{"tag": r["tag"], "launches": int(r["launches"] / steps), "ms_per_step": round(r["ms"] / steps, 4),
                    "tflops": round(r["flops"] / (r["ms"] * 1e-3) / 1e12, 1) if r["ms"] else 0.0,
                    "gbs": round(r["bytes"] / (r["ms"] * 1e-3) / 1e9, 1) if r["ms"] else 0.0} for r in table]
    return roof, layer_table, region_ms


def bench_extract(args, ctx, line, dump=None):
    import torch
    import synthdata as synth
    from dirb200 import ops
    world, rank, local = ctx.world, ctx.rank, ctx.local
    B, S = args.batch, args.size
    net = make_net(args, ctx)
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    u8 = torch.randint(0, 256, (B, 3, S, S), generator=g, device="cuda", dtype=torch.uint8)
    mean = torch.tensor(synth.RGB_MEANS, device="cuda").view(1, 3, 1, 1)
    std = torch.tensor(synth.RGB_STDS, device="cuda").view(1, 3, 1, 1)
    imgs = ((u8.float() / 255.0 - mean) / std).contiguous()
    del u8
    warmup = max(3, args.warmup)
    for _ in range(warmup):
        d = net.forward(imgs, want_f16=True)[0]
    torch.cuda.synchronize()
    assert bool(torch.isfinite(d).all()), "non-finite descriptors"
    launches_per_step, flops_per_step = net.last_launch_stats()

    sampler = ClockSampler(local)
    sampler.start()
    ms_per_step = ctx.timed(lambda: net.forward(imgs, want_f16=True), args.steps)
    clocks = sampler.finish()
    value = world * B / (ms_per_step * 1e-3)
    keep(dump, "descriptors", ctx.last[0])
    keep(dump, "descriptors_f16", ctx.last[1])

    # ---- roofline from launches timed inside a sustained region of the same K steps
    roof, layer_table, region_ms = conv_roofline(net, ctx, args.steps, lambda: net.forward(imgs, want_f16=True))
    # The per-launch events cost time themselves (a record between every two kernels also breaks the programmatic-dependent-
    # launch overlap): the instrumented region runs %-level slower than the timed K steps above.  Secondary figure: the
    # convolution launches' SHARE of the instrumented region applied to the un-instrumented step time.  `frac` stays the
    # instrumented (conservative) one.
    if roof.get("share_of_step") and roof.get("flops_per_launch"):
        conv_flops_step = roof["flops_per_launch"] * roof["launches_per_step"]
        if conv_flops_step > 0:
            conv_ms = ms_per_step * roof["share_of_step"]
            tf = conv_flops_step / (conv_ms * 1e-3) / 1e12
            roof["uninstrumented"] = {"achieved": tf, "frac": tf / ctx.peak_tf, "conv_ms_per_step": conv_ms,
                                      "instrumented_region_ms_per_step": region_ms, "timed_ms_per_step": ms_per_step,
                                      "note": "share of the convolution launches in the event-instrumented region x the timed step"}

    # ---- end to end through the C-ABI host entry point: pinned host images in, host descriptors out
    host = torch.empty((B, 3, S, S), dtype=torch.float32).pin_memory()
    host.copy_(imgs)
    e2e_steps = args.steps
    net.forward_host(host.numpy(), device=local)
    e2e_s = ctx.wall(lambda: net.forward_host(host.numpy(), device=local), e2e_steps)
    e2e_value = world * B / e2e_s
    keep(dump, "e2e_descriptors", ctx.last)
    host8 = torch.randint(0, 256, (B, S, S, 3), generator=torch.Generator().manual_seed(1234 + rank),
                          dtype=torch.uint8).pin_memory()
    net.forward_host_u8(host8.numpy(), device=local)
    e2e_u8 = world * B / ctx.wall(lambda: net.forward_host_u8(host8.numpy(), device=local), e2e_steps)
    keep(dump, "e2e_u8_descriptors", ctx.last)
    del host8, host

    line.update({
        "metric": "descriptor images/sec", "value": value, "unit": "images/s", "ms_per_step": ms_per_step,
        "dtype": "f16 operands, f32 accumulate",
        "config": {"workload": workload_name("c2", args), "arch": ARCH, "global_batch": world * B,
                   "parallelism": "image shards, dp%d, no collective" % world,
                   "l2": "inputs (%.0f MB/step) and activations exceed the 126 MB L2" % (B * 3 * S * S * 4 / 1e6),
                   "weights": "random init (synthdata.make_state_dict seed 0)"},
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": B * 3 * S * S * 4,
                "d2h_bytes_per_step": B * net.descriptor_dim * 4, "steps": e2e_steps,
                "api": "dirb200_net_forward_host (pinned host buffers, H2D of chunk i+1 overlaps compute of chunk i)",
                "uint8_input": {"value": e2e_u8, "unit": "images/s", "h2d_bytes_per_step": B * 3 * S * S,
                                "api": "dirb200_net_forward_host_u8 (uint8 HWC pixels, normalisation fused into the stem)"}},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks, "roofline": roof, "layer_table": layer_table,
        "step_tflops": flops_per_step / (ms_per_step * 1e-3) / 1e12,
    })
    # ---- small-batch latency (the reference's default evaluation mode is batch 1, test_dir.py:52-53,114)
    if not args.no_latency and rank == 0:
        lat = []
        for b in (1, 4, 8):
            x = imgs[:b].contiguous()
            for _ in range(3):
                net.forward(x)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_it = args.steps
            for _ in range(n_it):
                net.forward(x)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / n_it
            lat.append({"batch": b, "ms": round(dt * 1e3, 3), "images_per_s": round(b / dt, 1)})
        line["latency"] = {"size": "%dx%d" % (S, S), "rows": lat, "note": "net(imgs) wall clock incl. launch overhead, device-resident input"}
    return net, imgs


def make_db(ctx, n_rows, d, seed=99):
    import torch
    from dirb200 import ops
    from dirb200.dist import shard_rows
    s0, s1 = shard_rows(n_rows, ctx.world, ctx.rank)
    gen = torch.Generator(device="cuda").manual_seed(seed + ctx.rank)
    db = torch.randn((s1 - s0, d), generator=gen, device="cuda", dtype=torch.float32)
    db, db16 = ops.l2_normalize(db, want_f16=True)
    return db, db16, s0, s1


def bench_search(args, ctx, n_rows, n_q, aqe=False, whiten=False, dump=None, name="search"):
    """queries/s of the exact top-k search on the row-sharded database (optionally: PCA-whitening of the queries first,
    alpha query expansion = search + expand + search).  The last timed step's scores and indices go to dump as
    <name>_scores / <name>_indices."""
    import torch
    import synthdata as synth
    from dirb200 import ops
    from dirb200.dist import ShardedIndex
    world = ctx.world
    D, K = SEARCH_D, SEARCH_K
    db, db16, s0, s1 = make_db(ctx, n_rows, D)
    gq = torch.Generator(device="cuda").manual_seed(7)
    q = ops.l2_normalize(torch.randn((n_q, D), generator=gq, device="cuda", dtype=torch.float32))
    index = ShardedIndex(db, row_offset=s0, db16_local=db16)
    peer = world > 1 and not args.no_peer
    if peer:
        index.enable_peer_exchange(max_q=n_q, max_k=K)
    if whiten:
        pca = synth.make_pca(D, seed=11)
        import numpy as np
        comp = torch.from_numpy(np.ascontiguousarray(pca.components_, dtype=np.float32)).cuda()
        pmean = torch.from_numpy(np.ascontiguousarray(pca.mean_, dtype=np.float32)).cuda()
        pcs = torch.from_numpy((1.0 / np.power(pca.explained_variance_.astype(np.float64), 0.25)).astype(np.float32)).cuda()

    def step(qin=q):
        x = qin
        if whiten:
            x = ops.whiten(x, comp, pmean, pcs, l2norm=True)          # common.whiten_features(q, pca, whitenp=0.25)
        if aqe:
            x = index.expand_queries(x, 2, 0.5, check=False)          # test_dir.py:24-44 (search + expand)
        return index.search(x, K, check=False)

    for _ in range(3):
        step()
    index.check()
    ssteps = args.steps
    s_ms = ctx.timed(step, ssteps)
    index.check()
    keep(dump, name + "_scores", ctx.last[0])
    keep(dump, name + "_indices", ctx.last[1])
    # phase profile of one more search (CUDA events inside the library, same stream)
    index.local.set_option("profile", 1)
    step()
    index.check()
    prof = index.local.profile()
    index.local.set_option("profile", 0)
    st = index.local.stats()
    qh = q.cpu().pin_memory()

    def e2e_step():
        sc, ix = step(qh.cuda(non_blocking=True))
        index.check()
        return sc.cpu(), ix.cpu()
    e2e_step()
    s_e2e = ctx.wall(e2e_step, ssteps)
    passes = 2 if aqe else 1
    flops = passes * 2.0 * n_q * (n_rows + st["dense_rows"] * world) * D
    rows_local = s1 - s0
    filt_ms = prof.get("filter_gemm", 0.0)
    hbm_bytes = rows_local * D * 2 + n_q * D * 2 + n_q * K * 16
    tensor_bound = n_q >= 281
    tr = ctx.traffic.get("filter_gemm_%dq_%dk" % (n_q, rows_local // 1000), {})
    if tensor_bound:
        filt_tf = 2.0 * n_q * rows_local * D / (filt_ms * 1e-3) / 1e12 if filt_ms else 0.0
        roof = {"bound": "tensor", "kernel": "conv_pers_kernel<256,4,PERS_EPI_SIM_FILTER> (filter pass over this rank's %d rows)" % rows_local,
                "achieved": filt_tf, "peak": ctx.peak_tf_burst, "unit": "TFLOP/s", "frac": filt_tf / ctx.peak_tf_burst,
                "peak_source": ctx.peak_src + ", burst dense 16-bit (kernel timed alone inside the step)",
                "traffic": tr.get("dram_bytes_per_launch"), "algorithmic_bytes_per_launch": hbm_bytes,
                "launch_ms": filt_ms, "hbm_gbs": rows_local * D * 2 / (filt_ms * 1e-3) / 1e9 if filt_ms else 0.0,
                "whole_step_tflops_per_gpu": flops / world / (s_ms * 1e-3) / 1e12}
    else:
        gbs = hbm_bytes / (filt_ms * 1e-3) / 1e9 if filt_ms else 0.0
        roof = {"bound": "hbm", "kernel": "conv_pers_kernel<256,4,PERS_EPI_SIM_FILTER> (filter pass: the fp16 database is streamed once)",
                "achieved": gbs, "peak": ctx.peak_gbs, "unit": "GB/s", "frac": gbs / ctx.peak_gbs, "peak_source": ctx.peak_src,
                "traffic": tr.get("dram_bytes_per_launch"), "algorithmic_bytes_per_launch": hbm_bytes, "launch_ms": filt_ms,
                "whole_step_gbs": hbm_bytes * passes / (s_ms * 1e-3) / 1e9}
    out = {"metric": "queries/sec", "value": n_q / (s_ms * 1e-3), "unit": "queries/s", "ms_per_step": s_ms, "steps": ssteps,
           "config": {"workload": "%d queries x %d x %d fp16 database, k=%d, exact fp64 re-scoring%s%s" %
                                  (n_q, n_rows, D, K, ", whitening p=0.25 of the queries" if whiten else "",
                                   ", alpha-QE k=2 alpha=0.5 (two searches)" if aqe else ""),
                      "sharding": ("rows / %d ranks; per search %d B of thresholds and %d B of lists per rank are stored into every peer's "
                                   "exchange window over NVLink by the search kernels themselves (MIN + gather fused, no NCCL call)%s"
                                   if peer else "rows / %d ranks; per search one MIN all-reduce of %d B + one all-gather of %d B per rank%s") %
                                  (world, 4 * n_q, 16 * n_q * K, "; alpha-QE adds one SUM all-reduce of %d B" % (4 * n_q * D) if aqe else "")},
           "e2e": {"value": n_q / s_e2e, "unit": "queries/s", "h2d_bytes_per_step": n_q * D * 4, "d2h_bytes_per_step": n_q * K * 16},
           "roofline": roof, "phases_ms": {k: round(v, 4) for k, v in prof.items()}, "stats": st,
           "gpu_launches": st["launches"] * passes * ssteps}
    return out, db, index


def bench_whiten_block(ctx, db, D, steps, dump=None):
    import torch
    from dirb200 import ops
    gen = torch.Generator(device="cuda").manual_seed(5)
    wn = min(131072, db.shape[0])
    comp = torch.randn((D, D), generator=gen, device="cuda") / 45.0
    wmean = torch.zeros(D, device="cuda")
    wcs = torch.ones(D, device="cuda")
    x = db[:wn].contiguous()
    for _ in range(2):
        ops.whiten(x, comp, wmean, wcs)
    torch.cuda.synchronize()
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    for _ in range(steps):
        y = ops.whiten(x, comp, wmean, wcs)
    w1.record()
    torch.cuda.synchronize()
    w_ms = w0.elapsed_time(w1) / steps
    keep(dump, "whiten", y)
    return {"rows": wn, "ms": w_ms, "rows_per_s": wn / (w_ms * 1e-3), "tflops_algorithmic": 2.0 * wn * D * D / (w_ms * 1e-3) / 1e12,
            "note": "x-mean -> prescaled fp16 hi/lo split, 3 tcgen05 GEMM passes, column scale, row L2 (<= 2e-5 vs fp64)"}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    from dirb200 import ops
    ctx = Ctx()
    ops.require_gpu(ctx.local)
    world, rank = ctx.world, ctx.rank
    line = {"metric": None, "value": None, "unit": None, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": None, "data": "synthetic"}
    dump = {} if args.dump_outputs and rank == 0 else None

    if args.config == "c2":
        net, imgs = bench_extract(args, ctx, line, dump)
        if not args.no_search:
            del imgs
            net._release()
            torch.cuda.empty_cache()
            s, db, index = bench_search(args, ctx, args.search_n, args.search_q, dump=dump)
            s["metric"] = "1M-DB queries/sec"
            s["whiten"] = bench_whiten_block(ctx, db, SEARCH_D, args.steps, dump)
            line["search"] = s
            line["roofline"]["search"] = {"metric": s["metric"], "value": s["value"], "unit": s["unit"], "ms_per_step": s["ms_per_step"],
                                          "e2e": s["e2e"]["value"], "bound": s["roofline"]["bound"], "achieved": s["roofline"]["achieved"],
                                          "peak": s["roofline"]["peak"], "frac": s["roofline"]["frac"], "traffic": s["roofline"]["traffic"]}
            # The other two retrieval configurations of BASELINE.json, short forms of --config c5 / c3 on the same line:
            # alpha-QE (k=2, alpha=0.5: search + expand + search) on the 1M database, and 70 queries x 100k rows per GPU
            # with PCA-whitening p=0.25 (the HBM-bound search: the roofline is the filter pass against the copy peak).
            index.disable_peer_exchange()
            del s, db, index
            torch.cuda.empty_cache()
            sa, db, index = bench_search(args, ctx, args.search_n, args.search_q, aqe=True, dump=dump, name="search_aqe")
            line["roofline"]["search_aqe_c5"] = {"metric": "1M-DB alpha-QE queries/sec", "value": sa["value"], "unit": sa["unit"],
                                                 "ms_per_step": sa["ms_per_step"], "e2e": sa["e2e"]["value"], "config": sa["config"]}
            index.disable_peer_exchange()
            del sa, db, index
            torch.cuda.empty_cache()
            s3, db, index = bench_search(args, ctx, C3_N * world, C3_Q, whiten=True, dump=dump, name="search_c3")
            line["roofline"]["search_c3"] = {"metric": "queries/sec, 70 x 100k per GPU + whitening", "value": s3["value"], "unit": s3["unit"],
                                             "ms_per_step": s3["ms_per_step"], "e2e": s3["e2e"]["value"], "bound": s3["roofline"]["bound"],
                                             "achieved": s3["roofline"]["achieved"], "peak": s3["roofline"]["peak"], "unit_roofline": s3["roofline"]["unit"],
                                             "frac": s3["roofline"]["frac"], "traffic": s3["roofline"]["traffic"],
                                             "algorithmic_bytes_per_launch": s3["roofline"]["algorithmic_bytes_per_launch"],
                                             "launch_ms": s3["roofline"]["launch_ms"], "config": s3["config"]}
            index.disable_peer_exchange()
    elif args.config in ("c3", "c4"):
        sampler = ClockSampler(ctx.local)
        sampler.start()
        if args.config == "c3":
            s, db, index = bench_search(args, ctx, C3_N * world, C3_Q, whiten=True, dump=dump)
            line["scaling"] = "weak"
        else:
            s, db, index = bench_search(args, ctx, args.search_n, args.search_q, dump=dump)
            line["scaling"] = "strong"
        clocks = sampler.finish()
        line.update({"metric": "queries/sec", "value": s["value"], "unit": "queries/s", "ms_per_step": s["ms_per_step"], "steps": s["steps"],
                     "dtype": "f16 operands / f32 accumulate (filter), f64 (exact re-scoring)",
                     "config": dict(s["config"], workload=workload_name(args.config, args),
                                    l2="database shard (%.0f MB fp16) exceeds the 126 MB L2" % (db.shape[0] * SEARCH_D * 2 / 1e6)),
                     "e2e": s["e2e"], "roofline": s["roofline"], "gpu_launches": s["gpu_launches"], "clocks": clocks,
                     "phases_ms": s["phases_ms"], "stats": s["stats"]})
    else:   # c5
        import synthdata as synth
        net = make_net(args, ctx)
        B, S = min(args.batch, 16), args.size
        g = torch.Generator(device="cuda").manual_seed(4321 + rank)
        u8 = torch.randint(0, 256, (B, S, S, 3), generator=g, device="cuda", dtype=torch.uint8)
        fwd = lambda: net.forward_u8_multiscale(u8, scales=(0.7, 1.0, 1.4), pooling="gem", gemp=3)
        for _ in range(max(3, args.warmup)):
            d = fwd()
        torch.cuda.synchronize()
        assert bool(torch.isfinite(d).all())
        sampler = ClockSampler(ctx.local)
        sampler.start()
        ms = ctx.timed(fwd, args.steps)
        clocks = sampler.finish()
        keep(dump, "descriptors", ctx.last)
        roof, layer_table, _ = conv_roofline(net, ctx, args.steps, fwd)
        host8 = u8.cpu().pin_memory()

        def e2e():
            return fwd_host(net, host8)

        def fwd_host(net_, h8):
            out = net_.forward_u8_multiscale(h8.cuda(non_blocking=True), scales=(0.7, 1.0, 1.4), pooling="gem", gemp=3)
            return out.cpu()
        e2e()
        e2e_s = ctx.wall(e2e, args.steps)
        keep(dump, "e2e_descriptors", ctx.last)
        flops_img = (161.81 + 325.99 + 644.21) * (S / 1024.0) ** 2 * 1e9        # SURVEY 8d: R101 at 717 / 1024 / 1434
        line.update({"metric": "multi-scale descriptor images/sec", "value": world * B / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms,
                     "dtype": "f16 operands, f32 accumulate",
                     "config": {"workload": workload_name("c5", args), "arch": ARCH, "global_batch": world * B, "scales": [0.7, 1.0, 1.4],
                                "resize": "dirb200_resize_bilinear_u8 (byte-identical to PIL BILINEAR), uint8 input, normalisation fused into the stem",
                                "parallelism": "image shards, dp%d, no collective" % world,
                                "l2": "activations of every scale exceed the 126 MB L2"},
                     "e2e": {"value": world * B / e2e_s, "unit": "images/s", "h2d_bytes_per_step": B * S * S * 3, "d2h_bytes_per_step": B * net.descriptor_dim * 4},
                     "gpu_launches": net.last_launch_stats()[0] * 3 * args.steps, "clocks": clocks, "roofline": roof,
                     "step_tflops": B * flops_img / (ms * 1e-3) / 1e12})
        del u8
        net._release()
        torch.cuda.empty_cache()
        s, db, index = bench_search(args, ctx, args.search_n, args.search_q, aqe=True, dump=dump, name="search_aqe")
        s["metric"] = "1M-DB alpha-QE queries/sec"
        line["search"] = s
        line["roofline"]["search"] = {"metric": s["metric"], "value": s["value"], "unit": s["unit"], "ms_per_step": s["ms_per_step"],
                                      "e2e": s["e2e"]["value"], "frac": s["roofline"]["frac"]}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if args.config in ("c2", "c5"):
            rate, per_step, threads = cpu_extract_rate(2, args.size, 1)
            line["cpu_baseline"] = {"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
                                    "sample": "2 images of %dx%d through oracle/dir_oracle.py (torch CPU fp32, %d threads of %d logical cores)%s"
                                              % (args.size, args.size, threads, os.cpu_count(), "; single scale" if args.config == "c5" else "")}
            if "search" in line:
                qrate, qdt = cpu_search_rate(100_000, 16, SEARCH_D, SEARCH_K, aqe=args.config == "c5")
                line["search"]["cpu_baseline"] = {"value": qrate * 100_000 / args.search_n, "unit": "queries/s", "cores": os.cpu_count(), "kind": "port",
                                                  "sample": "16 queries x 100k x 2048 np.dot + argsort (%.2f s), scaled to %d rows" % (qdt, args.search_n)}
        else:
            n, q = (C3_N, C3_Q) if args.config == "c3" else (100_000, 16)
            full_n = C3_N if args.config == "c3" else args.search_n
            qrate, qdt = cpu_search_rate(n, q, SEARCH_D, SEARCH_K, whiten=args.config == "c3")
            line["cpu_baseline"] = {"value": qrate * n / full_n, "unit": "queries/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": "%d queries x %d x 2048 %snp.dot + argsort (%.2f s)%s" %
                                              (q, n, "whiten_features + " if args.config == "c3" else "", qdt,
                                               "" if n == full_n else ", scaled to %d rows" % full_n)}
    if rank == 0:
        print(json.dumps(line))
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    if "index" in locals():
        locals()["index"].disable_peer_exchange()      # unmap the peers' windows before any rank frees its own
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
