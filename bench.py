#!/usr/bin/env python
"""bench.py -- the BASELINE.json benchmarks of the B200 wavelet filter bank.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--gather]
                    [--dump-outputs DIR]

One "step" = one multi-level forward transform of one batch of synthetic data (per GPU).  Prints ONE JSON line (rank 0).

  --config 2  (default, the headline)  wavedec2  db4  level 4  reflect   64 x 4096 x 4096      float32
  --config 3                           wavedec3  sym4 level 3  zero       8 x 256 x 256 x 256  float32
  --config 4                           MatrixWavedec db6 level None (12) 1024 x 65536          float64
  --config 5                           wavedec2  db8  level 5  reflect  512 x 2048 x 2048      float32 per GPU
                                       (4096 images over 8 GPUs); --gather adds the NCCL collection of the shards

See DESIGN.md section "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

CONFIGS = {
    2: dict(kind="2d", wavelet="db4", level=4, mode="reflect", shape=(64, 4096, 4096), dtype="f32", cpu_batch=8,
            metric="Msamples/s, wavedec2 db4 L4 4096x4096 fp32 (forward)", baseline_cfg="BASELINE.json configs[1]",
            kernel="fwd2d_strip_f32_kernel<8,64,TMA> (level-1 launch)", kernel_level=1),
    3: dict(kind="3d", wavelet="sym4", level=3, mode="zero", shape=(8, 256, 256, 256), dtype="f32", cpu_batch=2,
            metric="Msamples/s, wavedec3 sym4 L3 256^3 fp32 (forward)", baseline_cfg="BASELINE.json configs[2]",
            kernel="fwd3d_tile_kernel<8> (level-1 launch)", kernel_level=1),
    4: dict(kind="matrix", wavelet="db6", level=None, mode="zero", shape=(1024, 65536), dtype="f64", cpu_batch=16,
            metric="Msamples/s, MatrixWavedec db6 65536 fp64 (forward)", baseline_cfg="BASELINE.json configs[3]",
            kernel="mat_fwd_dmma2_kernel<12,128> (FP64 tensor cores; first launch = levels 1 + 2)", kernel_level=2),
    5: dict(kind="2d", wavelet="db8", level=5, mode="reflect", shape=(512, 2048, 2048), dtype="f32", cpu_batch=8,
            metric="Msamples/s, wavedec2 db8 L5 2048x2048 fp32 (forward)", baseline_cfg="BASELINE.json configs[4]",
            kernel="fwd2d_strip_f32_kernel<16,64,TMA> (level-1 launch)", kernel_level=1),
}
DT = {"f32": torch.float32, "f64": torch.float64}


# --------------------------------------------------------------------------------------------------------------
# the transforms of one configuration, for our package and for any module with the reference's API
# --------------------------------------------------------------------------------------------------------------
def flat(coeffs):
    out = []
    for el in coeffs:
        if isinstance(el, torch.Tensor):
            out.append(el)
        elif isinstance(el, dict):
            out.extend(el[k] for k in sorted(el))
        else:
            out.extend(el)
    return out


def make_forward(mod, cfg, level="cfg"):
    lev = cfg["level"] if level == "cfg" else level
    if cfg["kind"] == "2d":
        return lambda x: mod.wavedec2(x, cfg["wavelet"], mode=cfg["mode"], level=lev)
    if cfg["kind"] == "3d":
        return lambda x: mod.wavedec3(x, cfg["wavelet"], mode=cfg["mode"], level=lev)
    op = mod.MatrixWavedec(cfg["wavelet"], lev)
    return lambda x: op(x)


def make_inverse(mod, cfg):
    if cfg["kind"] == "2d":
        return lambda c: mod.waverec2(c, cfg["wavelet"])
    if cfg["kind"] == "3d":
        return lambda c: mod.waverec3(c, cfg["wavelet"])
    op = mod.MatrixWaverec(cfg["wavelet"])
    return lambda c: op(c)


def named_outputs(coeffs) -> dict:
    """{name: tensor} of a coefficient list [approx, coarsest detail, ..., level-1 detail] as a caller receives it."""
    top = len(coeffs) - 1
    out = {"approx": coeffs[0]}
    for i, el in enumerate(coeffs[1:]):
        lev = f"detail_level{top - i}"
        if isinstance(el, torch.Tensor):
            out[lev] = el
        elif isinstance(el, dict):
            out.update((f"{lev}_{k}", el[k]) for k in sorted(el))
        else:
            out.update((f"{lev}_{k}", t) for k, t in zip(el._fields, el))
    return out


#: bound on what --dump-outputs writes (bytes of array data)
DUMP_BYTES = 60 * 10**6


def dump_outputs(coeffs, directory: str) -> None:
    """Write every returned array as <directory>/<name>.npy (its own float dtype).  When all of them together exceed
    DUMP_BYTES, each one is cut to a fixed sample of its elements -- the same positions for the same shapes in every
    run (seed 0), flattened in index order -- taking the same share of every array."""
    import numpy as np

    named = named_outputs(coeffs)
    total = sum(t.numel() * t.element_size() for t in named.values())
    share = min(1.0, DUMP_BYTES / total)
    os.makedirs(directory, exist_ok=True)
    for name, t in named.items():
        if share < 1.0:
            g = torch.Generator().manual_seed(0)
            k = max(int(t.numel() * share), 1)
            flat_idx = torch.randint(t.numel(), (k,), generator=g).unique().to(t.device)
            t = t[torch.unravel_index(flat_idx, t.shape)]
        np.save(os.path.join(directory, f"{name}.npy"), t.detach().cpu().numpy())


def nbytes(ts) -> int:
    return sum(t.numel() * t.element_size() for t in ts)


def samples_of(shape) -> int:
    n = 1
    for s in shape:
        n *= s
    return n


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe).  The sampler is started
    while the GPU is still idle (nvidia-smi needs a few hundred ms to come up, longer on an 8-GPU box; no load is added
    before the timed region: a long pre-load pushes the part into its 1 kW power cap, 1965 -> ~1630 MHz) and the samples
    are cut to the timed window by their timestamps; if the window is shorter than the sampling period, all samples since
    the start are used and the record says so."""

    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines: list[tuple[float, str]] = []
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def window_begin(self):
        self.t0 = time.time()

    def window_end(self):
        self.t1 = time.time()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()

        def parse(rows):
            sm, mx, reasons = [], [], set()
            for _, ln in rows:
                f = [v.strip() for v in ln.split(",")]
                if len(f) < 10:
                    continue
                try:
                    sm.append(float(f[2]))
                    mx.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[6:10]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            sm.sort()
            return sm, mx, reasons

        inside = [r for r in self.lines if self.t0 is not None and self.t0 - 0.01 <= r[0] <= (self.t1 or 1e30) + 0.03]
        window = "timed region"
        sm, mx, reasons = parse(inside)
        if not sm:
            window = "start of the run .. timed region (the timed region is shorter than the sampling period)"
            sm, mx, reasons = parse(self.lines)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def measured_peak_gbs() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------------------------
# the reference on the host cores
# --------------------------------------------------------------------------------------------------------------
def reference_module():
    """(module, kind): the UNMODIFIED reference from oracle/_ref when it was installed there (oracle/make_ref.py),
    else the oracle port (the reference's own torch-CPU operator sequence, pinned bit-identical to it)."""
    try:
        from oracle.make_ref import import_ref

        mod = import_ref()
        if mod is not None:
            return mod, "reference", "unmodified reference (oracle/_ref/ptwt, pywt shim for the filter taps)"
    except Exception:  # noqa: BLE001
        pass
    from oracle import ptwt_port as P

    return P, "port", "oracle/ptwt_port.py (the reference's F.pad + conv(stride 2) / sparse.mm operator sequence)"


def cpu_reference(cfg, sample_batch: int, reps: int, warm: int = 1):
    """Msamples/s of the reference forward transform on the host cores, best thread count among {all, half, 32}."""
    mod, kind, what = reference_module()
    ncpu = os.cpu_count() or 1
    g = torch.Generator().manual_seed(1234)
    x = torch.randn((sample_batch,) + tuple(cfg["shape"][1:]), generator=g, dtype=DT[cfg["dtype"]])
    fwd = make_forward(mod, cfg)
    build_s = None
    if cfg["kind"] == "matrix":
        t0 = time.perf_counter()
        fwd(x[:1])            # one-time operator construction of the reference (reported separately)
        build_s = time.perf_counter() - t0
    best, best_cores, times = float("inf"), ncpu, []
    for cores in sorted({ncpu, max(ncpu // 2, 1), min(32, ncpu)}, reverse=True):
        torch.set_num_threads(cores)
        for _ in range(warm):
            fwd(x[:1])
        for _ in range(reps):
            t0 = time.perf_counter()
            fwd(x)
            dt = time.perf_counter() - t0
            times.append(dt)
            if dt < best:
                best, best_cores = dt, cores
    torch.set_num_threads(best_cores)
    val = samples_of(x.shape) / best / 1e6
    info = {"value": val, "unit": "Msamples/s", "cores": best_cores, "kind": kind,
            "sample": f"{sample_batch} items of {tuple(cfg['shape'][1:])} {cfg['dtype']}, best of {len(times)} "
                      f"({', '.join(f'{t:.3f}s' for t in times[:6])}); {what}"}
    if build_s is not None:
        info["operator_build_s"] = build_s
    return info, mod, x, best_cores


def run_reference(args, cfg) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(args.steps, 1), max(args.warmup, 1)
    sample = args.cpu_batch or cfg["cpu_batch"]
    info, mod, x, cores = cpu_reference(cfg, sample, 1)
    fwd = make_forward(mod, cfg)
    for _ in range(warmup):
        fwd(x)
    t0 = time.perf_counter()
    for _ in range(steps):
        fwd(x)
    dt = (time.perf_counter() - t0) / steps
    val = samples_of(x.shape) / dt / 1e6
    info = dict(info, value=val, cores=cores)
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": val, "unit": "Msamples/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic (torch.randn, seed 1234)",
        "config": {"workload": f"{describe(cfg, sample)} per step (bounded sample of the {cfg['shape'][0]}-item batch) "
                               f"on the host CPU, {cfg['baseline_cfg']}"},
        "cpu_baseline": info,
        "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def describe(cfg, batch) -> str:
    name = {"2d": "wavedec2", "3d": "wavedec3", "matrix": "MatrixWavedec"}[cfg["kind"]]
    shp = "x".join(str(s) for s in cfg["shape"][1:])
    extra = "" if cfg["kind"] == "matrix" else f" mode={cfg['mode']}"
    return f"{name} {cfg['wavelet']} level={cfg['level']}{extra}, batch {batch} x {shp} {cfg['dtype']}"


# --------------------------------------------------------------------------------------------------------------
# host placement: each rank on the NUMA node of its GPU, before the first pinned allocation
# --------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(local: int) -> dict:
    info = {"bound": False}
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bdf}/numa_node").read_text().strip())
        info.update(pci=bdf, numa_node=node)
        if node < 0:
            return info
        cpus: set[int] = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info.update(bound=True, cpus=len(allowed))
    except Exception as ex:  # noqa: BLE001
        info["error"] = f"{type(ex).__name__}: {str(ex)[:80]}"
    return info


def host_link_probe(dev, seconds: float = 0.6) -> dict:
    """Pinned-memory copies in BOTH directions at once, no compute: the ceiling of the end-to-end number on this
    host (all ranks run it at the same time)."""
    n = 256 << 20
    hin = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    hout = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    din = torch.empty(n, dtype=torch.uint8, device=dev)
    dout = torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    torch.cuda.synchronize(dev)
    reps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        with torch.cuda.stream(s1):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s2):
            hout.copy_(dout, non_blocking=True)
        s1.synchronize()
        s2.synchronize()
        reps += 1
    dt = time.perf_counter() - t0
    return {"h2d_plus_d2h_gbs": 2 * n * reps / dt / 1e9, "seconds": dt}


def _dbg(msg: str) -> None:
    if os.environ.get("BENCH_DEBUG"):
        print(f"[bench rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="items per GPU per step (default: the BASELINE configuration)")
    ap.add_argument("--cpu-batch", type=int, default=0, help="items in the CPU-baseline sample")
    ap.add_argument("--gather", action="store_true", help="config 5: also time the NCCL collection of the shards")
    ap.add_argument("--gather-chunks", type=int, default=4)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-numa", action="store_true")
    ap.add_argument("--no-incumbent", action="store_true", help="skip timing the reference algorithm on the GPU")
    ap.add_argument("--incumbent-batch", type=int, default=16)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the coefficients of the last timed step to DIR/<name>.npy (a fixed sample beyond 60 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg)
        return

    import pytorch_wavelet_toolbox_b200 as wt
    from pytorch_wavelet_toolbox_b200 import _native

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    numa = {"bound": False, "skipped": True} if args.no_numa else bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        # NCCL announces its version on stdout at the first collective: keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v: float) -> float:
        if dist is None:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    _dbg("process group up")
    sampler = ClockSampler(local)
    sampler.start()                            # nvidia-smi needs a few hundred ms to come up: start it while the GPU is idle
    B = args.batch or cfg["shape"][0]
    shape = (B,) + tuple(cfg["shape"][1:])
    dtype = DT[cfg["dtype"]]
    n_samples = samples_of(shape)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.randn(shape, generator=g, device=dev, dtype=dtype)
    fwd = make_forward(wt, cfg)
    inv = make_inverse(wt, cfg)

    for _ in range(max(args.warmup, 3)):
        out = fwd(x)
    alg = nbytes([x]) + nbytes(flat(out))     # algorithmic bytes: input read once + every returned coefficient written once
    d2h_bytes = nbytes(flat(out))
    del out
    torch.cuda.synchronize(dev)

    _dbg("warm-up done")
    _native.launch_count_reset()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    sampler.window_begin()
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for i in range(args.steps):
        ev[i][0].record()
        out = fwd(x)
        ev[i][1].record()
    t_end.record()
    barrier()
    sampler.window_end()
    clocks = sampler.stop()
    launches = _native.launch_count()
    total_ms = max_over_ranks(t_start.elapsed_time(t_end))
    step_ms = sorted(a.elapsed_time(b) for a, b in ev)
    ms_per_step = total_ms / args.steps
    value = world * n_samples / (ms_per_step * 1e-3) / 1e6

    _dbg("timed region done")
    # parity of what was just timed against the oracle, outside the timed region: items from BOTH halves of the batch
    # (the second half runs on the library's auxiliary stream with reused scratch slots in the 2-D analysis)
    parity = None
    if rank == 0:
        from oracle import ptwt_port as P

        # matrix configuration: the port materialises the dense n x n operator before sparsifying it (34 GB at
        # n = 65536); the unmodified reference builds the same operator sparsely (slow Python, little memory)
        pmod = reference_module()[0] if cfg["kind"] == "matrix" else P
        ofwd = make_forward(pmod, cfg)
        items = sorted({0, B // 2 - 1, B // 2, B - 1} & set(range(B)))
        fg = flat(out)
        worst = 0.0
        for i in items:
            want = flat(ofwd(x[i:i + 1].cpu()))
            scale = max(float(t.abs().max()) for t in want)
            worst = max(worst, max(float((a[i:i + 1].cpu() - b).abs().max()) for a, b in zip(fg, want)) / scale)
        parity = {"max_rel_err_vs_oracle": worst, "items_checked": items,
                  "tolerance": 1e-5 if dtype == torch.float32 else 1e-11}
        if args.dump_outputs:
            dump_outputs(out, args.dump_outputs)
    del out

    _dbg("parity done")
    # roofline of the dominant kernel: timed alone with CUDA events on the launching stream (a transform with
    # level = kernel_level is exactly that launch); achieved = its algorithmic bytes / its average duration
    peak, peak_src = measured_peak_gbs()
    med_ms = step_ms[len(step_ms) // 2]
    step_achieved = alg / (med_ms * 1e-3) / 1e9
    kfwd = make_forward(wt, cfg, level=cfg["kernel_level"])
    for _ in range(3):
        ko = kfwd(x)
    alg_k = nbytes([x]) + nbytes(flat(ko))
    del ko
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    _native.launch_count_reset()
    k0.record()
    for _ in range(20):
        kfwd(x)
    k1.record()
    torch.cuda.synchronize(dev)
    k_launches = _native.launch_count()
    k_ms = k0.elapsed_time(k1) / 20
    achieved = alg_k / (k_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tf = ROOT / "profiles" / "traffic.json"
    if tf.exists():
        try:
            tj = json.loads(tf.read_text())
            traffic = tj.get(f"config{args.config}", {}).get("dominant_kernel_dram_bytes_per_launch")
            if traffic is None and args.config == 2:
                traffic = tj.get("dominant_kernel_dram_bytes_per_launch")
            traffic_src = "static: one ncu --set full capture kept in profiles/traffic.json (not re-measured by this run)"
        except Exception:  # noqa: BLE001
            traffic = None

    _dbg("kernel timing done")
    # inverse transform of the same coefficients (reported separately, SURVEY.md section 8d)
    coeffs = fwd(x)
    for _ in range(3):
        rec = inv(coeffs)
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    i0.record()
    for _ in range(10):
        rec = inv(coeffs)
    i1.record()
    torch.cuda.synchronize(dev)
    inv_ms = i0.elapsed_time(i1) / 10
    sl = (slice(0, 2),) + tuple(slice(0, s) for s in shape[1:])
    rt_err = float((rec[sl] - x[:2]).abs().max())
    inverse = {"ms_per_step": inv_ms, "value": n_samples / (inv_ms * 1e-3) / 1e6, "unit": "Msamples/s (per GPU)",
               "step_frac": alg / (inv_ms * 1e-3) / 1e9 / peak, "round_trip_max_abs_err": rt_err}
    del rec

    _dbg("inverse done")
    # the NCCL collection of the shards (SURVEY 8e): ONE all_gather of the already packed coefficient buffer per chunk,
    # issued on a second stream so that chunk k travels while chunk k+1 is transformed
    gather = None
    if args.gather and dist is not None:
        from pytorch_wavelet_toolbox_b200 import sharding

        del coeffs
        torch.cuda.empty_cache()
        res = sharding.transform_and_gather(fwd, x, chunks=args.gather_chunks)   # warm-up (NCCL buffers, allocator)
        gathered_bytes = sum(nbytes(flat(c)) for c in res)
        del res
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        nrep = max(min(args.steps, 5), 1)
        for _ in range(nrep):
            res = sharding.transform_and_gather(fwd, x, chunks=args.gather_chunks)
            del res
        g1.record()
        barrier()
        g_ms = max_over_ranks(g0.elapsed_time(g1) / nrep)
        gather = {"ms_per_step": g_ms, "value": world * n_samples / (g_ms * 1e-3) / 1e6, "unit": "Msamples/s",
                  "chunks": args.gather_chunks, "bytes_received_per_rank": gathered_bytes,
                  "what": "transform + one all_gather_into_tensor of the packed coefficient buffer per chunk, "
                          "overlapped on a second stream; every rank ends with all coefficients"}
    else:
        del coeffs

    _dbg("gather done")
    # end to end through the public API with HOST (pinned) buffers: H2D + transform + D2H every step
    e2e, link = None, None
    if not args.no_e2e:
        torch.cuda.empty_cache()
        link = host_link_probe(dev)
        link["h2d_plus_d2h_gbs_min_over_ranks"] = -max_over_ranks(-link["h2d_plus_d2h_gbs"])
        xh = torch.empty(shape, dtype=dtype, pin_memory=True)
        xh.copy_(x)
        with wt.host_staging(reuse=True):
            for _ in range(2):
                oh = fwd(xh)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                oh = fwd(xh)
            torch.cuda.synchronize(dev)
            dt = max_over_ranks((time.perf_counter() - t0) / args.e2e_steps)
        e2e = {"value": world * n_samples / dt / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": nbytes([xh]),
               "d2h_bytes_per_step": d2h_bytes, "ms_per_step": dt * 1e3,
               "staging": "pinned host output buffer reused across steps (wt.host_staging(reuse=True))"}
        del oh, xh

    _dbg("e2e done")
    # the incumbent on this GPU: the reference's own algorithm executed by torch/cuDNN on the same device -- what ptwt
    # does today when it is handed CUDA tensors.  Informational: a sample of the batch, device-resident, CUDA events.
    incumbent = None
    if rank == 0 and not args.no_incumbent and cfg["kind"] != "matrix":
        try:
            from oracle import ptwt_port as P

            nb = min(args.incumbent_batch, B)
            xs = x[:nb]
            ifwd = make_forward(P, cfg)
            for _ in range(2):
                ref_c = ifwd(xs)
            torch.cuda.synchronize(dev)
            j0, j1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            j0.record()
            for _ in range(3):
                ref_c = ifwd(xs)
            j1.record()
            torch.cuda.synchronize(dev)
            inc_ms = j0.elapsed_time(j1) / 3
            incumbent = {"value": samples_of(xs.shape) / (inc_ms * 1e-3) / 1e6, "unit": "Msamples/s (1 GPU)", "ms": inc_ms,
                         "sample": f"{nb} items, device resident",
                         "step_frac": alg * nb / B / (inc_ms * 1e-3) / 1e9 / peak,
                         "what": "reference algorithm (F.pad + conv stride 2, torch/cuDNN) on the same B200"}
            del ref_c, xs
            torch.cuda.empty_cache()
        except Exception as ex:  # noqa: BLE001
            incumbent = {"unavailable": f"{type(ex).__name__}: {str(ex)[:160]}"}

    cpu = None
    if rank == 0 and not args.no_cpu:
        cpu, _, _, _ = cpu_reference(cfg, args.cpu_batch or cfg["cpu_batch"], 3)

    _dbg("assembling the line")
    if rank == 0:
        in_mb, out_mb = nbytes([x]) / 1e6, d2h_bytes / 1e6
        line = {
            "metric": cfg["metric"], "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic (torch.randn on device, seed 1234+rank)",
            "config": {"workload": f"{describe(cfg, B)} per GPU ({cfg['baseline_cfg']})",
                       "l2": f"inputs ({in_mb:.0f} MB) and outputs ({out_mb:.0f} MB) exceed the 126 MB L2; no flush needed",
                       "parallelism": f"batch-sharded x{world}, no data-path collective"
                                      + (" (+ all_gather of the results, reported under 'gather')" if gather else ""),
                       "numa": numa},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": cfg["kernel"],
                         "kernel_algorithmic_bytes_per_launch": alg_k, "kernel_ms_per_launch": k_ms,
                         "kernel_launches_timed": int(k_launches),
                         "step_achieved": step_achieved, "step_frac": step_achieved / peak,
                         "algorithmic_bytes_per_step": alg, "median_step_ms": med_ms, "min_step_ms": step_ms[0]},
            "cpu_baseline": cpu, "e2e": e2e, "host_link": link, "inverse": inverse, "gather": gather,
            "incumbent_gpu": incumbent, "gpu_launches": int(launches), "clocks": clocks, "parity": parity,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
