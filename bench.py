#!/usr/bin/env python
"""bench.py -- headline benchmark of zignal_b200 (contract: see the task statement / DESIGN.md "Measurement").

Workload (BASELINE.json configs[1]): 15x15 separable Gaussian blur (sigma = 2.25, mirror border, the taps
`Image.gaussianBlur` computes) on 8192 x 8192 RGBA f32.  A "step" is one blur.

  N = 1   one zb_gaussian_blur-equivalent call on the device-resident image.
  N > 1   one process per GPU, everything through the C ABI's zb_shard_* entry points: the image is a stack of row blocks, one
          per rank, and a step is ONE kernel launch per rank -- the fused convolution kernel copies the 7 edge rows of its row
          neighbours from their memory over NVLink (CUDA IPC mappings) in its own prologue and synchronises with them through
          flags; there is no separate exchange.  Two partitionings are timed in the same run:
            weak   (the headline `value`, "scaling": "weak"): 8192 rows per GPU, the image is (N*8192) x 8192;
            strong (`extra.strong`): THE 8192 x 8192 image split into 8192/N rows per GPU.
          After the timed region every rank checks its block of the result against a single-GPU blur of (its block + the true
          neighbour rows, fetched through torch.distributed, not through the library) and the line carries `parity`.

  value      : Mpixels/s, whole job, inputs resident in HBM, timed with CUDA events (max over ranks)
  e2e        : the same metric through the host-pointer C-ABI entry point (pinned, NUMA-local host buffers; H2D of the input and
               D2H of the result inside the timed region).  N > 1: every rank's host buffer holds its row block plus the 7
               overlapping rows of its neighbours (SURVEY 8(e): no exchange needed when shards are uploaded with overlap)
  roofline   : algorithmic bytes (read once + write once = 32 B/px) / step time vs the measured HBM peak
  cpu_baseline: the CPU oracle port (the reference's algorithm, 4 planar Image(f32) convolutions) on rank 0
  extra      : the other BASELINE configs, timed in the same process (C3 bicubic 16384^2 -> 4096^2 Rgb at N = 1; C4 rotate batch and
               C5 fdm.update at every N, sharded over the ranks)

`--impl reference` times the reference's own CPU implementation of the path instead (the C++ port under oracle/: the Zig
reference cannot be built in this image) with all host threads, pinned (OMP_PROC_BIND=close) and first-touch placed, on the
full 8192 x 8192 image.

`--steps` sets the number of timed steps of every timed loop: the blur (weak and strong), e2e, each extra config and the
`--impl reference` arm.  Only `cpu_baseline` keeps its best of 2 single-threaded passes (about 4 s each).

`--dump-outputs DIR` writes DIR/gaussian_blur.npy: 256 rows of the image the headline's last timed step wrote (the weak or the strong
partitioning, as `--scaling` picks at N > 1; every block's first and last 8 rows and a seeded choice of interior rows), and their row
numbers in that image as DIR/gaussian_blur_rows.npy, so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

ROWS = COLS = 8192
SIGMA = 2.25
HALO = 7
METRIC = "Mpixels/sec Gaussian-blur 8K RGBA f32"
WORKLOAD = "gaussian_blur_15x15_sigma2.25_mirror_8192x8192_rgba_f32"
ALGO_BYTES_PER_PX = 32  # read 16 B + write 16 B (SURVEY.md 8d)
DUMP_ROWS = 256  # --dump-outputs: 256 x 8192 RGBA f32 = 32 MiB


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def bind_to_gpu_numa(index: int):
    """Run this process (and place its host memory: first touch) on the NUMA node the GPU hangs off.  Best effort; returns a
    description for the JSON line."""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=20).stdout.strip()
        bus = out.lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA affinity reported"}
        cpulist = Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus:
            return {"numa_node": node, "note": "node's CPUs not in the allowed set"}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:  # noqa: BLE001
        return {"numa_node": None, "note": f"unavailable: {type(e).__name__}"}


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons while the GPU is under load."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        loaded = [s for s in self.samples if s[6].isdigit() and int(s[6]) >= 50] or self.samples
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": len(self.samples), "samples_under_load": len(loaded)}
        try:
            out["sm_mhz"] = float(np.median([float(s[0]) for s in loaded]))
            out["sm_max_mhz"] = float(loaded[0][1])
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for i, n in enumerate(names):
                if any(s[2 + i].lower().startswith("active") for s in loaded):
                    out["reasons"].append(n)
        except Exception:
            pass
        return out


def cpu_reference_pass(zo, planes, outs, taps, threads):
    """One pass of the reference's CPU path for this workload: Image(f32).convolveSeparable on each of the 4 channel
    planes (the only form the reference accepts for float data, convolution.zig:322-436)."""
    zo.set_threads(threads)
    t0 = time.perf_counter()
    for p, o in zip(planes, outs):
        zo.conv_separable(p, taps, taps, "mirror", out=o)
    return time.perf_counter() - t0


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation (oracle port), all host threads, rank 0 only."""
    if rank != 0:
        return
    # thread placement must be decided before libgomp starts: threads pinned to cores, neighbours in rank order
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle_lib as zo
    threads = zo.hw_threads()
    zo.set_threads(threads)
    # the full 8192 x 8192 image as 4 planes; np.empty does not touch the pages, the parallel fill does (first touch = the thread
    # that will convolve those rows), and a warm-up pass places the outputs and the oracle's temp plane the same way
    planes = [zo.parallel_fill_f32(np.empty((ROWS, COLS), np.float32), 2 + k) for k in range(4)]
    outs = [np.empty((ROWS, COLS), np.float32) for _ in range(4)]
    taps = zo.gaussian_taps(SIGMA)
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_reference_pass(zo, planes, outs, taps, threads)
    steps = args.steps
    times = [cpu_reference_pass(zo, planes, outs, taps, threads) for _ in range(steps)]
    ms = float(np.mean(times)) * 1e3
    mpx = ROWS * COLS / 1e6 / (ms * 1e-3)
    line = {
        "impl": "reference", "metric": METRIC, "value": mpx, "unit": "Mpixels/s", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": ms, "ms_per_step_min": float(np.min(times)) * 1e3, "ms_per_step_max": float(np.max(times)) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": f"the full {ROWS}x{COLS} image per step", "same_config": True,
                   "parallelism": f"cpu{threads} (OpenMP rows, OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND')}, first-touch placed)"},
        "cpu_baseline": {"value": mpx, "unit": "Mpixels/s", "cores": threads, "kind": "port",
                         "sample": f"{ROWS}x{COLS} RGBA f32 as 4 planar Image(f32) convolutions, {steps} passes, OpenMP row-parallel, pinned threads"},
        "e2e": {"value": mpx, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def time_steps(torch, dist, world, dev, fn, steps, warmup):
    """W warm-up calls, then `steps` calls between two events on the current stream, barrier + synchronize on both sides, max over ranks.
    Returns ms per step."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps


def dump_outputs(torch, dist, rank, world, block, out_dir):
    """--dump-outputs: rows of the blurred image gathered on rank 0 in rank order, written as DIR/gaussian_blur.npy (DUMP_ROWS x COLS x 4
    f32) and their row numbers in the whole image as DIR/gaussian_blur_rows.npy (f64, exact for integers).  The rows are every rank's
    first and last 8 rows, which read the mirror border or a neighbour's rows, and a seeded choice of its interior rows."""
    rows = block.shape[0]
    inner = np.random.default_rng(0).choice(np.arange(8, rows - 8), max(DUMP_ROWS // world - 16, 0), replace=False)
    idx = np.concatenate([np.arange(8), np.sort(inner), np.arange(rows - 8, rows)])
    s = block[torch.from_numpy(idx).to(block.device)].contiguous()
    if world > 1:
        parts = [torch.empty_like(s) for _ in range(world)]
        dist.all_gather(parts, s)
        s = torch.cat(parts)
    if rank == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
        np.save(out_dir / "gaussian_blur.npy", s.cpu().numpy())
        np.save(out_dir / "gaussian_blur_rows.npy", np.concatenate([r * rows + idx for r in range(world)]).astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps of every timed loop (the blur, e2e, the extra configs, --impl reference) except cpu_baseline's best of 2")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="zignal_b200", choices=["zignal_b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="which partitioning is the headline `value` at N > 1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write a fixed sample of the output of the headline blur's last timed step (and its row numbers) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "zignal_b200":
        ap.error("--dump-outputs applies to --impl zignal_b200")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    numa = bind_to_gpu_numa(local_rank)   # before CUDA / torch allocate anything on the host

    import torch
    import torch.distributed as dist
    import zignal_b200 as zb
    from zignal_b200 import shard

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = zb.lib()  # raises if the CUDA library is missing -- there is no fallback
    comm = shard.ShardComm.from_torch_distributed()
    taps = zb.gaussian_taps(SIGMA)
    assert taps.size == 15

    def make_blocks(rows):
        src, dst = comm.image(rows, COLS, zb.PixFmt.RGBAF32, 8), comm.image(rows, COLS, zb.PixFmt.RGBAF32, 8)   # 8 halo rows: the kernel's landing zone for the neighbours' 7
        gen = torch.Generator(device=dev).manual_seed(2 + rank)
        src.interior_tensor().copy_(torch.rand(rows, COLS, 4, device=dev, dtype=torch.float32, generator=gen))
        return src, dst

    # ---- the timed region: weak partitioning (8192 rows per GPU) -------------------------------------------------------
    src, dst = make_blocks(ROWS)

    def step():
        src.conv_separable(dst, taps, taps, zb.BorderMode.MIRROR)   # zb_shard_conv_separable: ONE launch per rank

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = L.zb_kernel_launch_count()
    ms_weak = time_steps(torch, dist, world, dev, step, args.steps, 0)
    launches = L.zb_kernel_launch_count() - launches0
    kernel_name = L.zb_last_kernel().decode()
    comm.status()
    if args.dump_outputs is not None and (world == 1 or args.scaling == "weak"):
        dump_outputs(torch, dist, rank, world, dst.interior_tensor(), args.dump_outputs)
    # keep the GPU under the same load a little longer so the clock sampler sees it (every rank: the steps are collective)
    for _ in range(60):
        for _ in range(50):
            step()
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None

    # ---- parity of the sharded result, checked inside this run (N > 1) -------------------------------------------------
    parity = None
    if world > 1:
        def neighbour_rows(block):
            """(up7, down7): the true neighbour rows of this rank's block, moved by torch.distributed (independent of zb_shard)."""
            edges = torch.stack([block[:HALO], block[-HALO:]]).contiguous()          # my first / last rows
            allr = [torch.empty_like(edges) for _ in range(world)]
            dist.all_gather(allr, edges)
            up = allr[rank - 1][1] if rank > 0 else None
            down = allr[rank + 1][0] if rank < world - 1 else None
            return up, down

        def check(exact):
            L.zb_set_exact_f32(1 if exact else 0)
            step()
            torch.cuda.synchronize()
            blk = src.interior_tensor()
            up, down = neighbour_rows(blk)
            parts = ([up] if up is not None else []) + [blk] + ([down] if down is not None else [])
            ext = torch.cat(parts).contiguous()
            ref = zb.Image.from_tensor(ext).convolve_separable(taps, taps, zb.BorderMode.MIRROR).tensor()
            o = HALO if up is not None else 0
            ref = ref[o:o + blk.shape[0]]
            got = dst.interior_tensor()
            same = bool(torch.equal(got, ref))
            rel = float(((got - ref).abs() / ref.abs().clamp_min(1e-6)).max().item())
            L.zb_set_exact_f32(0)
            del ext, ref
            return same, rel
        same_fast, rel_fast = check(False)
        same_exact, rel_exact = check(True)
        t = torch.tensor([1.0 if same_fast else 0.0, 1.0 if same_exact else 0.0, -rel_fast, -rel_exact], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        parity = {"checked": True, "what": "every rank's block vs a single-GPU blur of (block + true neighbour rows)",
                  "bit_identical": bool(t[0].item() == 1.0), "bit_identical_exact_mode": bool(t[1].item() == 1.0),
                  "max_rel": float(max(-t[2].item(), -t[3].item())), "tolerance": 1e-5}
        if not (parity["bit_identical_exact_mode"] and parity["max_rel"] <= 1e-5):
            if rank == 0:
                print(json.dumps({"error": "sharded result differs from the single-GPU result", "parity": parity}), flush=True)
            sys.exit(1)
    src.free()
    dst.free()

    # ---- strong partitioning: THE 8192 x 8192 image over N GPUs --------------------------------------------------------
    extra = {}
    strong = None
    if world > 1:
        rows_s = ROWS // world
        s2, d2 = make_blocks(rows_s)
        ms_strong = time_steps(torch, dist, world, dev, lambda: s2.conv_separable(d2, taps, taps, zb.BorderMode.MIRROR), args.steps, args.warmup)
        comm.status()
        if args.dump_outputs is not None and args.scaling == "strong":
            dump_outputs(torch, dist, rank, world, d2.interior_tensor(), args.dump_outputs)
        s2.free()
        d2.free()
        strong = {"scaling": "strong", "image": [ROWS, COLS], "rows_per_gpu": rows_s, "ms_per_step": ms_strong,
                  "value": ROWS * COLS / 1e6 / (ms_strong * 1e-3), "unit": "Mpixels/s"}
        extra["strong"] = strong

    # ---- end to end through the host-pointer C ABI (pinned host buffers) ------------------------------------------------
    e2e = None
    if not args.no_e2e:
        # the host holds the global image; every rank's pinned buffer is its row block plus the 7 overlapping rows of each
        # neighbour, so the sharded blur needs no exchange at all (SURVEY 8(e)) and the 2 x 7 extra result rows are discarded
        up_h = HALO if rank > 0 else 0
        down_h = HALO if rank < world - 1 else 0
        rows_e = ROWS + up_h + down_h
        nbytes = rows_e * COLS * 16
        hin, hout = C.c_void_p(), C.c_void_p()
        zb._ffi.check(L.zb_malloc_host(C.byref(hin), nbytes))
        zb._ffi.check(L.zb_malloc_host(C.byref(hout), nbytes))
        harr = np.ctypeslib.as_array(C.cast(hin, C.POINTER(C.c_float)), shape=(rows_e, COLS, 4))
        rng = np.random.default_rng(2 + rank)
        for r0 in range(0, rows_e, 512):   # first touch by this (NUMA-bound) process
            harr[r0:r0 + 512] = rng.random((min(512, rows_e - r0), COLS, 4), dtype=np.float32)
        np.ctypeslib.as_array(C.cast(hout, C.POINTER(C.c_float)), shape=(rows_e, COLS, 4))[:] = 0
        hi = zb.ZbImage(hin.value, rows_e, COLS, COLS)
        ho = zb.ZbImage(hout.value, rows_e, COLS, COLS)
        esteps = args.steps
        zb._ffi.check(L.zb_host_gaussian_blur(hi, ho, int(zb.PixFmt.RGBAF32), C.c_float(SIGMA)))  # warm-up
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(esteps):
            zb._ffi.check(L.zb_host_gaussian_blur(hi, ho, int(zb.PixFmt.RGBAF32), C.c_float(SIGMA)))
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / esteps
        te = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_ms = float(te.item())
        tb = torch.tensor([float(nbytes)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tb, op=dist.ReduceOp.SUM)
        e2e = {"value": world * ROWS * COLS / 1e6 / (e2e_ms * 1e-3), "unit": "Mpixels/s", "h2d_bytes_per_step": int(tb.item()),
               "d2h_bytes_per_step": int(tb.item()), "ms_per_step": e2e_ms, "steps": esteps, "host_numa": numa,
               "api": "zb_host_gaussian_blur (host pointers, pinned; H2D + kernel + D2H per step"
                      + ("; every rank's buffer = its row block + 7 overlapping rows per neighbour, no exchange)" if world > 1 else ")")}
        L.zb_free_host(hin)
        L.zb_free_host(hout)

    # ---- the other BASELINE configs, same process (each a handful of launches) ------------------------------------------
    if not args.no_extra:
        peak_x, _ = measured_peak_gbs()
        try:
            if world == 1:
                # C3: bicubic 16384^2 -> 4096^2 Rgb u8
                g = torch.Generator(device=dev).manual_seed(3)
                x = torch.randint(0, 256, (16384, 16384, 3), device=dev, dtype=torch.uint8, generator=g)
                big, small = zb.Image.from_tensor(x), zb.Image.init(4096, 4096, zb.PixFmt.RGB8)
                ms = time_steps(torch, dist, world, dev, lambda: big.resize(small, zb.Interpolation.BICUBIC), args.steps, 5)
                extra["c3_bicubic_16384_to_4096_rgb8"] = {"ms": ms, "algorithmic_bytes": 855638016, "frac_of_hbm_peak": 855638016 / (ms * 1e-3) / 1e9 / peak_x}
                del x, big, small
                # PCA (the "SVD step" config): Pca.fit's device core on n = 1,048,576 x dim 256 f32 -- column means + centring,
                # X^T X / (n - 1) on the tcgen05 tensor cores (3xTF32), one-sided Jacobi SVD of the 256 x 256 covariance
                from zignal_b200 import matrix
                g = torch.Generator(device=dev).manual_seed(7)
                X = torch.randn(1 << 20, 256, device=dev, generator=g)
                mean = torch.empty(256, device=dev)
                cen = torch.empty_like(X)

                def gram():
                    return matrix.gemm_device(cen, cen, True, False, 1.0 / (X.shape[0] - 1), 0.0, None)
                matrix.center_columns(X, mean, True, cen)
                ms_gemm = time_steps(torch, dist, world, dev, gram, args.steps, 3)
                cov = gram()
                ms_svd = time_steps(torch, dist, world, dev, lambda: matrix.svd_device(cov, True, False), args.steps, 1)

                def fit():
                    matrix.center_columns(X, mean, True, cen)
                    matrix.svd_device(gram(), True, False)
                ms_fit = time_steps(torch, dist, world, dev, fit, args.steps, 1)
                extra["pca_fit_1048576x256_f32"] = {"ms": ms_fit, "gemm_xtx_ms": ms_gemm, "svd_256x256_ms": ms_svd,
                                                    "gemm_tflops_fp32_accurate": 2.0 * X.shape[0] * 256 * 256 / (ms_gemm * 1e-3) / 1e12,
                                                    "kernel": L.zb_last_kernel().decode()}
                del X, cen, cov
            # C4: rotate 45 deg bilinear .zero, 1920x1080 Rgba frames; 1024 frames split over the ranks (128 per step call)
            n_total = 1024
            lo, hi_ = comm.split(n_total)
            n_local = hi_ - lo
            per_call = min(128, n_local)
            g = torch.Generator(device=dev).manual_seed(4 + rank)
            x = torch.randint(0, 256, (per_call, 1080, 1920, 4), device=dev, dtype=torch.uint8, generator=g)
            angle = np.float32(np.pi / 4)
            cs = (np.float32(np.cos(np.float64(angle))), np.float32(np.sin(np.float64(angle))))
            orows, ocols = zb.Image.from_tensor(x[0]).rotate_bounds(angle)
            y = torch.empty((per_call, orows, ocols, 4), device=dev, dtype=torch.uint8)
            src0, dst0 = zb.Image.from_tensor(x[0])._zb(), zb.Image.from_tensor(y[0])._zb()
            calls = (n_local + per_call - 1) // per_call

            def rot():
                for _ in range(calls):   # the same 128-frame buffers are reused: 3.4 GB of traffic per call >> L2
                    zb._ffi.check(L.zb_rotate_into_batch(src0, 1080 * 1920, dst0, orows * ocols, per_call, int(zb.PixFmt.RGBA8), C.c_float(angle),
                                                         C.c_float(cs[0]), C.c_float(cs[1]), int(zb.Interpolation.BILINEAR), C.c_float(1 / 3),
                                                         C.c_float(1 / 3), int(zb.BorderMode.ZERO), torch.cuda.current_stream().cuda_stream))
            ms = time_steps(torch, dist, world, dev, rot, args.steps, 2)
            bytes_c4 = 26305936 * n_total
            extra["c4_rotate45_1024x1080p_rgba8"] = {"ms": ms, "frames": n_total, "frames_per_gpu": n_local, "algorithmic_bytes": bytes_c4,
                                                     "frac_of_hbm_peak": bytes_c4 / (ms * 1e-3) / 1e9 / (peak_x * world)}
            del x, y
            # C5: fdm.update on the 4096 x 4096 Rgb image, rows split over the ranks (moments all-gathered inside the statistics kernel)
            from zignal_b200.fdm import FeatureDistributionMatching
            rows5 = 4096 // world
            g = torch.Generator(device=dev).manual_seed(5 + rank)
            s5 = torch.randint(0, 256, (rows5, 4096, 3), device=dev, dtype=torch.uint8, generator=g)
            t5 = (torch.randint(0, 256, (rows5, 4096, 3), device=dev, dtype=torch.uint8, generator=g) // 2 + 40).to(torch.uint8)
            t5[..., 1] = (t5[..., 1].to(torch.int32) * 3 // 4 + t5[..., 0].to(torch.int32) // 4).to(torch.uint8)
            f = FeatureDistributionMatching(zb.PixFmt.RGB8)
            comm.fdm_set_target(f, zb.Image.from_tensor(t5))
            f.set_source(zb.Image.from_tensor(s5))
            ms = time_steps(torch, dist, world, dev, lambda: comm.fdm_update(f), args.steps, 5)
            f.status()
            comm.status()
            extra["c5_fdm_update_4096x4096_rgb8"] = {"ms": ms, "rows_per_gpu": rows5, "algorithmic_bytes": 150994944,
                                                     "frac_of_hbm_peak": 150994944 / (ms * 1e-3) / 1e9 / (peak_x * world)}
            f.deinit()
        except Exception as e:  # noqa: BLE001  (the headline must still be printed)
            extra["error"] = f"{type(e).__name__}: {e}"

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        headline_ms = ms_weak if (world == 1 or args.scaling == "weak") else strong["ms_per_step"]
        total_px = (world * ROWS * COLS) if (world == 1 or args.scaling == "weak") else ROWS * COLS
        # roofline of the step: every GPU moves 32 B per pixel of its block in `headline_ms` (the 2 x 7 neighbour rows are 0.2 %)
        px_per_launch = total_px // world
        achieved = ALGO_BYTES_PER_PX * px_per_launch / (headline_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tp = ROOT / "profiles" / "traffic.json"
        if tp.exists():
            try:
                tj = json.loads(tp.read_text())
                if world == 1 and tj.get("kernel") == kernel_name:
                    traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
            except Exception:
                pass
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            sys.path.insert(0, str(ROOT / "tests"))
            import oracle_lib as zo
            rng = np.random.default_rng(2)
            planes = [rng.random((ROWS, COLS), dtype=np.float32) for _ in range(4)]
            outs = [np.empty_like(p) for p in planes]
            ztaps = zo.gaussian_taps(SIGMA)
            best = min(cpu_reference_pass(zo, planes, outs, ztaps, 1) for _ in range(2))
            cpu = {"value": ROWS * COLS / 1e6 / best, "unit": "Mpixels/s", "cores": 1, "kind": "port",
                   "sample": "full 8192x8192 RGBA f32 as 4 planar Image(f32) separable convolutions, best of 2, 1 thread "
                             "(the reference is single-threaded); Zig reference not buildable here -> C++ port under oracle/"}
        line = {
            "metric": METRIC, "value": total_px / 1e6 / (headline_ms * 1e-3), "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": headline_ms, "higher_is_better": True, "scaling": args.scaling if world > 1 else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "image": [ROWS * world, COLS] if (world == 1 or args.scaling == "weak") else [ROWS, COLS],
                       "pixel": "RGBA f32 interleaved (16 B)", "taps": 15, "border": "mirror",
                       "parallelism": f"row-block x{world}" + (" (zb_shard_conv_separable: neighbours' 7 edge rows fetched over NVLink inside the kernel, "
                                                                f"peer_access={comm.peer_access})" if world > 1 else ""),
                       "l2": "input 1 GiB per GPU >> 126 MB L2 (no flush needed)", "kernel": kernel_name},
            "e2e": e2e, "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": traffic_src, "peak_source": peak_src, "kernel_ms": headline_ms,
                         "timing": "step time of the timed region (one launch per step per GPU), max over ranks",
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_PX * px_per_launch},
            "cpu_baseline": cpu, "clocks": clocks, "parity": parity, "extra": extra,
        }
        print(json.dumps(line), flush=True)
    comm.destroy()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
