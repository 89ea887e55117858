#!/usr/bin/env python
"""bench.py -- throughput of the conv hot path (convertWithModels) on B200, one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--size S] [--engine auto|tc|fp32]
                    [--dump-outputs DIR]

Workload (BASELINE.json config 3, the one the metric is quoted on): one full scale2.0x model pass
(7 layers, 574 272 algorithmic FLOP per output pixel) over a synthetic 4096x4096 fp32 Y plane.
With N > 1 ranks (torchrun, one process per GPU) the plane is 4096 wide x 4096*N tall, cut into N
row bands (weak scaling).  Default exchange (--halo peer, the north_star's per-layer exchange done INSIDE
the library): every rank maps its neighbours' band-session frames (CUDA IPC, handles travel once over
torch.distributed) and after every layer one small kernel stores its boundary row straight into the
neighbour's halo row over NVLink and handshakes through flag words -- nothing on the data path touches
torch or NCCL.  --halo nccl moves the same rows with torch.distributed send/recv (cross-check), --halo input
trades 7 input rows once and recomputes the overlap.  Before timing, N > 1 runs verify the exchange against the
one-shot mode bit for bit ("halo_check").
The line also carries `configs`: BASELINE config 4 (ONE 8192x8192 plane over the N GPUs, strong scaling) and
config 5 (64 tiles of 512x512, noise2, tile t on GPU t mod N) measured in the same run.

metric  Mpix/s = output pixels / time of the whole pass.
value   inputs already resident in HBM, device entry point (w2x_convert_plane_device).
e2e     same pass through the host-buffer C-ABI call (w2x_convert_plane): pinned host input,
        H2D and D2H copies inside the timed region.
--impl reference   the reference's own CPU code on the host cores, one 512x512 block per step:
        oracle/_ref/libw2x_reference.so = the reference's src/modelHandler.cpp + src/convertRoutine.cpp
        compiled against the OpenCV API shim (falls back to OpenCV's kernels through cv2 driven like
        Model::filterWorker, then to oracle/w2x_oracle.c), with the most worker threads the
        reference's own plane partition can use (32).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_PIXEL = 574272           # 2 * 9 * sum(Cin*Cout), SURVEY.md section 8(d)
LAYER_MACS = [288, 9216, 18432, 36864, 73728, 147456, 1152]   # per pixel, L0..L6
MODEL = "scale2.0x"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(pw)), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's CPU path on the host cores
# ---------------------------------------------------------------------------------------------------
def workload_text(W, H, world):
    return (f"{W}x{H} fp32 Y plane per GPU, scale2.0x_model.json weights (7x conv3x3 + bias + leaky-ReLU 0.1), "
            f"block_splitting=on; plane {W}x{H * world} in {world} row band(s)")


def reference_jobs():
    """Worker threads for the reference's CPU path.  Model::filter gives each of nJob threads nOutputPlanes / nJob planes and
    the remainder to the last one (src/modelHandler.cpp:46-65): with more jobs than output planes (32 on the narrowest layers)
    every thread but the last gets ZERO planes and the layer runs serially, so 32 is the most parallel setting the
    reference's own scheme supports (its default is -j 4)."""
    return max(1, min(os.cpu_count() or 4, 32))


_CPU_REF = {}


def cpu_reference_block(n_job, repeats=1, want=None):
    """One 512x512 block (498x498 output pixels) of the workload plane through the reference's CPU path.
    Returns (seconds per block, kind, description).  Preference order:
      1. oracle/_ref/libw2x_reference.so -- the reference's OWN src/modelHandler.cpp + src/convertRoutine.cpp compiled against
         the OpenCV API shim (oracle/cvshim): its threads, its loops ("reference");
      2. OpenCV's kernels through cv2, driven call-for-call like Model::filterWorker (oracle/ref_cv2.py, "port");
      3. the scalar C restatement (oracle/w2x_oracle.c, "port").
    W2X_BENCH_CPU=cv2|oracle forces one of the fallbacks."""
    from oracle import oracle
    x = oracle.seeded_plane(4096, 4096, 1, "uniform")[:498, :498]
    if want is None:
        want = os.environ.get("W2X_BENCH_CPU", "")
    om = oracle.OracleModel.golden(MODEL)
    fn = kind = desc = None
    if want in ("", "reference"):
        try:
            from oracle import reference_lib
            if reference_lib.available():
                if "ref" not in _CPU_REF:
                    import tempfile
                    path = os.path.join(tempfile.mkdtemp(prefix="w2x_bench_"), f"{MODEL}_model.json")
                    om.write_json(path)                       # the golden weights in the reference's JSON format
                    _CPU_REF["ref"] = reference_lib.ReferenceModels(path)
                reference_lib.configure(n_job, 9)
                rm = _CPU_REF["ref"]
                fn = lambda: rm.convert(x, True)
                kind, desc = "reference", ("the reference's own src/modelHandler.cpp + src/convertRoutine.cpp (compiled against the OpenCV API shim "
                                           "oracle/cvshim: its loader, threads and loops; fp32 filter2D/add/max/min/scaleAdd restated, AVX2 auto-vectorised)")
        except Exception:
            fn = None
    if fn is None and want in ("", "cv2", "reference"):
        try:
            from oracle import ref_cv2
            if ref_cv2.cv2 is None:
                raise ImportError
            models = []
            for w, b in zip(om.weights, om.biases):
                models.append(ref_cv2.Model({"nInputPlane": w.shape[1], "nOutputPlane": w.shape[0], "kW": 3, "kH": 3,
                                             "weight": w.astype(np.float64), "bias": b}))
            fn = lambda: ref_cv2.convert_with_models(x, models, block_splitting=True, n_job=n_job)
            kind, desc = "port", "OpenCV (cv2 %s) driven call-for-call like Model::filterWorker" % ref_cv2.cv2.__version__
        except Exception:
            fn = None
    if fn is None:
        fn = lambda: om.convert(x, n_job=n_job)
        kind, desc = "port", "oracle/w2x_oracle.c scalar restatement"
    ts = []
    for _ in range(repeats):
        t = time.perf_counter(); fn(); ts.append(time.perf_counter() - t)
    return min(ts), kind, desc


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_job = reference_jobs()
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_reference_block(n_job)
    t0 = time.perf_counter()
    per = []
    for _ in range(args.steps):
        s, kind, desc = cpu_reference_block(n_job)
        per.append(s)
    total = time.perf_counter() - t0
    mpix = 498 * 498 * args.steps / sum(per) / 1e6
    sample = f"{args.steps} x one 512x512 block (498x498 output px) of the 4096x4096 plane; {desc}; -j {n_job} of {os.cpu_count()} host threads (the reference's plane partition cannot use more, default -j 4)"
    line = {"metric": "Mpix/s full scale2.0x model pass", "value": mpix, "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(per) / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_text(args.size, args.size, max(1, args.gpus)), "weights": f"{MODEL}_model.json",
                       "sample": "bounded: one 512x512 block (498x498 output px) of that plane per step, on the host cores", "wall_s": total},
            "cpu_baseline": {"value": mpix, "unit": "Mpix/s", "cores": n_job, "kind": kind, "sample": sample},
            "e2e": {"value": mpix, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def write_model_json(npz_path, json_path):
    """The committed weight fixture (tests/golden/models/*.npz) in the reference's model-file format
    (array of {nInputPlane, nOutputPlane, kW, kH, weight[o][i][ky][kx], bias[o]}; src/modelHandler.cpp:74-115)."""
    z = np.load(npz_path)
    layers = []
    for i in range(int(z["n_layers"])):
        w, b = z[f"w{i}"], z[f"b{i}"]
        layers.append({"nInputPlane": int(w.shape[1]), "nOutputPlane": int(w.shape[0]), "kW": 3, "kH": 3,
                       "weight": [[[[float(np.float64(v)) for v in row] for row in k] for k in o] for o in w], "bias": [float(v) for v in b]})
    with open(json_path, "w") as f:
        json.dump(layers, f)


def pin_to_gpu_numa_node(torch, local):
    """Run this rank on the CPUs of its GPU's NUMA node, so that the page-locked host buffers it allocates (first touch) sit
    behind the same PCIe root as the GPU: with one rank per GPU and no affinity, half of the host<->device traffic of an 8-GPU
    box crosses the socket interconnect."""
    try:
        p = torch.cuda.get_device_properties(local)
        dev = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{dev}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def host_api_legs(w2x, steps, size):
    """The API a reference maintainer links, timed from C++ / the shell:
      e2e_cpp   w2xc::convertWithModels (host/w2xc.hpp: w2xc::Plane in / out, progress lines on stdout) on the bench plane;
      cli_cfg2  BASELINE config 2: the drop-in CLI on a 1920x1080 RGB image, -m noise_scale (noise1 + scale2.0x), wall clock."""
    import tempfile
    out = {}
    pkg = os.path.dirname(w2x.lib_path())
    d = tempfile.mkdtemp(prefix="w2x_bench_models_")
    for name in ("scale2.0x", "noise1"):
        write_model_json(os.path.join(ROOT, "tests", "golden", "models", f"{name}_model.npz"), os.path.join(d, f"{name}_model.json"))
    exe = os.path.join(pkg, "w2x-bench-host")
    if os.path.exists(exe):
        try:
            r = subprocess.run([exe, os.path.join(d, "scale2.0x_model.json"), str(size), str(size), str(steps), "2"], capture_output=True, text=True, timeout=300)
            line = [l for l in r.stdout.splitlines() if l.startswith("BENCH_JSON ")]
            if r.returncode == 0 and line:
                j = json.loads(line[-1][len("BENCH_JSON "):])
                out["e2e_cpp"] = {"value": j["mpix_per_s"], "unit": "Mpix/s", "ms_per_step": j["ms_per_step"], "api": j["api"],
                                  "note": "C++ caller, w2xc::Plane (page-locked) in/out, the reference's progress lines printed, copies inside the call"}
            else:
                out["e2e_cpp"] = {"error": (r.stderr or r.stdout)[-300:]}
        except Exception as e:
            out["e2e_cpp"] = {"error": f"{type(e).__name__}: {e}"}
    cli = os.path.join(pkg, "w2x-converter")
    if os.path.exists(cli):
        try:
            rgb = np.random.default_rng(4).integers(0, 256, size=(1080, 1920, 3), dtype=np.uint8)
            ppm = os.path.join(d, "in.ppm")
            with open(ppm, "wb") as f:
                f.write(b"P6\n1920 1080\n255\n" + rgb.tobytes())
            best, stages = None, None
            for _ in range(3):
                t = time.perf_counter()
                r = subprocess.run([cli, "-i", ppm, "-o", os.path.join(d, "out.png"), "-m", "noise_scale", "--model_dir", d], capture_output=True, text=True,
                                   timeout=300, env=dict(os.environ, W2X_CLI_TIMING="1"))
                dt = time.perf_counter() - t
                if r.returncode != 0:
                    raise RuntimeError((r.stderr or r.stdout)[-300:])
                if best is None or dt < best:
                    best = dt
                    tl = [l for l in r.stderr.splitlines() if "w2x_cli_timing_ms" in l]
                    stages = json.loads(tl[-1])["w2x_cli_timing_ms"] if tl else None
            out["cli_cfg2"] = {"workload": "1920x1080 RGB (uniform noise, PPM in, PNG out), -m noise_scale: noise1 pass on 1920x1080 Y + scale2.0x pass on 3840x2160 Y",
                               "wall_s_per_image": best, "conv_mpix_per_s": (1920 * 1080 * 5 / 1e6) / (stages["convertWithModels"] * 1e-3) if stages else None,
                               "stages_ms": stages, "note": "process start to exit, best of 3 (includes CUDA context creation, model JSON parsing, host colour/resize plumbing, PNG deflate)"}
        except Exception as e:
            out["cli_cfg2"] = {"error": f"{type(e).__name__}: {e}"}
    return out



DUMP_BYTES = 32 << 20


def dump_outputs(out_dir, plane, rank, world):
    """Write the output plane of the timed path's last step as <out_dir>/output.npy (float32), so that two builds can be
    compared output for output on the same seeded input.  A plane larger than this rank's share of DUMP_BYTES is cut to
    a fixed, seeded sample of whole rows; output_rows.npy (float64) lists which rows, in order.  With N > 1 ranks every
    rank writes its band as output_rank<r>.npy / output_rows_rank<r>.npy."""
    import torch
    h, w = plane.shape
    keep = min(h, max(1, DUMP_BYTES // world // (w * 4)))
    rows = np.arange(h) if keep == h else np.sort(np.random.default_rng(0).choice(h, size=keep, replace=False))
    sample = plane.index_select(0, torch.as_tensor(rows, device=plane.device)).cpu().numpy().astype(np.float32)
    suffix = "" if world == 1 else f"_rank{rank}"
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"output{suffix}.npy"), sample)
    np.save(os.path.join(out_dir, f"output_rows{suffix}.npy"), rows.astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    import w2x_loader
    w2x = w2x_loader.load()
    if not os.path.exists(w2x.lib_path()):
        raise SystemExit("libw2x_b200.so missing: run __graft_entry__.build() first (no fallback path exists)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    pin_to_gpu_numa_node(torch, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W = H = args.size
    if args.strong and world > 1:
        if H % world:
            raise SystemExit("--strong needs the plane height to divide by the number of ranks")
        H = H // world                         # ONE size x size plane, cut into `world` row bands
    n_model = 7
    # the shipped scale2.0x weights as committed fixtures (tests/golden/models, written by oracle/gen_golden.py from the reference's JSON)
    z = np.load(os.path.join(ROOT, "tests", "golden", "models", f"{MODEL}_model.npz"))
    n_layers = int(z["n_layers"])
    model = w2x.Model.from_arrays([z[f"w{i}"] for i in range(n_layers)], [z[f"b{i}"] for i in range(n_layers)])
    engine = {"auto": w2x.ENGINE_AUTO, "tc": w2x.ENGINE_TC, "fp32": w2x.ENGINE_FP32}[args.engine]
    ctx = w2x.Context(local, engine=engine)
    ctx.set_precision(w2x.PRECISION_F16_F8X2 if args.precision == "f8" else w2x.PRECISION_F16X3)
    passes = 2.0 if args.precision == "f8" else 3.0
    stream = torch.cuda.Stream()            # a real (non-default) stream: handle 0 would mean "the context's own stream"
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx.set_stream(stream.cuda_stream)

    # this rank's band of the (H*world) x W plane, seeded per rank
    host_in = torch.from_numpy(np.random.default_rng(1 + rank).random((H, W), dtype=np.float32)).pin_memory()   # uniform [0,1) noise, SURVEY 8(d)
    host_out = torch.empty((H, W), dtype=torch.float32).pin_memory()
    up, down = (rank - 1 if rank > 0 else None), (rank + 1 if rank < world - 1 else None)
    ra, rb = (n_model if up is not None else 0), (n_model if down is not None else 0)
    d_ext = torch.empty((H + ra + rb, W), dtype=torch.float32, device="cuda")   # [halo above | band | halo below]
    d_band = d_ext[ra:ra + H]
    d_band.copy_(host_in)
    d_out = torch.empty((H, W), dtype=torch.float32, device="cuda")

    from w2x_b200 import bands

    def exchange_halos():
        bands.exchange_halos(d_ext, H, rank, world, n_model, dist)

    def make_band(width, rows):
        """This rank's band session, wired to the neighbour ranks' sessions through peer memory (CUDA IPC)."""
        b = w2x.Band(ctx, model, width, rows, up is not None, down is not None)
        if args.halo == "peer":
            blobs = [None] * world
            dist.all_gather_object(blobs, b.export())
            b.connect(blobs[rank - 1] if up is not None else None, blobs[rank + 1] if down is not None else None)
        return b

    band = None
    if world > 1 and args.halo in ("peer", "nccl"):
        band = make_band(W, H)
        one_up = 1 if up is not None else 0

    def step_band(b, d_rows, d_res, width):
        if args.halo == "peer":
            b.run(d_rows.data_ptr(), width * 4, d_res.data_ptr(), width * 4)     # load, 7 x (layer, exchange kernel), gather: all in C++
        else:
            # the same 7-row buffer is reused: only the row adjacent to the band is needed here
            bands.exchange_halos(d_ext, H, rank, world, n_model, dist)
            first = d_ext[ra - one_up:]
            bands.run_band_per_layer(b, first.data_ptr(), width * 4, d_res.data_ptr(), width * 4, rank, world, dist, torch)

    def step_device():
        if band is not None:
            return step_band(band, d_band, d_out, W)
        exchange_halos()
        if world == 1:
            ctx.convert_plane_device(model, d_band.data_ptr(), W, H, W * 4, d_out.data_ptr(), W * 4, True)
        else:
            ctx.convert_band_device(model, d_ext.data_ptr(), W, H, ra, rb, W * 4, d_out.data_ptr(), W * 4)

    slab = None
    if world > 1 and args.halo == "peer":
        # host rows in / out: the rank's slab is cut into sub-bands (upload / layers / download overlap); its outer edges
        # exchange a halo row per layer with the neighbour ranks' slabs; odd ranks walk bottom -> top (see w2x_slab_create)
        slab = w2x.Slab(ctx, model, W, H, up is not None, down is not None, order=rank & 1)
        blobs = [None] * world
        dist.all_gather_object(blobs, slab.export())
        slab.connect(blobs[rank - 1] if up is not None else None, blobs[rank + 1] if down is not None else None)

    def step_e2e():
        if world == 1:
            ctx.convert_plane(model, host_in.numpy(), True, out=host_out.numpy())
        elif slab is not None:
            slab.convert(host_in.numpy(), host_out.numpy())
        else:
            d_band.copy_(host_in, non_blocking=True)
            step_device()
            host_out.copy_(d_out, non_blocking=True)
            stream.synchronize()

    def timed(fn, steps, with_layers=False, sampler=None):
        if sampler:
            sampler.start()          # BEFORE the barrier: forking nvidia-smi takes rank 0 tens of milliseconds, and with a per-layer
                                     # exchange every other rank would spend them waiting for rank 0 inside its timed region
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if with_layers:
            ctx.set_timing(True)
            ctx.layer_times(reset=True)
        n0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if world > 1:
            dist.barrier()
        clocks = sampler.stop() if sampler else None
        layers = ctx.layer_times(reset=True) if with_layers else None
        if with_layers:
            ctx.set_timing(False)
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms, wall * 1e3], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), ctx.launch_count() - n0, layers, clocks

    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    halo_check = None
    if world > 1:
        got = d_out.clone()
        exchange_halos()
        ctx.convert_band_device(model, d_ext.data_ptr(), W, H, ra, rb, W * 4, d_out.data_ptr(), W * 4)
        torch.cuda.synchronize()
        same = bool(torch.equal(got, d_out))
        flags = [None] * world
        dist.all_gather_object(flags, same)
        if rank == 0:
            print(f"[check] per-rank bit-equality of halo={args.halo} vs one-shot input-halo band mode: {flags}", file=sys.stderr, flush=True)
        if not all(flags):
            raise SystemExit("multi-GPU check failed")
        halo_check = True
    sampler = ClockSampler(local) if rank == 0 else None
    ms_dev, _, launches, layers, clocks = timed(step_device, args.steps, with_layers=True, sampler=sampler)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d_out, rank, world)
    for _ in range(min(args.warmup, 2)):
        step_e2e()
    _, ms_e2e_wall, _, _, _ = timed(step_e2e, args.steps)
    step_device()
    torch.cuda.synchronize()
    e2e_same = bool(torch.equal(host_out, d_out.cpu()))          # the host-buffer path returns the device-resident path's bits
    if world > 1:
        fl = [None] * world
        dist.all_gather_object(fl, e2e_same)
        e2e_same = all(fl)
    if not e2e_same:
        raise SystemExit("e2e result differs from the device-resident result")

    # ---- the other multi-GPU configurations of BASELINE.json, measured in the same run (driver-visible) ----
    configs = {}
    if not args.no_configs:
        k_cfg, w_cfg = max(3, min(args.steps, 5)), 2

        def leg(fn, sync_stream=False):
            for _ in range(w_cfg):
                fn()
            ms, wall, _, _, _ = timed(fn, k_cfg)
            return (wall if sync_stream else ms) / k_cfg

        # config 4: ONE 8192x8192 plane over the N GPUs (strong scaling), per-layer halo exchange through peer memory
        S = args.cfg4_size
        if S % world == 0 and (world == 1 or args.halo == "peer"):
            rows4 = S // world
            x4 = np.random.default_rng(2).random((S, S), dtype=np.float32)[rank * rows4:(rank + 1) * rows4]
            d4_in = torch.from_numpy(np.ascontiguousarray(x4)).cuda()
            d4_out = torch.empty_like(d4_in)
            del x4
            if world == 1:
                ms4 = leg(lambda: ctx.convert_plane_device(model, d4_in.data_ptr(), S, S, S * 4, d4_out.data_ptr(), S * 4, True))
            else:
                band4 = make_band(S, rows4)
                ms4 = leg(lambda: band4.run(d4_in.data_ptr(), S * 4, d4_out.data_ptr(), S * 4))
                torch.cuda.synchronize()
                dist.barrier()
                band4.close()
            configs["cfg4_strong"] = {"workload": f"ONE {S}x{S} fp32 Y plane, scale2.0x, cut into {world} row band(s) of {rows4} rows" +
                                      ("" if world == 1 else ", 1 boundary row per neighbour after every layer through peer memory"),
                                      "n_gpus": world, "ms_per_step": ms4, "value": S * S / (ms4 * 1e-3) / 1e6, "unit": "Mpix/s", "scaling": "strong",
                                      "steps": k_cfg, "timing": "CUDA events, max over ranks"}
            del d4_in, d4_out
            torch.cuda.empty_cache()
        # config 5: 64 tiles of 512x512, noise2 weights, tile t on GPU t mod N, every GPU runs its tiles as one batched pass
        z5 = np.load(os.path.join(ROOT, "tests", "golden", "models", "noise2_model.npz"))
        model5 = w2x.Model.from_arrays([z5[f"w{i}"] for i in range(int(z5["n_layers"]))], [z5[f"b{i}"] for i in range(int(z5["n_layers"]))])
        n_tiles, T = 64, 512
        mine = list(range(rank, n_tiles, world))
        if mine:
            tiles = np.random.default_rng(3).random((n_tiles, T, T), dtype=np.float32)[mine]
            h5_in = torch.from_numpy(np.ascontiguousarray(tiles)).pin_memory()
            h5_out = torch.empty_like(h5_in).pin_memory()
            d5_in = h5_in.cuda()
            d5_out = torch.empty_like(d5_in)
            ms5 = leg(lambda: ctx.convert_tiles_device(model5, d5_in.data_ptr(), d5_out.data_ptr(), len(mine), T, T))
            ms5_e2e = leg(lambda: ctx.convert_tiles(model5, h5_in.numpy(), out=h5_out.numpy()), sync_stream=True)
            configs["cfg5_tiles"] = {"workload": f"{n_tiles} tiles of {T}x{T} fp32, noise2_model.json weights, tile t on GPU t mod {world}; each GPU runs its "
                                                 f"{len(mine)} tiles as ONE stacked frame per layer launch (w2x_convert_tiles); no exchange",
                                     "n_gpus": world, "ms_per_batch": ms5, "value": n_tiles * T * T / (ms5 * 1e-3) / 1e6, "unit": "Mpix/s",
                                     "e2e_value": n_tiles * T * T / (ms5_e2e * 1e-3) / 1e6, "e2e_note": "host tiles (pinned) -> host tiles through w2x_convert_tiles, wall clock, max over ranks",
                                     "steps": k_cfg}
            del d5_in, d5_out

    if rank == 0:
        peaks = load_peaks()
        pix_total = W * H * world
        ms_step = ms_dev / args.steps
        mpix = pix_total / (ms_step * 1e-3) / 1e6
        mpix_e2e = pix_total / (ms_e2e_wall / args.steps * 1e-3) / 1e6
        # dominant kernel = the layer with the largest summed time
        roof = None
        if layers:
            k = max(range(len(layers)), key=lambda i: layers[i][0])
            ms_k, n_k, name_k = layers[k]
            flop_launch = 2.0 * LAYER_MACS[k] * W * H * args.steps / n_k            # algorithmic: output pixels only
            tensor = name_k.startswith("tcgen05")
            ach = flop_launch / (ms_k / n_k * 1e-3) / 1e12
            peak = peaks["tf_sustained"] if tensor else None
            traffic = None
            tp = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(tp):
                traffic = json.load(open(tp)).get(f"{name_k}:L{k}:{W}x{H}")
            roof = {"kernel": f"{name_k} (layer L{k}, {LAYER_MACS[k] // 9} MAC/tap/px)", "bound": "tensor" if tensor else "fp32-cuda-core",
                    "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": (ach / peak) if peak else None,
                    "peak_source": f"{peaks['source']}: cuBLAS bf16 sustained (kernel timed inside a long step); fp16 and bf16 share the rate",
                    "mma_passes": passes if tensor else None,
                    "frac_of_attainable": (ach * passes / peak) if peak else None,
                    "note": "achieved = ALGORITHMIC flops (one multiply-add per weight per output pixel); the fp32-faithful operand split issues "
                            "3 fp16 MMA passes (f16x3) or 1 fp16 + 2 double-rate e4m3 passes (f8: 2.0 pass-equivalents), so the attainable "
                            "ceiling is peak/passes",
                    "launch_ms": ms_k / n_k, "launches": n_k, "traffic": traffic,
                    "all_layers_ms": [round(l[0] / max(l[1], 1), 4) for l in layers],
                    "whole_pass_algorithmic_tflops": FLOP_PER_PIXEL * pix_total / (ms_step * 1e-3) / 1e12 / world}
        cpu = None
        if world == 1 and not args.no_cpu:
            nj = reference_jobs()
            try:
                s, kind, desc = cpu_reference_block(nj)
            except Exception as e:                      # never lose the GPU measurement to the baseline leg
                os.environ["W2X_BENCH_CPU"] = "oracle"
                s, kind, desc = cpu_reference_block(nj)
                desc += f" (preferred baseline failed: {type(e).__name__}: {e})"
            cpu = {"value": 498 * 498 / s / 1e6, "unit": "Mpix/s", "cores": nj, "kind": kind,
                   "sample": f"one 512x512 block (498x498 output px) of the same plane, {s:.2f} s; {desc}; -j {nj} of {os.cpu_count()} host threads (the reference's plane partition cannot use more; default -j 4)"}
            try:      # the same block through OpenCV's own kernels (cv2), driven call for call like Model::filterWorker: "the reference's OpenCV CPU path"
                s2, kind2, desc2 = cpu_reference_block(nj, want="cv2")
                if "cv2" in desc2:
                    cpu["opencv_variant"] = {"value": 498 * 498 / s2 / 1e6, "unit": "Mpix/s", "cores": nj, "kind": kind2, "sample": f"same block, {s2:.2f} s; {desc2}"}
            except Exception:
                pass
        host_api = host_api_legs(w2x, max(3, min(args.steps, 10)), args.size) if (world == 1 and not args.no_configs) else {}
        line = {"metric": "Mpix/s full scale2.0x model pass", "value": mpix, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if (args.strong and world > 1) else "weak", "vs_baseline": None,
                "dtype": ("f32" if args.engine == "fp32" else "f16x3 split operands, f32 accumulate (fp32-faithful)" if args.precision == "f16x3"
                          else "f16 + 2x e4m3 correction products, f32 accumulate (fp32-faithful to ~3e-5)"),
                "data": "synthetic",
                "config": {"workload": workload_text(W, H, world),
                           "weights": f"{MODEL}_model.json", "engine": args.engine,
                           "halo_exchange": ("none" if world == 1 else "7 input rows per neighbour once, NCCL send/recv" if band is None
                                             else "1 row of every intermediate activation per neighbour after every layer, " +
                                             ("stored straight into the neighbour's frame by the library (peer memory over NVLink, CUDA IPC; flag handshake, one kernel per layer)"
                                              if args.halo == "peer" else "torch.distributed send/recv (NCCL)")),
                           "comm": (None if world == 1 else "peer-memory stores + flags (csrc/engine_band.cu w2x_band_exchange)" if args.halo == "peer" else "NCCL send/recv"),
                           "l2": "no explicit flush: each step streams ~17 GB of activations per GPU, far beyond the 126 MB L2"},
                "e2e": {"value": mpix_e2e, "unit": "Mpix/s", "h2d_bytes_per_step": W * H * 4 * world, "d2h_bytes_per_step": W * H * 4 * world,
                        "timing": "host wall clock around K calls of the host-buffer C-ABI entry (sync inside the call), max over ranks"},
                "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "halo_check": halo_check, "e2e_check": e2e_same, "configs": configs, **host_api}
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--engine", default="auto", choices=["auto", "tc", "fp32"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--precision", default="f8", choices=["f16x3", "f8"],
                    help="tcgen05 arithmetic: fp16 + two e4m3 correction products (the library default) or three fp16 products")
    ap.add_argument("--strong", action="store_true", help="multi-GPU: cut ONE size x size plane into N row bands (strong scaling) instead of one plane per GPU")
    ap.add_argument("--check", action="store_true", help="(kept for compatibility: the halo check always runs for N > 1)")
    ap.add_argument("--halo", default="peer", choices=["input", "peer", "nccl"],
                    help="multi-GPU exchange: 1 activation row after every layer through peer memory inside the library (north_star; default), "
                         "the same rows through torch.distributed send/recv, or 7 input rows once (recompute)")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg4 (8192^2 strong) and cfg5 (64 tiles) legs")
    ap.add_argument("--cfg4-size", type=int, default=8192)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the output plane of the last one to DIR/output.npy (a seeded row sample above 32 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
