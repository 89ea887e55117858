"""cli_plumbing_ab.py -- the drop-in CLI on BASELINE config 2 (bench.py's cli_cfg2 image: seed 4, uniform 1920x1080 RGB, PPM in,
PNG out, -m noise_scale), alternating the host image plumbing (W2X_CLI_HOST_PLUMBING=1) and the device path.

    python tools/cli_plumbing_ab.py [pairs=7] [out.json]

Per path: median / min / max of every W2X_CLI_TIMING stage and of the process wall clock; the two outputs of every pair are
compared byte for byte.  The GPU's name and power limit are read in the same run and stored beside the numbers."""
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import write_model_json  # noqa: E402  (the same model files bench.py writes)

CLI = os.path.join(ROOT, "waifu2x-converter-cpp_b200", "w2x-converter")


def run(d, path):
    env = dict(os.environ, W2X_CLI_TIMING="1")
    env.pop("W2X_CLI_HOST_PLUMBING", None)
    if path == "host":
        env["W2X_CLI_HOST_PLUMBING"] = "1"
    out = os.path.join(d, f"out_{path}.png")
    t = time.perf_counter()
    r = subprocess.run([CLI, "-i", os.path.join(d, "in.ppm"), "-o", out, "-m", "noise_scale", "--model_dir", d], capture_output=True, text=True,
                       timeout=300, env=env)
    wall = (time.perf_counter() - t) * 1e3
    if r.returncode != 0:
        raise RuntimeError(f"{path}: exit {r.returncode}: {(r.stderr or r.stdout)[-400:]}")
    stages = json.loads([l for l in r.stderr.splitlines() if "w2x_cli_timing_ms" in l][-1])["w2x_cli_timing_ms"]
    stages["wall_clock"] = wall
    with open(out, "rb") as f:
        return stages, f.read(), r.stdout


def main():
    pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 7
    dest = sys.argv[2] if len(sys.argv) > 2 else None
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    d = tempfile.mkdtemp(prefix="w2x_cli_ab_")
    for name in ("scale2.0x", "noise1"):
        write_model_json(os.path.join(ROOT, "tests", "golden", "models", f"{name}_model.npz"), os.path.join(d, f"{name}_model.json"))
    rgb = np.random.default_rng(4).integers(0, 256, size=(1080, 1920, 3), dtype=np.uint8)
    with open(os.path.join(d, "in.ppm"), "wb") as f:
        f.write(b"P6\n1920 1080\n255\n" + rgb.tobytes())
    runs = {"host": [], "device": []}
    identical, plumbing_lower = [], []
    for i in range(pairs):
        order = ("host", "device") if i % 2 == 0 else ("device", "host")
        got = {p: run(d, p) for p in order}
        identical.append(got["host"][1] == got["device"][1] and got["host"][2] == got["device"][2])
        plumbing_lower.append(got["device"][0]["colour_resize_plumbing"] < got["host"][0]["colour_resize_plumbing"])
        for p in order:
            runs[p].append(got[p][0])
        print(f"pair {i}: host {got['host'][0]['wall_clock']:.0f} ms, device {got['device'][0]['wall_clock']:.0f} ms, "
              f"plumbing {got['host'][0]['colour_resize_plumbing']:.1f} -> {got['device'][0]['colour_resize_plumbing']:.1f} ms, "
              f"identical={identical[-1]}", flush=True)
    summary = {}
    for p, rs in runs.items():
        summary[p] = {k: {"median": statistics.median(r[k] for r in rs), "min": min(r[k] for r in rs), "max": max(r[k] for r in rs)}
                      for k in rs[0]}
    result = {"gpu": gpu, "workload": "BASELINE config 2: 1920x1080 RGB (uniform noise, seed 4), PPM in, PNG out, -m noise_scale",
              "pairs": pairs, "outputs_identical_every_pair": all(identical), "device_plumbing_lower_every_pair": all(plumbing_lower),
              "ms": summary, "runs": runs}
    print(json.dumps({k: v for k, v in result.items() if k != "runs"}, indent=1))
    if dest:
        with open(dest, "w") as f:
            json.dump(result, f, indent=1)
    return 0 if all(identical) else 1


if __name__ == "__main__":
    sys.exit(main())
