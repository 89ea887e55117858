"""reference_golden.py -- TEST INFRASTRUCTURE.  What the reference's own code computed, stored under
tests/golden/reference/ so that the tests comparing against it run from the repository alone.

    make -C oracle REF=<reference checkout>
    python oracle/reference_golden.py <reference checkout>

The first line builds oracle/_ref/libw2x_reference.so (the reference's src/modelHandler.cpp + src/convertRoutine.cpp
against the OpenCV API shim) and oracle/_ref/waifu2x-reference-cli (its src/main.cpp as well); the second runs them
on the seeded inputs of tests/test_reference_build.py, tests/test_reference_cli.py and tests/test_model_loader.py.

Written files
  runs.json              the reference's outputs: sha256 digests (see digest()) of every array a test compares bit
                         for bit, block orders traced from its progress output, CLI texts and exit codes
  cli_images.npz         the reference CLI's output images (uint8 BGR) of the restated-pipeline cases
  model_excerpts.json.gz the text of the first and last layer object of each shipped models/<name>_model.json, as
                         the reference ships it (the whole files are 5.5 MB each)
"""
from __future__ import annotations

import gzip
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "reference")
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "waifu2x-reference-cli")
EXCERPT_LAYERS = (0, 6)


def digest(a) -> str:
    """sha256 of an fp32 array's shape and bytes: equal digests mean bit-identical outputs."""
    a = np.ascontiguousarray(a, np.float32)
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()


def load():
    with open(os.path.join(OUT, "runs.json")) as f:
        return json.load(f)


def cli_images():
    return np.load(os.path.join(OUT, "cli_images.npz"))


def model_excerpts():
    with gzip.open(os.path.join(OUT, "model_excerpts.json.gz"), "rt") as f:
        return json.load(f)


def norm_cli_text(text, exe):
    """CLI messages modulo the program name / path TCLAP prints"""
    text = text.replace(exe, "PROG").replace(os.path.basename(exe), "PROG")
    return re.sub(r"[ \t]+", " ", text).strip()


def identity_model_json(path, n_layers=7):
    """n_layers of 1 -> 1 planes, kernel = delta, bias 0: convertWithModels becomes the identity on positive input, cheap
    enough to push the reference's block-split code through full-size planes."""
    layer = {"nInputPlane": 1, "nOutputPlane": 1, "kW": 3, "kH": 3, "weight": [[[[0, 0, 0], [0, 1, 0], [0, 0, 0]]]], "bias": [0.0]}
    with open(path, "w") as f:
        json.dump([layer] * n_layers, f)


def block_trace(log):
    """(c, r) of every block, in the order the reference's progress output names them (src/convertRoutine.cpp:100-134)"""
    return [[int(c), int(r)] for c, r in re.findall(r"start process block \((\d+),(\d+)\)", log)]


# ---------------------------------------------------------------------------------------------------
# the cases the tests compare on
# ---------------------------------------------------------------------------------------------------
CONVERT_SIZES = ((1, 1, 11), (15, 13, 25), (37, 61, 47), (64, 48, 3))
SPLIT64_SIZES = ((120, 90, 4), (101, 64, 5), (51, 121, 6), (150, 50, 7))
ODD_SIZES = ((1, 1), (15, 13), (37, 61))
FULL_SIZES = ((512, 768), (513, 768), (768, 512), (499, 1), (1, 1), (1920, 1080), (3840, 2160), (4096, 4096), (1234, 3211))
CLI_PIPELINE_CASES = (("noise_scale", 1, 2.0, "in(noise_scale)(Level1)(x2.000000).png"), ("scale", 1, 3.0, "in(scale)(x3.000000).png"),
                      ("scale", 1, 1.5, "in(scale)(x1.500000).png"), ("noise", 2, 2.0, "in(noise)(Level2).png"))
CLI_FAIL_CASES = (
    [],                                                     # required -i missing -> TCLAP parse error, exit 1
    ["-i", "a.png", "-m", "bogus"],                         # value not in the allowed set
    ["-i", "a.png", "--noise_level", "3"],
    ["-i", "a.png", "--jobs", "x"],                         # not an integer
    ["-i", "a.png", "--nope", "1"],                         # unknown flag
    ["-i", "a.png", "-i", "b.png"],                         # flag given twice
    ["--version"],
    ["-i", "in.png", "--model_dir", "no_such_dir"],         # model file missing after a successful image read: exit(-1)
    ["-i", "in.png", "-m", "scale", "--model_dir", "no_such_dir"],
)


def cli_case_id(args):
    return " ".join(args) or "(none)"


def random_block_cases():
    """Seeded random plane sizes x block sizes 2^5..2^9, plus planes at / just past the split threshold and exact multiples of
    the block stride."""
    rng = np.random.default_rng(2024)
    cases = []
    for exp in (5, 6, 7, 9):
        b = 1 << exp
        for _ in range(8):
            cases.append((exp, int(rng.integers(1, 6 * b)), int(rng.integers(1, 6 * b))))
        thr = b * b * 3 // 2
        cases += [(exp, thr // 8, 8), (exp, thr // 8 + 1, 8), (exp, b - 14, 3 * b), (exp, 2 * (b - 14) + 1, b)]
    return [(exp, min(w, 1500), min(h, 1500)) if exp == 9 and w * h > 1500 * 1500 else (exp, w, h) for exp, w, h in cases]


def _fmt_number(rng, v):
    """one of the spellings a JSON writer may produce for the double v"""
    k = int(rng.integers(0, 8))
    if k == 0:
        return repr(float(v))
    if k == 1:
        return "%.17g" % v
    if k == 2:
        return "%.20e" % v
    if k == 3:
        return ("%.12E" % v).replace("E-0", "E-").replace("E+0", "E+")
    if k == 4:
        return "%.25f" % v
    if k == 5:
        return ("%.15g" % v).replace("e-0", "e-")
    if k == 6:
        return "%.9g" % v              # fewer digits than fp32 needs: a different double, same test (both loaders see it)
    return "%.30g" % v


def fuzz_model_texts(n_trials=12):
    """Model files whose numbers are spelt every which way (long decimals, exponents, subnormal magnitudes, integers, -0),
    with shuffled keys and odd whitespace."""
    rng = np.random.default_rng(77)
    dims = [(1, 3), (3, 2), (2, 1)]
    texts = []
    for trial in range(n_trials):
        layers = []
        for (ci, co) in dims:
            scale = 10.0 ** float(rng.integers(-3, 1))
            w = rng.standard_normal((co, ci, 3, 3)) * scale
            b = rng.standard_normal(co) * 0.1
            if trial % 3 == 0:
                w.flat[0], w.flat[1], w.flat[2], b[0] = 1.0, -0.0, 1e-42, 0.0          # integer-valued, negative zero, fp32-subnormal
            wtxt = "[" + ",".join("[" + ",".join("[" + ",".join("[" + ", ".join(_fmt_number(rng, v) for v in row) + "]" for row in k) + "]" for k in o) + "]" for o in w) + "]"
            btxt = "[" + ",\n ".join(_fmt_number(rng, v) for v in b) + "]"
            items = [('"nInputPlane"', str(ci)), ('"nOutputPlane"', str(co)), ('"kW"', "3"), ('"kH"', "3.0" if trial % 2 else "3"), ('"weight"', wtxt), ('"bias"', btxt)]
            order = rng.permutation(len(items))
            sep = ["", " ", "\n", "\t  "][trial % 4]
            layers.append("{" + ("," + sep).join(items[i][0] + sep + ":" + sep + items[i][1] for i in order) + "}")
        texts.append("[" + ",\n".join(layers) + "]\n")
    return texts


# ---------------------------------------------------------------------------------------------------
# recording
# ---------------------------------------------------------------------------------------------------
def _layer_texts(text):
    """the raw text of each layer object of a model file, spelt as in the file"""
    dec, i, out = json.JSONDecoder(), text.index("[") + 1, []
    while True:
        while text[i] in ", \n\r\t":
            i += 1
        if text[i] == "]":
            return out
        _, j = dec.raw_decode(text, i)
        out.append(text[i:j])
        i = j


def _library_runs(ref_dir, tmp):
    from oracle import oracle
    from oracle import reference_lib as R
    R.configure(4, 9)
    oms = {n: oracle.OracleModel.golden(n) for n in oracle.MODEL_NAMES}
    rms = {}
    for n, om in oms.items():
        om.write_json(os.path.join(tmp, f"{n}_model.json"))
        rms[n] = R.ReferenceModels(os.path.join(tmp, f"{n}_model.json"))
    runs = {"dims": {n: rm.dims for n, rm in rms.items()}}

    conv = {}
    for name in ("scale2.0x", "noise1"):
        for n_job in (1, 3, 4):
            R.configure(n_job, 9)
            for (w, h, seed) in CONVERT_SIZES:
                conv[f"{name}/j{n_job}/{w}x{h}"] = digest(rms[name].convert(oracle.seeded_plane(w, h, seed, "uniform"), True))
    runs["convert"] = conv

    R.configure(4, 6)
    split = {}
    for (w, h, seed) in SPLIT64_SIZES + ((96, 64, 8),):
        x = oracle.seeded_plane(w, h, seed, "uniform")
        split[f"{w}x{h}"] = {"split": digest(rms["scale2.0x"].convert(x, True)), "nosplit": digest(rms["scale2.0x"].convert(x, False))}
    runs["split64"] = split
    R.configure(4, 9)

    z = np.load(os.path.join(ROOT, "tests", "golden", "layers_32x24.npz"))
    runs["filter"] = [digest(rms["scale2.0x"].filter(li, z[f"in{li}"])) for li in range(rms["scale2.0x"].n)]
    runs["odd"] = {f"{w}x{h}": digest(rms["scale2.0x"].convert(oracle.seeded_plane(w, h, 10 + w, "uniform"), True)) for (w, h) in ODD_SIZES}
    R.configure(os.cpu_count() or 4, 9)
    runs["cfg1_scale2.0x_uniform"] = digest(rms["scale2.0x"].convert(oracle.seeded_plane(256, 256, 0, "uniform"), True))
    R.configure(4, 9)

    x = oracle.seeded_plane(40, 30, 9, "smooth")
    shipped = {}
    for name in oracle.MODEL_NAMES:
        real = R.ReferenceModels(os.path.join(ref_dir, "models", f"{name}_model.json"))
        shipped[name] = digest(real.convert(x, True))
        real.close()
    runs["shipped_models_smooth_40x30"] = shipped

    ident = os.path.join(tmp, "identity.json")
    identity_model_json(ident)
    rm = R.ReferenceModels(ident)
    full = {}
    for (w, h) in FULL_SIZES:
        x = oracle.seeded_plane(w, h, 3, "uniform") + np.float32(0.25)
        y, log = rm.convert_with_log(x, True)
        full[f"{w}x{h}"] = {"blocks": block_trace(log), "iterations_7": log.count("Iteration #7..."), "identity": bool(np.array_equal(y, x))}
    runs["identity_full_size"] = full
    rnd = []
    for exp, w, h in random_block_cases():
        R.configure(4, exp)
        x = oracle.seeded_plane(w, h, exp, "uniform") + np.float32(0.25)
        y, log = rm.convert_with_log(x, True)
        rnd.append({"exp": exp, "w": w, "h": h, "blocks": block_trace(log), "identity": bool(np.array_equal(y, x))})
    runs["identity_random_shapes"] = rnd
    rm.close()

    R.configure(2, 9)
    x = oracle.seeded_plane(23, 17, 5, "uniform")
    texts, outs = fuzz_model_texts(), []
    for trial, text in enumerate(texts):
        p = os.path.join(tmp, f"fuzz{trial}.json")
        with open(p, "w") as f:
            f.write(text)
        r = R.ReferenceModels(p)
        outs.append(digest(r.convert(x, True)))
        r.close()
    runs["json_fuzz"] = {"texts": texts, "outputs": outs}
    R.configure(4, 9)
    for r in rms.values():
        r.close()
    return runs


def _cli_runs(tmp):
    import cv2
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_cli import _test_image
    runs, images = {}, {}
    for mode, level, ratio, name in CLI_PIPELINE_CASES:
        d = tempfile.mkdtemp(dir=tmp)
        cv2.imwrite(os.path.join(d, "in.png"), _test_image(21, 17, 11))
        r = subprocess.run([REF_CLI, "-i", "in.png", "-m", mode, "--noise_level", str(level), "--scale_ratio", str(ratio),
                            "--model_dir", tmp, "-j", "4"], capture_output=True, text=True, cwd=d)
        assert r.returncode == 0, r.stdout + r.stderr
        key = f"{mode}/{level}/{ratio}"
        runs[key] = {"stdout": r.stdout, "files": sorted(f for f in os.listdir(d) if f != "in.png")}
        images[key] = cv2.imread(os.path.join(d, name), cv2.IMREAD_COLOR)
    fail = {}
    for args in CLI_FAIL_CASES:
        d = tempfile.mkdtemp(dir=tmp)
        cv2.imwrite(os.path.join(d, "in.png"), _test_image(16, 16))
        r = subprocess.run([REF_CLI, *args], capture_output=True, text=True, cwd=d)
        fail[cli_case_id(args)] = {"returncode": r.returncode, "stdout": norm_cli_text(r.stdout, REF_CLI), "stderr": norm_cli_text(r.stderr, REF_CLI)}
    r = subprocess.run([REF_CLI, "--help"], capture_output=True, text=True)
    return {"pipeline": runs, "fail": fail, "help": {"returncode": r.returncode, "stdout": norm_cli_text(r.stdout, REF_CLI)}}, images


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    ref_dir = sys.argv[1]
    sys.path.insert(0, ROOT)
    os.makedirs(OUT, exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        runs = _library_runs(ref_dir, tmp)
        runs["cli"], images = _cli_runs(tmp)
    with open(os.path.join(OUT, "runs.json"), "w") as f:
        json.dump(runs, f, indent=1)
    np.savez_compressed(os.path.join(OUT, "cli_images.npz"), **images)
    excerpts = {}
    for name in ("scale2.0x", "noise1", "noise2"):
        with open(os.path.join(ref_dir, "models", f"{name}_model.json")) as f:
            layers = _layer_texts(f.read())
        excerpts[name] = {str(li): layers[li] for li in EXCERPT_LAYERS}
    with gzip.GzipFile(os.path.join(OUT, "model_excerpts.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(excerpts).encode())
    print("written", OUT)


if __name__ == "__main__":
    main()
