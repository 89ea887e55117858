"""The reference's OWN CLI -- src/main.cpp + src/modelHandler.cpp + src/convertRoutine.cpp compiled unmodified against
the OpenCV API shim (oracle/cvshim) -- pins:

  * the restated pipeline tests/test_cli.py::_reference_pipeline (cv2 plumbing + CPU oracle), which is what the GPU test
    of the product CLI is compared with: same pixels (<= 1 LSB), same auto output name, same progress lines;
  * the product CLI's flag surface: for every malformed / failing invocation both binaries give the same exit code and
    the same messages (no GPU needed: these paths end before any conversion).

What the reference CLI printed, returned and wrote for these invocations is stored in tests/golden/reference (recorded by
oracle/reference_golden.py)."""
import re
import subprocess

import numpy as np
import pytest

from oracle import reference_golden as RG

cv2 = pytest.importorskip("cv2")
from test_cli import _reference_pipeline, _test_image, cli  # noqa: E402,F401  (the product CLI fixture and the restated pipeline)


@pytest.fixture(scope="module")
def ref_cli():
    return RG.load()["cli"]


@pytest.mark.parametrize("mode,level,ratio,name", RG.CLI_PIPELINE_CASES)
def test_reference_cli_equals_the_restated_pipeline(ref_cli, oracle_models, ncpu, mode, level, ratio, name):
    bgr = _test_image(21, 17, 11)
    key = f"{mode}/{level}/{ratio}"
    run = ref_cli["pipeline"][key]
    assert run["stdout"].strip().endswith("process successfully done!")                  # src/main.cpp:192
    if "scale" in mode:
        assert "start scaling" in run["stdout"] and "#1 2x scaling..." in run["stdout"]  # :123,129-130
    assert "Iteration #7..." in run["stdout"]                                             # src/convertRoutine.cpp:67
    assert run["files"] == [name]                                                         # auto name rule, :173-189
    out = RG.cli_images()[key]
    ref = _reference_pipeline(bgr, mode, level, ratio, oracle_models, ncpu)
    assert out.shape == ref.shape
    diff = np.abs(out.astype(int) - ref.astype(int))
    assert diff.max() <= 1 and (diff > 0).mean() < 0.01                                   # 8-bit rounding ties only


@pytest.mark.parametrize("args", RG.CLI_FAIL_CASES, ids=[RG.cli_case_id(a) for a in RG.CLI_FAIL_CASES])
def test_product_cli_fails_exactly_like_the_reference_cli(cli, ref_cli, tmp_path, args):  # noqa: F811
    cv2.imwrite(str(tmp_path / "in.png"), _test_image(16, 16))
    ours = subprocess.run([cli, *args], capture_output=True, text=True, cwd=tmp_path)
    ref = ref_cli["fail"][RG.cli_case_id(args)]
    assert ours.returncode == ref["returncode"], (ours.returncode, ref["returncode"], ours.stderr, ref["stderr"])
    if args == ["--version"]:
        assert RG.norm_cli_text(ours.stdout, cli).split("version:")[1] == ref["stdout"].split("version:")[1]
        return
    # first line of the diagnostic: "PARSE ERROR: ..." + the offending argument, or the model loader's message
    def key_lines(normed):
        lines = [l for l in normed.splitlines() if l.strip()]
        return [l for l in lines if "PARSE ERROR" in l or "Argument" in l or "couldn't open" in l or "Required" in l or "Value" in l or "Couldn't" in l]
    assert key_lines(RG.norm_cli_text(ours.stderr, cli)) == key_lines(ref["stderr"]), (ours.stderr, ref["stderr"])


def test_help_lists_the_same_flags(cli, ref_cli):  # noqa: F811
    ours = subprocess.run([cli, "--help"], capture_output=True, text=True)
    ref = ref_cli["help"]
    assert ours.returncode == ref["returncode"] == 0
    flags = lambda t: sorted(set(re.findall(r"(?<![\w-])(--?[a-z_]+)", t)))
    ours_text = RG.norm_cli_text(ours.stdout, cli)
    assert flags(ours_text) == flags(ref["stdout"])
    for line in ("number of threads launching at the same time", "path to custom model directory (don't append last / )",
                 "custom scale ratio", "noise reduction level", "image processing mode", "waifu2x reimplementation using OpenCV"):
        assert line in ours_text and line in ref["stdout"], line
