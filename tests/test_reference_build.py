"""The reference's OWN hot-path sources (src/modelHandler.cpp, src/convertRoutine.cpp), compiled against the OpenCV API
shim in oracle/cvshim, pin the restated oracle and the golden vectors against the reference's real control flow:
picojson model loading, the thread partition of Model::filter, the layer loop, replicate padding, the block-split
arithmetic, crop and stitch.

What that build computed on the seeded inputs below is stored in tests/golden/reference (recorded by
oracle/reference_golden.py): digests of every output compared bit for bit, and the block order traced from its progress
output.  The model JSONs it read were written from tests/golden/models."""
import numpy as np
import pytest

from conftest import golden_path
from oracle import reference_golden as RG

# restated fp32 arithmetic of the shim vs OpenCV's SIMD kernels: re-association / FMA only
SHIM_VS_CV2_TOL = 3e-6


@pytest.fixture(scope="module")
def ref():
    return RG.load()


def test_reference_loader_reads_the_model_files(ref, oracle_models):
    for name, om in oracle_models.items():
        assert len(ref["dims"][name]) == 7 and [tuple(d) for d in ref["dims"][name]] == [tuple(d) for d in om.dims]


@pytest.mark.parametrize("name", ["scale2.0x", "noise1"])
@pytest.mark.parametrize("n_job", [1, 3, 4])
def test_oracle_is_bit_identical_to_the_reference_control_flow(ref, oracle_mod, oracle_models, name, n_job):
    """convertWithModels, no-split path (src/convertRoutine.cpp:31-48), for every thread partition the reference forms
    (nOutputPlanes / nJob with the remainder on the last thread, src/modelHandler.cpp:46-65)."""
    for (w, h, seed) in RG.CONVERT_SIZES:
        x = oracle_mod.seeded_plane(w, h, seed, "uniform")
        y_orc = oracle_models[name].convert(x, n_job=n_job)
        assert y_orc.shape == (h, w)
        assert RG.digest(y_orc) == ref["convert"][f"{name}/j{n_job}/{w}x{h}"], (w, h)


def test_block_split_path_is_bit_identical(ref, oracle_mod, oracle_models):
    """convertWithModelsBlockSplit (src/convertRoutine.cpp:84-169) with 64x64 blocks (threshold 64*64*3/2 = 6144 px):
    block rectangles, last-block handling, crop and stitch -- against the oracle's restatement and against no-split."""
    om = oracle_models["scale2.0x"]
    for (w, h, seed) in RG.SPLIT64_SIZES:
        assert w * h > 6144
        x = oracle_mod.seeded_plane(w, h, seed, "uniform")
        y_split, y_nosplit = om.convert(x, True, block=(64, 64)), om.convert(x, False)
        assert RG.digest(y_split) == ref["split64"][f"{w}x{h}"]["split"], (w, h)
        assert RG.digest(y_nosplit) == ref["split64"][f"{w}x{h}"]["nosplit"], (w, h)
        assert np.abs(y_split - y_nosplit).max() <= 1e-6, (w, h)
    x = oracle_mod.seeded_plane(96, 64, 8, "uniform")            # exactly AT the threshold: the reference does not split
    assert ref["split64"]["96x64"]["split"] == ref["split64"]["96x64"]["nosplit"]
    assert RG.digest(om.convert(x, True, block=(64, 64))) == ref["split64"]["96x64"]["split"]


def test_model_filter_per_layer(ref, oracle_models):
    """Model::filter of every layer on the golden 32x24 inputs: bit-equal to the oracle, within fp32 re-association of cv2."""
    z = np.load(golden_path("layers_32x24.npz"))
    om = oracle_models["scale2.0x"]
    assert len(ref["filter"]) == len(om)
    for li in range(len(om)):
        out = om.filter(li, z[f"in{li}"], n_job=4)
        assert RG.digest(out) == ref["filter"][li], li
        assert np.abs(out - z[f"out{li}"]).max() <= SHIM_VS_CV2_TOL * max(1.0, float(np.abs(z[f"out{li}"]).max())), li


def test_reference_control_flow_reproduces_the_cv2_golden_odd_sizes(ref, oracle_mod, oracle_models):
    z = np.load(golden_path("odd_sizes.npz"))
    for (w, h) in RG.ODD_SIZES:
        y = oracle_models["scale2.0x"].convert(oracle_mod.seeded_plane(w, h, 10 + w, "uniform"))
        assert RG.digest(y) == ref["odd"][f"{w}x{h}"], (w, h)
        assert np.abs(y - z[f"out_{w}x{h}"]).max() <= SHIM_VS_CV2_TOL


@pytest.mark.slow
def test_cfg1_256_reference_control_flow_vs_cv2_golden(ref, oracle_mod, oracle_models, ncpu):
    """BASELINE config 1 through the reference's own code (shim arithmetic) against the output of real OpenCV arithmetic."""
    y = oracle_models["scale2.0x"].convert(oracle_mod.seeded_plane(256, 256, 0, "uniform"), n_job=ncpu)
    assert RG.digest(y) == ref["cfg1_scale2.0x_uniform"]
    g = np.load(golden_path("cfg1_scale2.0x_uniform.npy"))
    assert np.abs(y - g).max() <= SHIM_VS_CV2_TOL


def test_shipped_model_files_equal_the_golden_weights(ref, oracle_mod, oracle_models):
    """The reference's real JSON files through its real loader give the same output bits as the committed weights
    (i.e. the committed weights ARE the shipped weights after double->float)."""
    x = oracle_mod.seeded_plane(40, 30, 9, "smooth")
    for name in ("scale2.0x", "noise1", "noise2"):
        assert RG.digest(oracle_models[name].convert(x)) == ref["shipped_models_smooth_40x30"][name], name


@pytest.mark.parametrize("w,h", RG.FULL_SIZES)
def test_block_order_and_split_decision_of_the_reference_at_full_size(w2x, ref, w, h):
    """BASELINE shapes through the reference's own convertWithModels with a 7-layer identity model: the split decision and
    the (c, r) processing order it prints (src/convertRoutine.cpp:25-26,100-134) are the product's w2x_requires_splitting /
    w2x_block_table, block for block; and the stitched output is the input (every pixel written exactly once)."""
    run = ref["identity_full_size"][f"{w}x{h}"]
    assert run["identity"]
    blocks = [tuple(b) for b in run["blocks"]]
    assert (len(blocks) > 0) == w2x.requires_splitting(w, h)
    if blocks:
        tab, sc, sr = w2x.block_table(w, h, 7)
        assert [(int(t[1]), int(t[0])) for t in tab] == blocks          # table rows are (r, c, ...): reference order = r outer, c inner
        assert sc * sr == len(blocks)
        assert run["iterations_7"] == len(blocks)
    else:
        assert run["iterations_7"] == 1


def test_block_arithmetic_against_the_reference_on_random_shapes(w2x, ref):
    """Seeded random plane sizes x block sizes 2^5..2^9: the reference's own split decision and block order (traced through
    its progress output with the identity model) against w2x_requires_splitting / w2x_block_table -- including planes
    thinner than a block, last blocks of 1 row / column, and sizes exactly at the split threshold."""
    runs = ref["identity_random_shapes"]
    try:
        for r in runs:
            exp, w, h = r["exp"], r["w"], r["h"]
            w2x.set_block_size_exp2_square(exp)
            assert r["identity"], (exp, w, h)
            blocks = [tuple(b) for b in r["blocks"]]
            assert (len(blocks) > 0) == w2x.requires_splitting(w, h), (exp, w, h)
            if blocks:
                tab, sc, sr = w2x.block_table(w, h, 7)
                assert [(int(t[1]), int(t[0])) for t in tab] == blocks, (exp, w, h)
    finally:
        w2x.set_block_size_exp2_square(9)


def test_json_number_parsing_agrees_with_the_reference_loader(w2x, ref, oracle_mod, tmp_path):
    """The product's loader (csrc/model.cpp: hand-written JSON reader, std::from_chars, double -> float) against the
    reference's (picojson + strtod, src/modelHandler.cpp:74-115) on model files whose numbers are spelt every which way
    (long decimals, exponents, subnormal magnitudes, integers, -0), with shuffled keys and odd whitespace.  The weights
    the product parsed are run through the oracle and compared with what the reference's own loader and
    convertWithModels made of the same file: one differing ulp in any weight or bias would show up in the output bits."""
    x = oracle_mod.seeded_plane(23, 17, 5, "uniform")
    fuzz = ref["json_fuzz"]
    for trial, text in enumerate(fuzz["texts"]):
        path = tmp_path / f"fuzz{trial}.json"
        path.write_text(text)
        m = w2x.Model.load_json(str(path))
        ws, bs = zip(*[m.params(li) for li in range(len(m))])
        ours = oracle_mod.OracleModel(list(ws), list(bs)).convert(x, n_job=2)
        assert RG.digest(ours) == fuzz["outputs"][trial], trial
