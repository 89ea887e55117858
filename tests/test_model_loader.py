"""Host side of the boundary: JSON model loader (w2x_model_load_json), in-memory constructor and the
tcgen05 operand packing.  No GPU needed."""
import json

import numpy as np
import pytest

from conftest import golden_path
from oracle import reference_golden as RG


def test_load_json_roundtrip_matches_golden_params(w2x, oracle_models, json_models):
    for name, path in json_models.items():
        m = w2x.Model.load_json(path)
        om = oracle_models[name]
        assert len(m) == 7
        for li in range(7):
            assert m.dims(li) == (om.dims[li][0], om.dims[li][1], 3)
            w, b = m.params(li)
            assert np.array_equal(w, om.weights[li])       # double -> float, src/modelHandler.cpp:96-97
            assert np.array_equal(b, om.biases[li])        # biases stay double


def test_load_reference_json_files_known_answers(w2x, oracle_models, tmp_path):
    """The first and last layer of each shipped model file, spelt as the reference ships them (tests/golden/reference)."""
    kat = json.load(open(golden_path("model_kat.json")))
    excerpts = RG.model_excerpts()
    for name in kat:
        for li, text in excerpts[name].items():
            li = int(li)
            path = tmp_path / f"{name}_layer{li}.json"
            path.write_text("[" + text + "]")
            m = w2x.Model.load_json(str(path))
            k = kat[name]["layers"][li]
            w, b = m.params(0)
            assert m.dims(0) == (*kat[name]["dims"][li], 3)
            assert float(w.reshape(-1)[0]) == k["w_first"] and float(w.reshape(-1)[-1]) == k["w_last"]
            assert float(b[0]) == k["b_first"] and float(b[-1]) == k["b_last"]
            assert float(w.astype(np.float64).sum()) == k["w_sum64"]
            assert np.array_equal(w, oracle_models[name].weights[li])
            assert np.array_equal(b, oracle_models[name].biases[li])


def test_key_order_whitespace_and_exponents(w2x, tmp_path):
    layer = {"nInputPlane": 1, "kH": 3, "bias": [1e-05, -2.5E+1], "kW": 3, "nOutputPlane": 2,
             "weight": [[[[1, -4.618060120265e-05, 3], [4, 5, 6], [7, 8, 0.1]]], [[[0, 0, 0], [0, 1.5, 0], [0, 0, -0.0]]]]}
    last = {"nInputPlane": 2, "nOutputPlane": 1, "kW": 3, "kH": 3, "bias": [0.25],
            "weight": [[[[0.5] * 3] * 3, [[0.125] * 3] * 3]]}
    p = tmp_path / "m.json"
    p.write_text(json.dumps([layer, last], indent=3))
    m = w2x.Model.load_json(str(p))
    w, b = m.params(0)
    assert w.dtype == np.float32 and w[0, 0, 0, 1] == np.float32(-4.618060120265e-05) and w[0, 0, 2, 2] == np.float32(0.1)
    assert b.tolist() == [1e-05, -25.0]
    assert m.dims(1) == (2, 1, 3)


def test_loader_error_paths(w2x, tmp_path):
    def expect(status, text=None, path=None):
        if path is None:
            path = tmp_path / "bad.json"
            path.write_text(text)
        with pytest.raises(w2x.W2xError) as ei:
            w2x.Model.load_json(str(path))
        assert ei.value.status == status, ei.value
        return ei.value.message

    assert "couldn't open" in expect(2, path=tmp_path / "missing.json")            # src/modelHandler.cpp:176-179
    assert "PicoJSON Error" in expect(3, "[{\"nInputPlane\": 1,")                  # :183-187
    expect(4, "{}")                                                                # root not an array
    sq = {"nInputPlane": 1, "nOutputPlane": 1, "kW": 3, "kH": 5, "bias": [0], "weight": [[[[0] * 3] * 5]]}
    assert "not square" in expect(4, json.dumps([sq]))                              # src/modelHandler.hpp:52-58
    k5 = {"nInputPlane": 1, "nOutputPlane": 1, "kW": 5, "kH": 5, "bias": [0], "weight": [[[[0] * 5] * 5]]}
    expect(4, json.dumps([k5]))                                                    # only 3x3 kernels exist in any model file
    ok = {"nInputPlane": 1, "nOutputPlane": 2, "kW": 3, "kH": 3, "bias": [0, 0], "weight": [[[[0] * 3] * 3]] * 2}
    chain = {"nInputPlane": 3, "nOutputPlane": 1, "kW": 3, "kH": 3, "bias": [0], "weight": [[[[0] * 3] * 3] * 3]}
    expect(4, json.dumps([ok, chain]))                                             # 2 planes out, 3 planes in
    short = dict(ok, bias=[0])
    expect(4, json.dumps([short]))
    expect(4, json.dumps([dict(ok, weight="x")]))
    # arrays of bare numbers take the reader's flat fast path: where arrays were expected the diagnostics are still the
    # element-by-element ones, and a mixed array falls back to the generic path
    assert "is not an object" in expect(4, "[1, 2, 3]")
    assert "weight has 3 output planes" in expect(4, json.dumps([dict(ok, weight=[1, 2, 3])]))
    assert "weight[o] is not an array" in expect(4, json.dumps([dict(ok, weight=[1, 2])]))
    assert "kernel matrix has too few rows" in expect(4, json.dumps([dict(ok, weight=[[7], [7]])]))
    assert "kernel row has too few columns" in expect(4, json.dumps([dict(ok, weight=[[[1, 2, 3]], [[1, 2, 3]]])]))
    assert "kernel row has too few columns" in expect(4, json.dumps([dict(ok, weight=[[[[0, 0], [0, 0, 0], [0, 0, 0]]]] * 2)]))
    assert "non-numeric weight" in expect(4, json.dumps([dict(ok, weight=[[[[0, "a", 0], [0, 0, 0], [0, 0, 0]]]] * 2)]))
    assert "non-numeric bias" in expect(4, json.dumps([dict(ok, bias=[0, None])]))
    assert "PicoJSON Error" in expect(3, "[{\"nInputPlane\": 1, \"bias\": [1, 2e+, 3]}]")          # malformed number inside a numeric array
    mixed = dict(ok, weight=[[[[0, 1.5e-3, -2], [0, 0, 0], [0, 0, 0, "extra columns are ignored"]]]] * 2)
    m = w2x.Model.load_json(str((tmp_path / "mixed.json").write_text(json.dumps([mixed])) and tmp_path / "mixed.json"))
    assert m.params(0)[0][0, 0, 0].tolist() == [0.0, float(np.float32(1.5e-3)), -2.0]


def test_model_create_from_arrays(w2x, oracle_models):
    om = oracle_models["noise2"]
    m = w2x.Model.from_arrays(om.weights, om.biases)
    for li in range(7):
        w, b = m.params(li)
        assert np.array_equal(w, om.weights[li]) and np.array_equal(b, om.biases[li])


def _swizzle(off, row_bytes):
    mask = row_bytes // 16 - 1
    return off ^ (((off >> 7) & mask) << 4)


def test_tc_operand_pack_layout_and_split(w2x, oracle_models):
    """[32-ch block][tap][hi|lo][n_out x 32] fp16, K-major rows of 64 B, 16-byte units XOR-swizzled
    (SWIZZLE_64B); hi+lo == w*scale to ~22 bits."""
    m = w2x.Model.from_arrays(oracle_models["scale2.0x"].weights, oracle_models["scale2.0x"].biases)
    assert m.debug_tc_pack(0)[0] is None and m.debug_tc_pack(6)[0] is None      # 1->32 and 128->1 are not MMA layers
    for li in range(1, 6):
        data, nch, kbl, ws = m.debug_tc_pack(li)
        w = oracle_models["scale2.0x"].weights[li]
        co, ci = w.shape[:2]
        kc_a = 32                          # channels per staged activation box (one block of 128-byte records)
        assert nch == ci // kc_a and kbl == kc_a // 32 and ws == 2.0 ** np.floor(np.log2(1024.0 / np.abs(w).max()))
        data = data.view(np.float16).reshape(nch, 9, kbl, 2, co * 32)
        ws_w = (w * np.float32(ws)).astype(np.float32)
        hi = ws_w.astype(np.float16)
        lo = (ws_w - hi.astype(np.float32)).astype(np.float16)
        n_idx, k_idx = np.meshgrid(np.arange(co), np.arange(32), indexing="ij")
        off = np.vectorize(_swizzle)(n_idx * 64 + 2 * k_idx, 64) // 2
        for c in range(nch):
            for t in range(9):
                for kb in range(kbl):
                    c0 = c * kc_a + kb * 32
                    exp_hi = hi[:, c0:c0 + 32, t // 3, t % 3]
                    exp_lo = lo[:, c0:c0 + 32, t // 3, t % 3]
                    assert np.array_equal(data[c, t, kb, 0][off].view(np.uint16), exp_hi.view(np.uint16)), (li, c, t, kb)
                    assert np.array_equal(data[c, t, kb, 1][off].view(np.uint16), exp_lo.view(np.uint16)), (li, c, t, kb)
        # the split keeps ~22 significant bits: |w*s - (hi+lo)| <= 2^-22 |w*s| + 2^-25
        res = np.abs(ws_w.astype(np.float64) - hi.astype(np.float64) - lo.astype(np.float64))
        assert np.all(res <= 2.0 ** -22 * np.abs(ws_w) + 2.0 ** -25)


def test_f16_rounding_edge_cases_via_pack(w2x):
    """The host f32->f16 converter (round-to-nearest-even incl. subnormals) against numpy, through a
    32->32 layer whose weights are the probe values (scale is 1 when max|w| is in (512,1024])."""
    probes = np.array([1000.0, 0.0, -0.0, 1.0, 1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 65504.0 / 128, 2.0 ** -14, 2.0 ** -15,
                       2.0 ** -24, 2.0 ** -25, 1.5 * 2.0 ** -25, 3 * 2.0 ** -25, 6.1e-5, 5.96e-8, 1e-9, -0.333, 0.1,
                       2.0 ** -14 - 2.0 ** -26, 512.25, 999.9, 2.5 * 2.0 ** -24], np.float32)
    rng = np.random.default_rng(4)
    w = np.zeros((32, 32, 3, 3), np.float32)
    flat = w.reshape(-1)
    flat[:probes.size] = probes
    flat[probes.size:] = (rng.standard_normal(flat.size - probes.size) * np.exp(rng.uniform(-18, 5, flat.size - probes.size))).astype(np.float32)
    flat[probes.size:] = np.clip(flat[probes.size:], -1000, 1000)
    first = np.zeros((32, 1, 3, 3), np.float32)
    last = np.zeros((1, 32, 3, 3), np.float32)
    m = w2x.Model.from_arrays([first, w, last], [np.zeros(32), np.zeros(32), np.zeros(1)])
    data, nch, kbl, ws = m.debug_tc_pack(1)
    assert ws == 1.0 and nch == 1 and kbl == 1
    data = data.reshape(1, 9, 2, 32 * 32)
    hi = w.astype(np.float16)
    lo = (w - hi.astype(np.float32)).astype(np.float16)
    n_idx, k_idx = np.meshgrid(np.arange(32), np.arange(32), indexing="ij")
    off = np.vectorize(_swizzle)(n_idx * 64 + 2 * k_idx, 64) // 2
    for t in range(9):
        assert np.array_equal(data[0, t, 0][off], hi[:, :, t // 3, t % 3].view(np.uint16))
        assert np.array_equal(data[0, t, 1][off], lo[:, :, t // 3, t % 3].view(np.uint16))
