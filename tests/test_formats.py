"""SavedModel / tensor-bundle formats on the CPU: oracle reader vs the reference's own fixture (shrunk to commit size,
tests/golden/make_golden.py), product C++ reader vs oracle reader, product writer -> both readers, golden known answers."""
import json
import os

import numpy as np
import pytest

from oracle import shifu_oracle as so
from oracle import tf_formats as tff

GOLDEN_DIR = os.path.join(os.path.dirname(__file__), "golden")
GOLDEN = os.path.join(GOLDEN_DIR, "dummydl_known_answers.json")
HEAD_LAYERS = (0, 1, 2, 20)       # the layers tests/golden/dummydl_head.npz holds whole


@pytest.fixture(scope="module")
def fixture_dir(tmp_path_factory):
    """The reference's dummydl SavedModel rebuilt from tests/golden: its serving graph and bundle index as TF wrote them,
    and a data shard of the original length with every stored tensor byte at its original offset.  The kernels of the
    17 middle layers are a seeded sample there; their other elements read as zeros."""
    d = tmp_path_factory.mktemp("dummydl")
    os.makedirs(d / "variables")
    (d / "saved_model.pb").write_bytes(open(os.path.join(GOLDEN_DIR, "dummydl_serving.pb"), "rb").read())
    index = open(os.path.join(GOLDEN_DIR, "dummydl_variables.index"), "rb").read()
    (d / "variables" / "variables.index").write_bytes(index)
    head = np.load(os.path.join(GOLDEN_DIR, "dummydl_head.npz"))
    sample = np.load(os.path.join(GOLDEN_DIR, "dummydl_sample.npz"))
    entries = {}
    for key, val in tff.read_table(str(d / "variables" / "variables.index")):
        if key:
            m = tff.parse_proto(val)
            entries[key.decode()] = ((tff._fields(m, 4) or [0])[0], (tff._fields(m, 5) or [0])[0])
    with open(d / "variables" / "variables.data-00000-of-00001", "wb") as f:
        f.truncate(int(sample["data_bytes"]))
        for l in range(21):
            name = "dense_%d/" % (46 + l)
            if l in HEAD_LAYERS:
                kernel = head["W%d" % HEAD_LAYERS.index(l)].ravel()
                spans = [(0, kernel)]
            else:
                idx, val = sample["W%d_idx" % l], sample["W%d_val" % l]
                spans = [(int(i), val[j:j + 1]) for j, i in enumerate(idx)]
            off, size = entries[name + "kernel"]
            for i, v in spans:
                assert 4 * (i + v.size) <= size
                f.seek(off + 4 * i); f.write(v.astype("<f4").tobytes())
            off, size = entries[name + "bias"]
            assert size == 4 * sample["b%d" % l].size
            f.seek(off); f.write(sample["b%d" % l].astype("<f4").tobytes())
    return str(d)


def _check_against_golden(layers):
    """every stored value of the fixture read back where it belongs"""
    head = np.load(os.path.join(GOLDEN_DIR, "dummydl_head.npz"))
    sample = np.load(os.path.join(GOLDEN_DIR, "dummydl_sample.npz"))
    for l, (W, b, _act) in enumerate(layers):
        np.testing.assert_array_equal(b, sample["b%d" % l])
        if l in HEAD_LAYERS:
            np.testing.assert_array_equal(W, head["W%d" % HEAD_LAYERS.index(l)])
        else:
            np.testing.assert_array_equal(W.ravel()[sample["W%d_idx" % l]], sample["W%d_val" % l])
    return sample


def test_crc32c_known_answers():
    assert tff.crc32c(b"123456789") == 0xE3069283          # the standard CRC-32C check value
    assert tff.crc32c(b"\x00" * 32) == 0x8A9136AA           # RFC 3720 B.4


def test_oracle_reader_on_reference_fixture_matches_golden(fixture_dir):
    """TensorflowModelTest.java:35-60 loads this model (inputs dense_46_input, output dense_66/Sigmoid).  The known
    answers run through the layers the fixture holds whole; the 17 middle layers are bridged by the activations the full
    model computes there (stored with the fixture)."""
    layers, names = tff.extract_mlp(fixture_dir, "dense_46_input", "dense_66/Sigmoid")
    assert len(layers) == 21 and layers[0][0].shape == (1522, 100) and layers[-1][0].shape == (100, 1)
    assert [l[2] for l in layers] == [so.ACT_RELU] * 20 + [so.ACT_SIGMOID]
    assert names == [("dense_%d/kernel" % i, "dense_%d/bias" % i) for i in range(46, 67)]
    sample = _check_against_golden(layers)
    g = json.load(open(GOLDEN))
    X = []
    for case in g["cases"]:
        if case["input_fn"] == "const":
            X.append(np.full((1, 1522), case["value"], np.float32))
        else:
            X.append(np.random.RandomState(case["seed"]).rand(case["rows"], 1522).astype(np.float32))
    X = np.concatenate(X)
    want = np.concatenate([np.asarray(case["expected"], np.float32) for case in g["cases"]])
    np.testing.assert_allclose(tff.mlp_forward(layers[:3], X), sample["A3"], atol=2e-6)
    np.testing.assert_allclose(tff.mlp_forward(layers[20:], sample["A20"]).ravel(), want, atol=2e-6)


def test_bundle_crcs_of_reference_fixture(fixture_dir):
    b = tff.read_bundle(os.path.join(fixture_dir, "variables", "variables"), verify_crc=False)
    assert b["dense_46/kernel"].shape == (1522, 100)
    # verify the stored per-tensor crc32c of two tensors (full verify of 27 MB in pure python is slow)
    entries = dict(tff.read_table(os.path.join(fixture_dir, "variables", "variables.index")))
    for key in (b"dense_66/bias", b"dense_66/kernel"):
        m = tff.parse_proto(entries[key])
        stored = [v for f, _, v in m if f == 6][0]
        assert tff.crc_mask(tff.crc32c(b[key.decode()].tobytes())) == stored


def test_cpp_reader_equals_oracle_reader_on_fixture(sb, fixture_dir):
    F, hidden, acts, out_act, flat = sb.capi.savedmodel_read(fixture_dir, "dense_46_input", "dense_66/Sigmoid")
    layers, _ = tff.extract_mlp(fixture_dir, "dense_46_input", "dense_66/Sigmoid")
    _check_against_golden(layers)
    assert F == 1522 and hidden == [100] * 20 and acts == [so.ACT_RELU] * 20 and out_act == so.ACT_SIGMOID
    ref = np.concatenate([np.concatenate([W.ravel(), b.ravel()]) for W, b, _ in layers])
    np.testing.assert_array_equal(flat, ref)


def test_writer_roundtrip_both_readers(sb, tmp_path):
    net = so.NetDesc(13, [8, 5, 3], [so.ACT_SIGMOID, so.ACT_TANH, so.ACT_LEAKYRELU])
    params = so.xavier_init(net, 9)
    flat = so.flatten_params(params)
    desc = sb.make_desc(13, net.hidden, net.acts)
    d = str(tmp_path / "export")
    sb.capi.savedmodel_write(d, desc, flat)
    assert sorted(os.listdir(d)) == ["GenericModelConfig.json", "saved_model.pb", "variables"]
    # product reader
    F, hidden, acts, out_act, got = sb.capi.savedmodel_read(d, "shifu_input_0", "shifu_output_0")
    assert (F, hidden, acts, out_act) == (13, [8, 5, 3], net.acts, so.ACT_SIGMOID)
    np.testing.assert_array_equal(got, flat)
    # independent oracle reader (checks block crcs and per-tensor crcs too)
    layers, names = tff.extract_mlp(d, "shifu_input_0", "shifu_output_0")
    assert names == [("weight_hidden_layer%d" % i, "biases_hidden_layer%d" % i) for i in range(3)] + \
        [("weight_shifu_output_0", "biases_shifu_output_0")]
    for (W, b, a), Wr, br in zip(layers, params[0::2], params[1::2]):
        np.testing.assert_array_equal(W, Wr); np.testing.assert_array_equal(b, br)
    tff.read_bundle(os.path.join(d, "variables", "variables"), verify_crc=True)
    # signature + GenericModelConfig.json exactly as export_generic_config writes it (ssgd_monitor.py:476-490)
    nodes, sigs = tff.read_graph_nodes(os.path.join(d, "saved_model.pb"))
    assert "serving_default" in sigs
    assert nodes["hidden_layer0"][0] == "Sigmoid" and nodes["shifu_output_0"][0] == "Sigmoid"
    assert nodes["MatMul_2"][1] == ["hidden_layer1", "weight_hidden_layer2/read"]
    cfg = json.load(open(os.path.join(d, "GenericModelConfig.json")))
    assert cfg == {"inputnames": ["shifu_input_0"],
                   "properties": {"algorithm": "tensorflow", "tags": ["serve"], "outputnames": "shifu_output_0",
                                  "normtype": "ZSCALE"}}


def test_reader_errors(sb, tmp_path):
    with pytest.raises(sb.ShifuB200Error) as e:
        sb.capi.savedmodel_read(str(tmp_path / "missing"), "a", "b")
    assert e.value.code == sb.capi.SB_ERR_IO
    net = so.NetDesc(4, [3], [so.ACT_RELU])
    d = str(tmp_path / "m")
    sb.capi.savedmodel_write(d, sb.make_desc(4, [3], [so.ACT_RELU]), so.flatten_params(so.xavier_init(net, 1)))
    with pytest.raises(sb.ShifuB200Error) as e:
        sb.capi.savedmodel_read(d, "shifu_input_0", "no_such_op")
    assert e.value.code == sb.capi.SB_ERR_FORMAT
    with pytest.raises(sb.ShifuB200Error):
        sb.capi.savedmodel_read(d, "shifu_input_0", "shifu_output_0", tag="train")
    # corrupt one byte of the index: block crc must catch it
    p = os.path.join(d, "variables", "variables.index")
    raw = bytearray(open(p, "rb").read()); raw[10] ^= 0xFF; open(p, "wb").write(bytes(raw))
    with pytest.raises(sb.ShifuB200Error) as e:
        sb.capi.savedmodel_read(d, "shifu_input_0", "shifu_output_0")
    assert e.value.code == sb.capi.SB_ERR_FORMAT


def test_writer_nodes_carry_the_attributes_tf_writes(sb, tmp_path):
    """Structural lint of our SavedModel writer against a GraphDef written by a real TF 1.x (the reference's dummydl
    fixture, attribute keys committed as tests/golden/dummydl_op_attrs.json): every op type we emit that TF also emitted
    there must carry exactly TF's attribute keys, minus the optional `_output_shapes` / `_class` hints (we may add
    `_class` colocation on Assign / Identity like TF does).  An importer rejects nodes with missing non-default attrs."""
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "dummydl_op_attrs.json")))["op_attr_keys"]
    net = so.NetDesc(13, [8, 5, 3], [so.ACT_SIGMOID, so.ACT_RELU, so.ACT_TANH])
    d = str(tmp_path / "export")
    sb.capi.savedmodel_write(d, sb.make_desc(13, net.hidden, net.acts), so.flatten_params(so.xavier_init(net, 9)))
    nodes, _ = tff.read_graph_nodes(os.path.join(d, "saved_model.pb"))
    ours = {}
    for _name, (op, _inputs, attrs) in nodes.items():
        ours.setdefault(op, set()).update(attrs.keys())
    optional = {"_output_shapes", "_class"}
    checked = 0
    for op, keys in ours.items():
        if op not in golden:
            assert op in ("Tanh", "LeakyRelu"), "op %s is not in the TF-written fixture" % op   # unary ops: attr T (+ alpha)
            continue
        assert keys - optional == set(golden[op]) - optional, (op, sorted(keys), golden[op])
        checked += 1
    assert checked >= 8 and {"Placeholder", "VariableV2", "MatMul", "Add", "Sigmoid", "RestoreV2", "Assign"} <= set(ours)
