"""Generates tests/golden/*.json|npz|pb|index from the reference's OWN artefacts; needs a checkout of the reference
project, whose SavedModel fixture is shifu-tensorflow-eval/src/test/resources/dummydl.  Run:

    python tests/golden/make_golden.py <path to dummydl>

dummydl_known_answers.json : forward outputs of the reference's SavedModel fixture
    (shifu-tensorflow-eval/src/test/resources/dummydl, loaded by TensorflowModelTest.java:35-60) computed by the
    oracle reader + fp32 numpy forward.  NOT TF-verified (TF is not installable here); they agree with the values
    SURVEY.md section 8c lists, which were derived independently.
dummydl_op_attrs.json : for every op type in the fixture's GraphDef (written by a real TF 1.x), the attribute keys its
    nodes carry, plus the attribute keys of the SignatureDef / SaverDef plumbing - the structural reference our own
    SavedModel writer is linted against (tests/test_formats.py).
dummydl_head.npz : the first 3 and the last layer of that model + a 16-row input/output pair, small enough to
    commit, so the GPU box can check the scorer kernels against the fixture's real weights.
dummydl_serving.pb, dummydl_variables.index, dummydl_sample.npz : the fixture shrunk to commit size (it is 4.6 MB of
    graph and 27 MB of variables), from which tests/test_formats.py rebuilds a SavedModel directory to read:
      * dummydl_serving.pb  the fixture's saved_model.pb with the "serve" meta graph only, its GraphDef cut down to the
        nodes the prediction output dense_66/Sigmoid depends on and its collection_defs dropped; every kept NodeDef,
        the MetaInfoDef, SaverDef and SignatureDef are the bytes TF wrote;
      * dummydl_variables.index  the bundle index, byte for byte;
      * dummydl_sample.npz  for each of the 21 layers its bias and a seeded sample of its kernel (the kernels of the
        layers in dummydl_head.npz are complete there), the length of the data shard, and the activations entering
        layer 3 and the output layer for the known-answer inputs, so the known answers stay checkable without the
        17 middle kernels.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import tf_formats as tff  # noqa: E402

INPUT, OUTPUT = "dense_46_input", "dense_66/Sigmoid"
HEAD = (0, 1, 2, 20)           # layers stored whole in dummydl_head.npz
KERNEL_SAMPLE = 256            # sampled elements per kernel of the other layers


def known_answer_inputs(cases):
    """the inputs of dummydl_known_answers.json, one row per expected value"""
    rows = []
    for case in cases:
        if case["input_fn"] == "const":
            rows.append(np.full((1, 1522), case["value"], np.float32))
        else:
            rows.append(np.random.RandomState(case["seed"]).rand(case["rows"], 1522).astype(np.float32))
    return np.concatenate(rows)


def _varint(v):
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _len_field(fn, payload):
    return _varint(fn << 3 | 2) + _varint(len(payload)) + payload


def serving_graph(fixture):
    """saved_model.pb -> the same SavedModel with only the serve meta graph and, in it, only the nodes OUTPUT depends on"""
    sm = tff.parse_proto(open(os.path.join(fixture, "saved_model.pb"), "rb").read())
    for mg_raw in tff._fields(sm, 2):
        mg = tff.parse_proto(mg_raw)
        tags = [t.decode() for mi in tff._fields(mg, 1) for t in tff._fields(tff.parse_proto(mi), 4)]
        if "serve" in tags:
            break
    else:
        raise ValueError("no serve meta graph")
    gd = tff.parse_proto(tff._fields(mg, 2)[0])
    raw = {}
    for nd_raw in tff._fields(gd, 1):
        nd = tff.parse_proto(nd_raw)
        raw[tff._fields(nd, 1)[0].decode()] = (nd_raw, [tff._strip(i.decode()) for i in tff._fields(nd, 3)])
    keep, todo = set(), [OUTPUT]
    while todo:
        n = todo.pop()
        if n not in keep:
            keep.add(n)
            todo.extend(raw[n][1])
    graph = b"".join(_len_field(1, raw[n][0]) for n in raw if n in keep)          # GraphDef order kept
    graph += b"".join(_len_field(fn, v) for fn, _, v in gd if fn != 1)             # versions, library
    meta = b"".join(_len_field(fn, graph if fn == 2 else v) for fn, _, v in mg if fn != 4)
    schema = b"".join(_varint(fn << 3) + _varint(v) for fn, wt, v in sm if fn == 1)
    return schema + _len_field(2, meta)


def main(fixture):
    layers, names = tff.extract_mlp(fixture, INPUT, OUTPUT)
    cases = []
    for value in (0.5, 0.0):
        X = np.full((1, 1522), value, np.float32)
        cases.append({"input_fn": "const", "value": value, "expected": [float(v) for v in tff.mlp_forward(layers, X).ravel()]})
    X = np.random.RandomState(0).rand(4, 1522).astype(np.float32)
    cases.append({"input_fn": "rand", "seed": 0, "rows": 4, "expected": [float(v) for v in tff.mlp_forward(layers, X).ravel()]})
    json.dump({"source": "dummydl fixture via oracle/tf_formats.py", "input": INPUT, "output": OUTPUT,
               "cases": cases}, open(os.path.join(HERE, "dummydl_known_answers.json"), "w"), indent=1)
    # reduced model: layers 0,1,2 + output layer (1522->100->100->100->1), fp16-free, ~650 KB compressed
    sub = [layers[i] for i in HEAD]
    X = np.random.RandomState(1).rand(16, 1522).astype(np.float32)
    Y = tff.mlp_forward(sub, X)
    np.savez_compressed(os.path.join(HERE, "dummydl_head.npz"), X=X, Y=Y,
                        **{"W%d" % i: l[0] for i, l in enumerate(sub)}, **{"b%d" % i: l[1] for i, l in enumerate(sub)})
    nodes, sigs = tff.read_graph_nodes(os.path.join(fixture, "saved_model.pb"))
    ops = {}
    for _name, (op, _inputs, attrs) in nodes.items():
        ops.setdefault(op, set()).update(attrs.keys())
    json.dump({"source": "dummydl/saved_model.pb (TF-written GraphDef), via oracle/tf_formats.read_graph_nodes",
               "op_attr_keys": {op: sorted(keys) for op, keys in sorted(ops.items())}, "signatures": sorted(sigs)},
              open(os.path.join(HERE, "dummydl_op_attrs.json"), "w"), indent=1)
    # shrunk fixture
    with open(os.path.join(HERE, "dummydl_serving.pb"), "wb") as f:
        f.write(serving_graph(fixture))
    index = os.path.join(fixture, "variables", "variables.index")
    with open(os.path.join(HERE, "dummydl_variables.index"), "wb") as f:
        f.write(open(index, "rb").read())
    rng = np.random.default_rng(20261017)
    sample = {"data_bytes": np.int64(os.path.getsize(os.path.join(fixture, "variables", "variables.data-00000-of-00001")))}
    for l, (W, b, _act) in enumerate(layers):
        sample["b%d" % l] = b
        if l not in HEAD:
            idx = np.sort(rng.choice(W.size, KERNEL_SAMPLE, replace=False))
            sample["W%d_idx" % l], sample["W%d_val" % l] = idx.astype(np.int32), W.ravel()[idx]
    X = known_answer_inputs(cases)
    sample["A3"] = tff.mlp_forward(layers[:3], X)           # enters layer 3
    sample["A20"] = tff.mlp_forward(layers[:20], X)         # enters the output layer
    np.savez_compressed(os.path.join(HERE, "dummydl_sample.npz"), **sample)
    print("wrote", sorted(os.listdir(HERE)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
