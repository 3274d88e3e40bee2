"""The GNN half of the oracle is pinned to the reference's OWN saved TensorFlow graph.

tests/golden/gnn_<cfg>.npz hold the outputs of checkpoints/<cfg>/model-N.meta (the MetaGraphDef
train.py saved) executed node by node by oracle/graphdef.py on a seeded frame with the trained
weights (tools/make_golden.py).  Here:
* the protobuf wire reader is unit-tested on hand-encoded messages,
* oracle/gnn.py (the restatement every GPU parity test uses as its checker) must reproduce those
  vectors to 1e-5 for all seven shipped checkpoints,
* a restatement with a swapped concat / subtraction order must NOT (the vectors discriminate),
* the forward part of two saved graphs (tests/golden/checkpoints/, with the checkpoints rebuilt byte for byte by
  oracle/golden_checkpoint.py) is re-interpreted and must equal the fixtures.
"""
import glob
import json
import os
import struct

import numpy as np
import pytest

from conftest import ALL_CHECKPOINTS, GOLDEN, load_golden
from oracle import gnn as ognn
from oracle import graphdef

def _v(n):
    out = b''
    while True:
        b = n & 0x7F
        n >>= 7
        if n:
            out += bytes([b | 0x80])
        else:
            return out + bytes([b])


def _ld(num, payload):
    return _v(num << 3 | 2) + _v(len(payload)) + payload


def test_wire_reader_decodes_nodedef(tmp_path):
    # TensorProto{dtype=DT_FLOAT, shape=[2,2], tensor_content}
    shape = _ld(2, _v(1 << 3) + _v(2)) + _ld(2, _v(1 << 3) + _v(2))
    tensor = _v(1 << 3) + _v(1) + _ld(2, shape) + _ld(4, struct.pack('<4f', 1, 2, 3, 4))
    attr_value = _ld(8, tensor)
    attr_i = _v(3 << 3) + _v((1 << 64) - 2)                      # i = -2 (two's complement varint)
    node = (_ld(1, b'scope/op') + _ld(2, b'Const') + _ld(3, b'a:1') + _ld(3, b'^ctl')
            + _ld(5, _ld(1, b'value') + _ld(2, attr_value)) + _ld(5, _ld(1, b'axis') + _ld(2, attr_i)))
    meta = _ld(2, _ld(1, node))                                   # MetaGraphDef.graph_def.node
    path = str(tmp_path / 'meta.pb')
    with open(path, 'wb') as f:
        f.write(meta)
    nodes = graphdef.load_meta_graph(path)
    n = nodes['scope/op']
    assert n.op == 'Const' and n.inputs == ['a:1', '^ctl']
    interp = graphdef.GraphInterpreter(nodes, {}, {'a': np.zeros(1)})
    assert np.array_equal(interp.attr(n, 'value'), np.array([[1, 2], [3, 4]], np.float32))
    assert interp.attr(n, 'axis') == -2
    # splat-encoded constant: one float_val for a [3] tensor
    t = _v(1 << 3) + _v(1) + _ld(2, _ld(2, _v(1 << 3) + _v(3))) + _v(5 << 3 | 5) + struct.pack('<f', 7.5)
    assert np.array_equal(graphdef._tensor(memoryview(t)), np.full(3, 7.5, np.float32))


def test_interpreter_ops():
    x = np.arange(12, dtype=np.float32).reshape(4, 3)
    a = {'begin_mask': 1, 'end_mask': 1, 'shrink_axis_mask': 2, 'ellipsis_mask': 0, 'new_axis_mask': 0}
    assert np.array_equal(graphdef._strided_slice(x, [0, 1], [0, 2], [1, 1], a), x[:, 1])
    a = {'shrink_axis_mask': 1}
    assert graphdef._strided_slice(np.array([5, 6]), [0], [1], [1], a) == 5


def _predict(g):
    coords, keypoints, edges = g.graph_tuple()
    return ognn.predict(g.weights, g.layer_configs, g.config['num_classes'], 7, g.graph['intensity'], coords,
                        keypoints, edges, return_features=True)


@pytest.mark.parametrize('name', ALL_CHECKPOINTS)
def test_restatement_matches_reference_graph(name):
    g = load_golden(name)
    logits, boxes, feats = _predict(g)
    assert np.abs(logits - g.gnn['logits']).max() <= 1e-5
    assert np.abs(boxes - g.gnn['boxes']).max() <= 1e-5
    assert np.abs(feats[1] - g.gnn['features_pool']).max() <= 1e-5
    assert np.abs(feats[-1] - g.gnn['features_last']).max() <= 1e-5
    assert np.abs(ognn.postprocess(logits) - g.gnn['probs']).max() <= 1e-6
    with open(os.path.join(GOLDEN, 'graphdef_ops_%s.json' % name)) as f:
        ops = json.load(f)['ops_executed']
    num_gnn = sum(1 for l in g.layer_configs if l['type'] == 'scatter_max_graph_auto_center_net')
    assert ops['UnsortedSegmentMax'] == 1 + num_gnn and ops['Softmax'] == 1
    assert ops['MatMul'] == ops['BiasAdd'] == len([k for k in g.weights if k.endswith('/weights')])


def test_fixtures_discriminate_operand_order(monkeypatch):
    """A restatement with (dst - src) relative coordinates, or coordinates before features in the
    concat, misses the reference vectors by far more than any tolerance in this repo."""
    g = load_golden('car_auto_T3_train')
    real_concat = np.concatenate

    def swapped(arrs, axis=0, **kw):
        if axis in (-1, 1) and len(arrs) == 2 and arrs[1].shape[1] == 3:
            return real_concat([arrs[1], arrs[0]], axis=axis, **kw)
        return real_concat(arrs, axis=axis, **kw)

    monkeypatch.setattr(ognn.np, 'concatenate', swapped)
    try:
        logits, _, _ = _predict(g)
    finally:
        monkeypatch.undo()
    assert np.abs(logits - g.gnn['logits']).max() > 0.1


@pytest.mark.parametrize('name', ['car_auto_T1_train', 'car_fixed_T3_train'])
def test_live_saved_graph_equals_fixture(name, tmp_path):
    from oracle import golden_checkpoint
    from pointgnn_b200.utils import tf_checkpoint
    g = load_golden(name)
    ckpt = golden_checkpoint.rebuild(name, str(tmp_path))
    meta = sorted(glob.glob(os.path.join(ckpt, 'model-*.meta')))[-1]
    coords, keypoints, edges = g.graph_tuple()
    out = graphdef.run_forward(meta, tf_checkpoint.load_checkpoint(ckpt), g.graph['intensity'], coords, keypoints,
                               edges)
    assert np.array_equal(out['logits'], g.gnn['logits']) and np.array_equal(out['boxes'], g.gnn['boxes'])
    # the sub-graph is cut from the full training graph (forward + loss + gradients), not a toy, and executes the
    # same ops as the full graph did
    with open(os.path.join(GOLDEN, 'graphdef_ops_%s.json' % name)) as f:
        full = json.load(f)
    assert full['meta'] == os.path.basename(meta) and full['nodes_total'] > 5000
    assert out['ops'] == full['ops_executed']
