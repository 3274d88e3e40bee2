"""The reference's OWN frozen TensorFlow graph, executed in NumPy.

TEST INFRASTRUCTURE (see oracle/__init__.py).  ``train.py`` saves, next to every
checkpoint, ``model-N.meta``: a serialised ``MetaGraphDef`` holding the exact op
graph that ``models/models.py::predict`` + ``models/gnn.py`` BUILT under
TensorFlow 1.15 (/root/reference/train.py:578-593 -> tf.train.Saver.save).  That
graph is the reference itself, not a restatement: every Gather / ConcatV2 / Sub /
MatMul / BiasAdd / Relu / UnsortedSegmentMax node, its input order and its
attributes are what the reference's Python emitted.  TensorFlow cannot be
installed here, so this module

1. decodes the protobuf wire format by hand (MetaGraphDef.graph_def = field 2,
   GraphDef.node = field 1, NodeDef{name=1, op=2, input=3, attr=5}, AttrValue,
   TensorProto, TensorShapeProto - field numbers from tensorflow/core/framework/
   *.proto, r1.15), and
2. interprets the forward sub-graph of tower 0 (placeholders -> logits / box
   encodings / Softmax) with NumPy, each op following its TF kernel's documented
   semantics (fp32; ``UnsortedSegmentMax`` initialises with
   numeric_limits<float>::lowest()).

The variables (``VariableV2`` nodes) are read from the checkpoint's data file by
name.  Used by tools/make_golden.py to produce tests/golden/gnn_*.npz and by
tests/test_graphdef_cpu.py (on the forward sub-graphs kept under
tests/golden/checkpoints/) to pin oracle/gnn.py - and through it the CUDA path -
to the reference.
"""
import struct

import numpy as np

# --------------------------------------------------------------------------------------------
# protobuf wire format
# --------------------------------------------------------------------------------------------


def _varint(buf, pos):
    result = 0
    shift = 0
    while True:
        b = buf[pos]
        pos += 1
        result |= (b & 0x7F) << shift
        if not b & 0x80:
            return result, pos
        shift += 7


def fields(buf):
    """Yield (field_number, wire_type, value) of one message; value is int or a memoryview."""
    pos = 0
    n = len(buf)
    while pos < n:
        key, pos = _varint(buf, pos)
        num, wt = key >> 3, key & 7
        if wt == 0:
            val, pos = _varint(buf, pos)
        elif wt == 1:
            val = buf[pos:pos + 8]
            pos += 8
        elif wt == 2:
            ln, pos = _varint(buf, pos)
            val = buf[pos:pos + ln]
            pos += ln
        elif wt == 5:
            val = buf[pos:pos + 4]
            pos += 4
        else:
            raise ValueError('unsupported protobuf wire type %d' % wt)
        yield num, wt, val


def _signed(v):
    return v - (1 << 64) if v >= (1 << 63) else v


_DTYPES = {1: np.float32, 2: np.float64, 3: np.int32, 4: np.uint8, 6: np.int8, 9: np.int64, 10: np.bool_}


def _shape(buf):
    """TensorShapeProto: dim = 2 {size = 1}; unknown_rank = 3."""
    dims = []
    unknown = False
    for num, _, val in fields(buf):
        if num == 2:
            size = 0
            for n2, _, v2 in fields(val):
                if n2 == 1:
                    size = _signed(v2)
            dims.append(size)
        elif num == 3:
            unknown = bool(val)
    return None if unknown else tuple(dims)


def _packed(val, wt, fmt, size):
    if wt == 2:
        return list(struct.unpack('<%d%s' % (len(val) // size, fmt), bytes(val)))
    return [struct.unpack('<' + fmt, bytes(val))[0]]


def _packed_varints(val, wt):
    if wt != 2:
        return [_signed(val)]
    out = []
    pos = 0
    while pos < len(val):
        v, pos = _varint(val, pos)
        out.append(_signed(v))
    return out


def _tensor(buf):
    """TensorProto -> ndarray (dtype=1, tensor_shape=2, tensor_content=4, *_val = 5/6/7/10/11)."""
    dtype, shape, content, vals = None, (), None, []
    for num, wt, val in fields(buf):
        if num == 1:
            dtype = val
        elif num == 2:
            shape = _shape(val)
        elif num == 4:
            content = bytes(val)
        elif num == 5:
            vals += _packed(val, wt, 'f', 4)
        elif num == 6:
            vals += _packed(val, wt, 'd', 8)
        elif num in (7, 10, 11):
            vals += _packed_varints(val, wt)
        elif num == 8:
            vals.append(bytes(val))
    if dtype == 7:          # DT_STRING
        return np.array(vals, dtype=object).reshape(shape)
    np_dtype = _DTYPES[dtype]
    count = int(np.prod(shape)) if shape else 1
    if content is not None and len(content):
        return np.frombuffer(content, dtype=np_dtype).reshape(shape).copy()
    if len(vals) == 0:
        return np.zeros(shape, np_dtype)
    arr = np.array(vals, dtype=np_dtype)
    if arr.size == 1 and count != 1:
        arr = np.full(count, arr[0], dtype=np_dtype)       # splat encoding
    elif arr.size < count:
        arr = np.concatenate([arr, np.full(count - arr.size, arr[-1], np_dtype)])
    return arr.reshape(shape)


def _attr_value(buf):
    """AttrValue oneof: list=1, s=2, i=3, f=4, b=5, type=6, shape=7, tensor=8."""
    for num, wt, val in fields(buf):
        if num == 2:
            return bytes(val)
        if num == 3:
            return _signed(val)
        if num == 4:
            return struct.unpack('<f', bytes(val))[0]
        if num == 5:
            return bool(val)
        if num == 6:
            return ('type', val)
        if num == 7:
            return ('shape', _shape(val))
        if num == 8:
            return _tensor(val)
        if num == 1:
            out = []
            for n2, w2, v2 in fields(val):
                if n2 == 2:
                    out.append(bytes(v2))
                elif n2 == 3:
                    out += _packed_varints(v2, w2)
                elif n2 == 6:
                    out += [('type', t) for t in _packed_varints(v2, w2)]
                elif n2 == 7:
                    out.append(('shape', _shape(v2)))
            return out
    return None


class Node(object):
    __slots__ = ('name', 'op', 'inputs', 'attr')

    def __init__(self, name, op, inputs, attr):
        self.name, self.op, self.inputs, self.attr = name, op, inputs, attr

    def __repr__(self):
        return 'Node(%s, %s, %s)' % (self.name, self.op, self.inputs)


def _node(buf):
    name = op = ''
    inputs, attr = [], {}
    for num, _, val in fields(buf):
        if num == 1:
            name = bytes(val).decode()
        elif num == 2:
            op = bytes(val).decode()
        elif num == 3:
            inputs.append(bytes(val).decode())
        elif num == 5:
            key, value = None, None
            for n2, _, v2 in fields(val):
                if n2 == 1:
                    key = bytes(v2).decode()
                elif n2 == 2:
                    value = v2
            attr[key] = value          # decoded lazily (Const tensors can be large)
    return Node(name, op, inputs, attr)


def load_meta_graph(path):
    """-> {node name: Node} of MetaGraphDef.graph_def."""
    with open(path, 'rb') as f:
        buf = memoryview(f.read())
    nodes = {}
    for num, _, val in fields(buf):
        if num == 2:                              # graph_def
            for n2, _, v2 in fields(val):
                if n2 == 1:                       # node
                    node = _node(v2)
                    nodes[node.name] = node
    return nodes


# --------------------------------------------------------------------------------------------
# NumPy interpreter of the forward sub-graph
# --------------------------------------------------------------------------------------------
FLT_LOWEST = np.float32(-3.4028234663852886e38)


def _strided_slice(x, begin, end, strides, a):
    """tf.strided_slice with begin/end/ellipsis/new_axis/shrink_axis masks (dense spec)."""
    begin_mask, end_mask = a.get('begin_mask', 0), a.get('end_mask', 0)
    ellipsis_mask, new_axis_mask = a.get('ellipsis_mask', 0), a.get('new_axis_mask', 0)
    shrink_mask = a.get('shrink_axis_mask', 0)
    index = []
    for i in range(len(begin)):
        bit = 1 << i
        if ellipsis_mask & bit:
            index.append(Ellipsis)
        elif new_axis_mask & bit:
            index.append(np.newaxis)
        elif shrink_mask & bit:
            index.append(int(begin[i]))
        else:
            b = None if begin_mask & bit else int(begin[i])
            e = None if end_mask & bit else int(end[i])
            index.append(slice(b, e, int(strides[i])))
    return x[tuple(index)]


class GraphInterpreter(object):
    """Evaluates nodes of a TF-1 GraphDef on demand (memoised), fp32 throughout.

    feeds:     {placeholder node name: array}
    variables: {variable name: array} (the checkpoint), looked up by VariableV2 node name.
    """

    def __init__(self, nodes, variables, feeds):
        self.nodes = nodes
        self.variables = variables
        self.cache = {}
        self.ops_used = {}
        for k, v in feeds.items():
            self.cache[(k, 0)] = v

    def attr(self, node, key, default=None):
        raw = node.attr.get(key)
        if raw is None:
            return default
        if isinstance(raw, memoryview):
            raw = _attr_value(raw)
            node.attr[key] = raw if raw is not None else default
        return node.attr[key]

    def value(self, ref):
        if ref.startswith('^'):
            raise ValueError('control input %s' % ref)
        name, _, port = ref.partition(':')
        port = int(port) if port else 0
        key = (name, port)
        if key not in self.cache:
            # iterative evaluation (the chains are deeper than Python's recursion limit allows for some graphs)
            stack = [name]
            while stack:
                cur = stack[-1]
                if (cur, 0) in self.cache:
                    stack.pop()
                    continue
                node = self.nodes[cur]
                missing = [i.partition(':')[0] for i in node.inputs
                           if not i.startswith('^') and (i.partition(':')[0], 0) not in self.cache]
                if missing:
                    stack.extend(missing)
                    continue
                outs = self._run(node)
                if not isinstance(outs, tuple):
                    outs = (outs,)
                for p, o in enumerate(outs):
                    self.cache[(cur, p)] = o
                stack.pop()
        return self.cache[key]

    def _in(self, node):
        out = []
        for i in node.inputs:
            if i.startswith('^'):
                continue
            name, _, port = i.partition(':')
            out.append(self.cache[(name, int(port) if port else 0)])
        return out

    def _run(self, node):
        op = node.op
        self.ops_used[op] = self.ops_used.get(op, 0) + 1
        x = self._in(node)
        if op == 'Placeholder':
            raise KeyError('placeholder %s was not fed' % node.name)
        if op == 'Const':
            return self.attr(node, 'value')
        if op in ('Identity', 'StopGradient', 'Snapshot'):
            return x[0]
        if op in ('VariableV2', 'Variable'):
            return self.variables[node.name]
        if op == 'MatMul':
            a, b = x
            if self.attr(node, 'transpose_a', False):
                a = a.T
            if self.attr(node, 'transpose_b', False):
                b = b.T
            return np.matmul(a, b)
        if op == 'BiasAdd':
            return x[0] + x[1]
        if op in ('Add', 'AddV2'):
            return x[0] + x[1]
        if op == 'Sub':
            return x[0] - x[1]
        if op == 'Mul':
            return x[0] * x[1]
        if op == 'Relu':
            return np.maximum(x[0], 0)
        if op in ('GatherV2', 'Gather'):
            axis = int(x[2]) if len(x) > 2 else 0
            return np.take(x[0], x[1], axis=axis)
        if op == 'ConcatV2':
            return np.concatenate(x[:-1], axis=int(x[-1]))
        if op == 'ExpandDims':
            return np.expand_dims(x[0], int(x[1]))
        if op == 'Squeeze':
            dims = self.attr(node, 'squeeze_dims', [])
            return np.squeeze(x[0], axis=tuple(dims) if dims else None)
        if op == 'Pack':
            return np.stack(x, axis=int(self.attr(node, 'axis', 0)))
        if op == 'Shape':
            return np.array(x[0].shape, dtype=np.int32)
        if op == 'Reshape':
            return x[0].reshape([int(v) for v in x[1]])
        if op == 'Cast':
            return x[0].astype(_DTYPES[self.attr(node, 'DstT')[1]])
        if op == 'StridedSlice':
            a = {k: self.attr(node, k, 0) for k in ('begin_mask', 'end_mask', 'ellipsis_mask',
                                                     'new_axis_mask', 'shrink_axis_mask')}
            return _strided_slice(x[0], x[1], x[2], x[3], a)
        if op == 'UnsortedSegmentMax':
            data, ids, num = x[0], np.asarray(x[1]).reshape(-1), int(x[2])
            out = np.full((num,) + data.shape[1:], FLT_LOWEST, dtype=data.dtype)
            np.maximum.at(out, ids, data)
            return out
        if op == 'Softmax':
            z = x[0] - x[0].max(axis=-1, keepdims=True)
            e = np.exp(z)
            return e / e.sum(axis=-1, keepdims=True)
        raise NotImplementedError('op %s (node %s) is not part of the forward sub-graph' % (op, node.name))


# --------------------------------------------------------------------------------------------
# tower-0 forward pass of a saved Point-GNN model
# --------------------------------------------------------------------------------------------
LOGITS_NODE = 'output/predictor/cls/fully_connected_1/BiasAdd'
BOXES_NODE = 'output/predictor/concat'
PROBS_NODE = 'Softmax'


def _closure(nodes, roots):
    seen = set()
    stack = list(roots)
    while stack:
        n = stack.pop()
        if n in seen:
            continue
        seen.add(n)
        for i in nodes[n].inputs:
            stack.append(i.lstrip('^').partition(':')[0])
    return seen


def tower0_placeholders(nodes):
    """Map the placeholders the tower-0 forward sub-graph reads to the arguments of
    models.py::predict, by creation order (/root/reference/train.py:181-216: features, then one
    [None,3] float per graph level, then one [None,None] int32 per edge level, then one [None,1]
    int32 per keypoint level)."""
    reach = _closure(nodes, [LOGITS_NODE, BOXES_NODE])
    phs = sorted((n for n in reach if nodes[n].op == 'Placeholder'),
                 key=lambda n: int(n.partition('_')[2] or 0))
    feats, coords, edges, keypoints = [], [], [], []
    for n in phs:
        dtype = _attr_value(nodes[n].attr['dtype'])[1]
        shape = _attr_value(nodes[n].attr['shape'])[1]
        if dtype == 1 and shape[1] == 3 and len(shape) == 2:
            coords.append(n)
        elif dtype == 1:
            feats.append(n)
        elif dtype == 3 and shape[1] == -1:
            edges.append(n)
        elif dtype == 3:
            keypoints.append(n)
    assert len(feats) == 1, feats
    return feats[0], coords, edges, keypoints


def run_forward(meta_path, variables, features, vertex_coord_list, keypoint_indices_list, edges_list,
                extra_nodes=()):
    """Execute the saved graph of ``meta_path`` on one frame.  -> dict with 'logits', 'boxes', 'probs'
    (+ every name in extra_nodes), and 'ops' = op-type histogram of what was executed."""
    nodes = load_meta_graph(meta_path)
    f, coords, edges, keypoints = tower0_placeholders(nodes)
    feeds = {f: np.asarray(features, np.float32)}
    # the sub-graph may read fewer levels than the lists hold (placeholders created in list order)
    all_ph = sorted((n for n in nodes if nodes[n].op == 'Placeholder'), key=lambda n: int(n.partition('_')[2] or 0))
    first = all_ph.index(f)
    num_levels = len(vertex_coord_list)
    coord_ph = all_ph[first + 1:first + 1 + num_levels]
    edge_ph = all_ph[first + 1 + num_levels:first + 1 + num_levels + len(edges_list)]
    kp_ph = all_ph[first + 1 + num_levels + len(edges_list):first + 1 + num_levels + 2 * len(edges_list)]
    assert set(coords) <= set(coord_ph) and set(edges) <= set(edge_ph) and set(keypoints) <= set(kp_ph), \
        'placeholder layout differs from train.py:181-216'
    for n, v in zip(coord_ph, vertex_coord_list):
        feeds[n] = np.asarray(v, np.float32)
    for n, v in zip(edge_ph, edges_list):
        feeds[n] = np.asarray(v, np.int32)
    for n, v in zip(kp_ph, keypoint_indices_list):
        feeds[n] = np.asarray(v, np.int32).reshape(-1, 1)
    interp = GraphInterpreter(nodes, variables, feeds)
    out = {'logits': interp.value(LOGITS_NODE), 'boxes': interp.value(BOXES_NODE),
           'probs': interp.value(PROBS_NODE)}
    for n in extra_nodes:
        out[n] = interp.value(n)
    out['ops'] = dict(interp.ops_used)
    return out
