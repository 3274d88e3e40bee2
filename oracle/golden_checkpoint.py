"""The shipped TensorFlow checkpoints, rebuilt byte for byte from tests/golden/.

TEST INFRASTRUCTURE.  A checkpoint's ``.data`` file is the concatenation of its tensors; every tensor but the global
step is in ``weights_<cfg>.npz``.  tests/golden/checkpoints/<cfg>/ keeps the ``checkpoint`` state file and the
``.index`` table verbatim, ``data.json`` (name, offset and size of each tensor in the ``.data`` file, the bytes of the
tensors not in the weights file, the sha256 of the original file) and, for some checkpoints, the forward sub-graph of
the ``.meta`` graph (gzipped).  ``rebuild`` writes a checkpoint directory that ``utils/tf_checkpoint.py`` and
``oracle/graphdef.py`` read as they would the original (tools/make_golden.py checkpoints writes the fixtures).
"""
import gzip
import hashlib
import json
import os
import shutil

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')


def names():
    return sorted(os.listdir(os.path.join(GOLDEN, 'checkpoints')))


def rebuild(name, dest):
    """Write checkpoint <name> into directory ``dest``; raise unless the ``.data`` file equals the original."""
    src = os.path.join(GOLDEN, 'checkpoints', name)
    os.makedirs(dest, exist_ok=True)
    with open(os.path.join(src, 'data.json')) as f:
        layout = json.load(f)
    weights = np.load(os.path.join(GOLDEN, 'weights_%s.npz' % name))
    blob = bytearray(layout['size'])
    for key, offset, size in layout['tensors']:
        raw = bytes.fromhex(layout['extra_hex'][key]) if key in layout['extra_hex'] else \
            np.ascontiguousarray(weights[key], dtype='<f4').tobytes()
        if len(raw) != size:
            raise ValueError('%s: %d bytes, the checkpoint holds %d' % (key, len(raw), size))
        blob[offset:offset + size] = raw
    if hashlib.sha256(blob).hexdigest() != layout['sha256']:
        raise ValueError('%s: the rebuilt .data file differs from the original' % name)
    with open(os.path.join(dest, layout['data_file']), 'wb') as f:
        f.write(blob)
    for fname in os.listdir(src):
        if fname == 'data.json':
            continue
        if fname.endswith('.gz'):
            with gzip.open(os.path.join(src, fname), 'rb') as fi, open(os.path.join(dest, fname[:-3]), 'wb') as fo:
                shutil.copyfileobj(fi, fo)
        else:
            shutil.copyfile(os.path.join(src, fname), os.path.join(dest, fname))
    return dest
