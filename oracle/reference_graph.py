"""Run the reference's OWN models/graph_gen.py (where the reference tree is present).

TEST INFRASTRUCTURE, used only by tools/make_golden.py to generate fixtures: the
tests read what it computed from tests/golden/.  graph_gen.py imports
``open3d`` and ``tensorflow`` at module top (graph_gen.py:8-9) but uses neither
in the radius-graph builder; empty stub modules make the import succeed.
"""
import importlib.util
import os
import sys
import types

REFERENCE_ROOT = '/root/reference'


def load():
    for name in ('open3d', 'tensorflow'):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    spec = importlib.util.spec_from_file_location(
        '_reference_graph_gen', os.path.join(REFERENCE_ROOT, 'models', 'graph_gen.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod
