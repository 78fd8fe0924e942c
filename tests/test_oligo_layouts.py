"""The read-2 layouts of the GPU tests and tools (tests/oligo_layouts.py) are those the reference's oligo fixtures were
recorded with (oracle/make_golden_collapse_oligos.py), and relayout_array applies them as the per-read functions do."""
import ast
import os
import random

import numpy as np

import oligo_layouts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _layouts_node(path):
    with open(path) as fh:
        tree = ast.parse(fh.read())
    for node in tree.body:
        if isinstance(node, ast.Assign) and any(isinstance(t, ast.Name) and t.id == "LAYOUTS" for t in node.targets):
            return ast.dump(node.value)
    raise AssertionError("no LAYOUTS in " + path)


def test_layouts_are_those_the_fixtures_were_recorded_with():
    recorder = os.path.join(ROOT, "oracle", "make_golden_collapse_oligos.py")
    assert _layouts_node(oligo_layouts.__file__) == _layouts_node(recorder)


def test_relayout_array_equals_the_layout_functions():
    rng = random.Random(5)
    for width in (62, 250):
        reads = ["".join(rng.choice("ACGTN") for _ in range(width)) for _ in range(40)]
        arr = np.frombuffer("".join(reads).encode(), dtype=np.uint8).reshape(len(reads), width)
        for oligo, (layout, _) in oligo_layouts.LAYOUTS.items():
            got = oligo_layouts.relayout_array(arr, oligo)
            assert [bytes(r).decode() for r in got] == [layout(x)[:width] for x in reads], (oligo, width)
