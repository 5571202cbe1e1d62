"""The training-path kernels reduce in a fixed order (per-block partials summed in slot order): no atomics in their
sources, so the summation order never depends on block scheduling."""
import os
import re

import pytest

CSRC = os.path.join(os.path.dirname(__file__), "..", "image-super-resolution_b200", "csrc")


@pytest.mark.parametrize("name", ["train_ops.cu", "lka_depthwise.cu", "losses.cu", "optim.cu", "common.cuh"])
def test_no_atomics_in_training_kernels(name):
    code = re.sub(r"//[^\n]*", "", open(os.path.join(CSRC, name)).read())
    assert re.search(r"\batomic\w*\s*\(", code) is None, name
