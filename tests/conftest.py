import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_cuda = torch.cuda.is_available()
    except Exception:
        has_cuda = False
    if has_cuda:
        return
    skip = pytest.mark.skip(reason='no CUDA device')
    for item in items:
        if 'gpu' in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope='session')
def golden():
    import numpy as np
    return np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_ops_golden.npz'))


@pytest.fixture(scope='session')
def host_gold():
    """What the original project's host code returned on the tests' inputs (tests/golden/make_reference_golden.py)."""
    import json
    with open(os.path.join(ROOT, 'tests', 'golden', 'ref_host.json')) as f:
        return json.load(f)


@pytest.fixture(scope='session')
def host_arrays():
    import numpy as np
    return np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_host.npz'))


@pytest.fixture
def host_instance_ops(monkeypatch):
    """CPU tests of get_instances: the GPU bitmap ops (softgroup_b200.ops.instances) are replaced by the dense
    reference steps of oracle/ops_cpu.py (test infrastructure), like the ball query / clustering stand-ins."""
    from oracle import ops_cpu
    from softgroup_b200.ops import instances as inst_ops
    for name in ('instance_point_counts', 'instance_bitmaps', 'bitmaps_to_rle'):
        monkeypatch.setattr(inst_ops, name, getattr(ops_cpu, name))
    return inst_ops
