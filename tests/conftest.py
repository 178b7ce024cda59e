import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle_built():
    from oracle import ref
    ref.build()
    return ref


@pytest.fixture(scope="session")
def ctx():
    import multipathnet_b200 as mpn
    c = mpn.Context(0)       # raises loudly if the .so or the GPU is missing: no fallback
    yield c
    c.close()


def rel_err(a, b):
    """normwise relative error max|a-b| / max|b| (SURVEY 7 hard-part 1: elementwise is meaningless near 0)"""
    import numpy as np
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


_LITERAL = {}


def literal_golden(key):
    """an array stored by tests/golden/make_golden.py from the reference's own nms.c (nms_literal_golden.npz)"""
    import numpy as np
    if not _LITERAL:
        _LITERAL.update(np.load(os.path.join(ROOT, "tests", "golden", "nms_literal_golden.npz")))
    return _LITERAL[key]


def literal_nms_rows(key, scored_boxes, thr):
    """the rows the reference's own nms.c keeps from `scored_boxes` at `thr`, in its emission order, as stored under `key`;
    fails when the seeded input is no longer the one the golden was made from"""
    import hashlib
    import numpy as np
    sb = np.ascontiguousarray(scored_boxes, np.float32).reshape(-1, 5)
    assert hashlib.sha1(sb.tobytes()).hexdigest() == str(literal_golden(key + "_sha1")), f"{key}: input differs from the golden's"
    assert np.float32(thr) == literal_golden(key + "_thr"), key
    return sb[literal_golden(key + "_keep")]


def record_parity(name, **values):
    """append one JSON line of measured parity figures to $MPN_PARITY_LOG (the GPU run scripts set it; the numbers end up
    under profiles/): the bars are asserted by the tests, the log keeps HOW FAR inside them a run was"""
    import json, os
    path = os.environ.get("MPN_PARITY_LOG")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps({"test": name, **{k: (float(v) if not isinstance(v, (list, tuple, str)) else v) for k, v in values.items()}}) + "\n")
