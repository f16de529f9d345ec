import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (select with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


# ---- parity ledger: every GPU parity test records its numbers; written once per session -------------------------
_PARITY = {}


def record_parity(case, **numbers):
    """case -> {e16, e32, floor, argmax_agree, ...}; merged into $B200_PARITY_DIR/PARITY_r02.json when that variable names
    a directory (the test run itself writes nothing into the repository)."""
    _PARITY[case] = {k: (float(v) if hasattr(v, "__float__") else v) for k, v in numbers.items()}


def pytest_sessionfinish(session, exitstatus):
    out_dir = os.environ.get("B200_PARITY_DIR")
    if not _PARITY or not out_dir:
        return
    import json
    out = {"rule": "pass iff |eng-ref16|max <= 1e-3 OR |eng-ref32|max <= RULE_FACTOR * |ref16-ref32|max; "
                   "ref16/ref32 = the unmodified reference (goldens / oracle/_ref) or its bit-pinned port in fp16 / fp32",
           "cases": _PARITY}
    try:
        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, "PARITY_r02.json")
        old = {}
        if os.path.isfile(path):
            try:
                old = json.load(open(path)).get("cases", {})
            except Exception:
                old = {}
        old.update(_PARITY)
        out["cases"] = old
        with open(path, "w") as f:
            json.dump(out, f, indent=1, sort_keys=True)
    except OSError:
        pass
