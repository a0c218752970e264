"""Records tests/golden/ring_buffer_log.json: a seeded sequence of RingBuffer operations
(write / read / read_all / seek / rewind / reset / fill, over- and underflow included) and
what each one observed, for test_host.py::test_ring_buffer_matches_reference_semantics.

    python tests/golden/make_golden_ring_buffer.py [REFERENCE_CHECKOUT]

With a checkout of the reference project the log is that of its own
spokestack/ring_buffer.py; without one it is that of wakeword_detection_b200.ring_buffer
(the file records which).
"""
import importlib.util
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from test_host import _drive  # noqa: E402


def ring_ops():
    rng = np.random.default_rng(0)
    ops = [("fill", 0.0)]
    for _ in range(400):
        k = rng.integers(0, 10)
        ops.append([("write", float(rng.random())), ("write", float(rng.random())), ("read", None),
                    ("read_all", None), ("seek", int(rng.integers(0, 3))), ("rewind", None), ("reset", None),
                    ("write", float(rng.random())), ("write", float(rng.random())), ("fill", float(k))][k])
    return ops


def main():
    if len(sys.argv) > 1:
        path = os.path.join(sys.argv[1], "spokestack", "ring_buffer.py")
        spec = importlib.util.spec_from_file_location("ref_ring_buffer", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        cls, source = mod.RingBuffer, "spokestack/ring_buffer.py of the reference"
    else:
        from wakeword_detection_b200.ring_buffer import RingBuffer as cls
        source = "wakeword_detection_b200/ring_buffer.py"
    ops = ring_ops()
    log = []
    _drive(cls(shape=[5]), ops, log)
    log = [[e[0], [float(v) for v in e[1].reshape(-1)]] if isinstance(e[1], np.ndarray) else
           [e[0]] + [x if isinstance(x, str) else bool(x) for x in e[1:]] for e in log]
    out = {"source": source, "capacity": 5, "ops": [list(o) for o in ops], "log": log}
    with open(os.path.join(HERE, "ring_buffer_log.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print("%d ops, %d log entries from %s" % (len(ops), len(log), source))


if __name__ == "__main__":
    main()
