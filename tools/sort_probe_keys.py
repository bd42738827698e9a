"""Writes the input of tools/sort_probe.cu: the engine's hashes of the key ids of one bench.py tick (Zipf-1.0 over
10 M keys, tests/traces.py config2, 2^20 requests) as raw little-endian u64."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import throttlecrab_b200 as tc  # noqa: E402
import traces  # noqa: E402

if __name__ == "__main__":
    tick = traces.config2(n_keys=10_000_000, n_ticks=1, tick_size=1 << 20)
    tc.hash_key_ids(tick["key"]).astype("<u8").tofile(sys.argv[1])
