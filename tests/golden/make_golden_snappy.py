#!/usr/bin/env python
"""Snappy streams written by the Snappy library itself (pyarrow's codec) for the inputs of
tests/test_checkpoint.py::snappy_cases; writes tests/golden/golden_snappy.npz, one uint8 array
per case. The test decodes them with the checkpoint reader's own decoder.
Re-run: python tests/golden/make_golden_snappy.py
"""
import os
import sys

import numpy as np
import pyarrow as pa

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests.test_checkpoint import snappy_cases  # noqa: E402


def main():
    codec = pa.Codec('snappy')
    out = {'case_%d' % i: np.frombuffer(codec.compress(raw, asbytes=True), np.uint8)
           for i, raw in enumerate(snappy_cases())}
    np.savez_compressed(os.path.join(HERE, 'golden_snappy.npz'), **out)
    print({k: len(v) for k, v in out.items()})


if __name__ == '__main__':
    main()
