#!/usr/bin/env python
"""Writes the fixtures of tests/test_gpu_small_packed_exact.py (tests/golden/small_packed_<scene>.npz) with the build
of the library that PYTRACER_B200_LIB names, or the in-tree one.  Needs a GPU.

    PYTRACER_B200_LIB=/path/to/libpytracer_b200.so python tests/golden/make_golden_small_packed.py

The committed files were rendered on a B200 by the build of the parent commit of the change that moved the SMALL
kernel's transform and plane arithmetic onto the paired FP32 pipe."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]

import test_gpu_small_packed_exact as t  # noqa: E402


def main():
    for name in t.SCENES:
        arrays = {}
        for setting in t.SETTINGS:
            for key, value in t.render(name, setting).items():
                arrays[f"{setting}_{key}"] = value
        np.savez_compressed(t.fixture_path(name), **arrays)
        print(f"{t.fixture_path(name)}: {os.path.getsize(t.fixture_path(name))} bytes, rays "
              f"{ {s: int(arrays[s + '_rays_closest'][0]) for s in t.SETTINGS} }")


if __name__ == "__main__":
    main()
