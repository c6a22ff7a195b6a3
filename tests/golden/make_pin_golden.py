#!/usr/bin/env python
"""Writes tests/golden/reference_pin/<test>.npz from the REFERENCE'S OWN CODE (oracle/_ref/libstomp_ref.so, see
oracle/ref/Makefile): every value tests/test_reference_pin.py takes from the reference, so that the comparison runs on
machines without the reference's sources.  Each test also runs against the live reference while it is recorded.
Run where the reference build exists:   python tests/golden/make_pin_golden.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_reference_pin as pin  # noqa: E402


def main():
    assert pin.LIVE, "needs the reference build (oracle/ref/Makefile)"
    os.makedirs(pin.RECORDINGS, exist_ok=True)
    for name in sorted(n for n in dir(pin) if n.startswith("test_")):
        pin._CURRENT[0], pin._RECORD = name, {}
        getattr(pin, name)()
        np.savez_compressed(pin._recording(), **pin._RECORD)
        print(name, os.path.getsize(pin._recording()), "bytes")
    pin._RECORD = None


if __name__ == "__main__":
    main()
