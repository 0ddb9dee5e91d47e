"""Loads the golden vectors under tests/golden/: range_coder_golden.npz (oracle/make_golden.py) and
reference_outputs.npz (oracle/make_reference_outputs.py), both written from the compiled reference."""
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "range_coder_golden.npz")
REFERENCE_OUTPUTS_PATH = os.path.join(os.path.dirname(PATH), "reference_outputs.npz")


def load():
  return dict(np.load(PATH))


def load_reference_outputs():
  """The compiled reference's outputs on the seeded inputs of the tests that compare against it."""
  return dict(np.load(REFERENCE_OUTPUTS_PATH))


def split(flat, lens):
  out, at = [], 0
  for n in lens:
    out.append(bytes(flat[at:at + int(n)]))
    at += int(n)
  return out
