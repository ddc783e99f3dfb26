"""Writes tests/golden/ldm_golden.json: size + SHA-256 of what OUR encoder emits in prefix mode with long-distance matching (every tier at
window log ilog2(len(OLD)) + 1, and level 3 at window log 17) for the rotated-and-edited pair of tests/test_patch_ldm.py (ldm_golden_cases),
from the CPU emulation build of the sources (tests/emul), whose output does not depend on the warp-scheduling seed (ZK_EMUL_SEED).  The GPU
suite asserts that the nvcc build reproduces these bytes (tests/test_patch_ldm.py test_gpu_ldm_golden).
Re-run after any intended change of the encoder's output:   python tests/golden/make_ldm_golden.py"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE))); sys.path.insert(0, os.path.dirname(HERE))
from zeekstd_b200 import _native
from zeekstd_b200.build import build_emul
from util import make_ctx
import test_patch_ldm

out = test_patch_ldm.ldm_golden(make_ctx(_native.load(build_emul())))
json.dump(out, open(os.path.join(HERE, "ldm_golden.json"), "w"), indent=1)
print(json.dumps(out, indent=1))
