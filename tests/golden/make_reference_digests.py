"""Writes tests/golden/reference_digests.json: SHA-256 digests of what the reference's CPU path computes on the inputs of
the tests that compare with it (test_oracle.py, test_math.py, test_gpu_parity.py), so that those tests need no build of
the reference. The inputs come from the test modules themselves; their own digests are stored too, so a changed input
fails the test instead of comparing against a stale digest.

Source: the unmodified reference (oracle/_ref, built by oracle/build_ref.sh from the reference's sources) where it has
been built, else the oracle in strict mode -- the C restatement that these tests had checked bit-exact against that
build on exactly these inputs, including the reference's lost-RSTn aborts. The file records which one wrote it.
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np

import test_gpu_parity
import test_math
import test_oracle
from oracle import GATE_EXTENDED, GATE_REFERENCE, Oracle, Reference, reference_available


def sha(a):
    return hashlib.sha256(a if isinstance(a, bytes) else a.tobytes()).hexdigest()


class Source:
    def __init__(self):
        if reference_available():
            self.kind = "reference build (oracle/_ref)"
            self.ref = Reference()
        else:
            self.kind = "oracle, strict mode (oracle/oracle.c)"
            self.ref = None
        self.orc = Oracle()
        self.orc.set_strict(True)

    def decode(self, data, skip_gate, want_pixels=True):
        """(ok, coef, bgra) as the reference decodes the file."""
        if self.ref is not None:
            ok, _, coef, bgra, _ = self.ref.decode(data, skip_gate=skip_gate, want_pixels=want_pixels)
            return ok, coef, bgra
        rc, _, coef, bgra = self.orc.decode(data, gate=GATE_EXTENDED if skip_gate else GATE_REFERENCE, want_pixels=want_pixels)
        return rc == 0, coef, bgra

    def idct(self, block):
        return self.ref.fast_idct(block) if self.ref is not None else self.orc.idct(block)

    def yuv_to_rgb32(self, y, u, v):
        return self.ref.yuv_to_rgb32(y, u, v) if self.ref is not None else self.orc.yuv_to_rgb32(y, u, v)


def entry(src, data, skip_gate, want_pixels=True):
    ok, coef, bgra = src.decode(data, skip_gate, want_pixels)
    e = {"file_sha256": sha(data), "ok": bool(ok)}
    if ok:
        e["coef_sha256"] = sha(coef)
        if want_pixels:
            e["pixel_sha256"] = sha(bgra)
    return e


def main():
    src = Source()
    out = {"source": src.kind}
    out["oracle_cases"] = {test_oracle.case_key(c): entry(src, test_oracle.case_jpeg(c), c[2] == "422") for c in test_oracle.CASES}
    out["rst_defect"] = [entry(src, f, False, want_pixels=False) for f in test_oracle.rst_defect_jpegs()]
    out["crafted"] = [entry(src, s[0], True, want_pixels=False) for s in test_oracle.crafted_streams()]
    out["generic_luma"] = {test_oracle.generic_luma_key(s, ri): entry(src, test_oracle.generic_luma_jpeg(s, ri), True)
                           for s in test_oracle.GENERIC_LAYOUTS for ri in (0, 2)}
    out["idct"] = [{"block_sha256": sha(b), "idct_sha256": sha(np.ascontiguousarray(src.idct(b), np.int32))} for b in test_math.idct_blocks()]
    out["colour_spot_sha256"] = sha(np.array([src.yuv_to_rgb32(*t) for t in test_math.colour_triples()], np.uint32))
    specs = test_gpu_parity.SPECS[:12]
    out["gpu_batch"] = [entry(src, f, s[2] == "422") for s, f in zip(specs, test_gpu_parity.reference_build_jpegs())]
    with open(os.path.join(HERE, "reference_digests.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote tests/golden/reference_digests.json from the %s" % src.kind)


if __name__ == "__main__":
    main()
