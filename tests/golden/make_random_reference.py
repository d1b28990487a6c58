#!/usr/bin/env python3
"""Writes tests/golden/random_reference.npz: the reference's results on the five seeded adversarial batches of
tests/test_host_logic.py (random_reference_cases), with a digest of each batch's inputs, so that the port is compared with
the reference on them in every checkout, with or without oracle/_ref.

    python tests/golden/make_random_reference.py              results of the compiled reference (needs oracle/_ref built)
    python tests/golden/make_random_reference.py port         results of the plain-C port

The committed file was written with `port`.  On exactly these inputs the port equals the compiled reference in every field
parity.compare checks (QUAL bit for bit, no near-ties): test_restatement_equals_compiled_reference_on_random_inputs
asserted that with oracle/_ref built, at commit 321e77c, and the port (oracle/mcall_oracle.c), the batch generator
(tests/parity.py) and the batches have not changed since.  Re-run with the reference where it is built.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle import pyoracle  # noqa: E402
from tests import test_host_logic as T  # noqa: E402

kind = sys.argv[1] if len(sys.argv) > 1 else "reference"
pyoracle.build(want_ref=kind == "reference")
if kind == "reference" and not pyoracle.have_ref():
    raise SystemExit("oracle/_ref is not built: run `make -C oracle ref REF=<bcftools source tree>` first")
out = {}
for k, (params, b, tab, want_gp) in enumerate(T.random_reference_cases()):
    res, _ = pyoracle.call(kind, params, b, tab, want_gp=want_gp)
    out[f"{k}_inputs"] = np.array(T.inputs_digest(params, b, tab))
    for name in T.RANDOM_REFERENCE_FIELDS:
        if getattr(res, name) is not None:
            out[f"{k}_{name}"] = getattr(res, name)
np.savez_compressed(T.RANDOM_REFERENCE, **out)
print(T.RANDOM_REFERENCE, os.path.getsize(T.RANDOM_REFERENCE), "bytes,", kind)
