"""INTEGRATION.md's reference-side adapter is a real C file (integration/mcall_b200_glue.c): it must type-check against the
reference's own call.h and the htslib API subset of oracle/ref_shim/htslib (htslib itself is not in this image)."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"


@pytest.mark.skipif(not os.path.exists(os.path.join(REF, "call.h")) or not shutil.which("gcc"),
                    reason="needs bcftools' own call.h (a copy of it would check the glue against itself, so the repository carries none) and gcc")
def test_glue_type_checks_against_the_reference_headers():
    cmd = ["gcc", "-std=gnu99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "oracle", "ref_shim"), "-I", REF,
           "-I", os.path.join(ROOT, "include"), "-include", os.path.join(ROOT, "tests", "glue_decls.h"),
           os.path.join(ROOT, "integration", "mcall_b200_glue.c")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
