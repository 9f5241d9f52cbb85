"""The ctypes mirrors of spcu_guide and spcu_denoise_params have the C layout (no GPU needed)."""
import ctypes
import shutil
import subprocess
import tempfile

import pytest

from conftest import ROOT
from simplepath_b200 import capi


def test_guide_dtype_matches_ctypes():
    assert ctypes.sizeof(capi.Guide) == capi.GUIDE_DTYPE.itemsize == 32
    for name in ("normal", "depth", "albedo", "id"):
        assert getattr(capi.Guide, name).offset == capi.GUIDE_DTYPE.fields[name][1]
    assert ctypes.sizeof(capi.DenoiseParams) == 16


@pytest.mark.skipif(shutil.which("cc") is None, reason="no C compiler")
def test_mirrors_match_header():
    probe = r'''
    #include "spcu.h"
    #include <stddef.h>
    #include <stdio.h>
    int main(void){ printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(spcu_guide), offsetof(spcu_guide, normal),
        offsetof(spcu_guide, depth), offsetof(spcu_guide, albedo), offsetof(spcu_guide, id), sizeof(spcu_denoise_params),
        offsetof(spcu_denoise_params, iterations), offsetof(spcu_denoise_params, sigma_l), offsetof(spcu_denoise_params, sigma_z),
        offsetof(spcu_denoise_params, sigma_a)); return 0; }
    '''
    with tempfile.TemporaryDirectory() as d:
        src, exe = f"{d}/p.c", f"{d}/p"
        open(src, "w").write(probe)
        subprocess.run(["cc", "-I", str(ROOT / "include"), src, "-o", exe], check=True)
        got = [int(x) for x in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    G, P = capi.Guide, capi.DenoiseParams
    want = [ctypes.sizeof(G), G.normal.offset, G.depth.offset, G.albedo.offset, G.id.offset, ctypes.sizeof(P),
            P.iterations.offset, P.sigma_l.offset, P.sigma_z.offset, P.sigma_a.offset]
    assert got == want
