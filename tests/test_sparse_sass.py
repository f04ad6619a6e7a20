"""The sparse kernels as built (cuobjdump -sass of libmarlin_b200.so, no GPU needed): the three products round every
multiply and every add separately (DMUL + DADD, never DFMA), write no output with atomics, and spill nothing."""
import collections
import re
import shutil
import subprocess

import pytest

from marlin_b200 import _native as nat

PRODUCTS = ("spmm_dense_sparse_kernel", "spmm_sparse_scatter_kernelILb0", "spmm_sparse_scatter_kernelILb1")


@pytest.fixture(scope="module")
def sparse_kernels():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    nat.load()
    out = subprocess.run([exe, "-sass", str(nat.lib_path())], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                         timeout=600)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable: " + out.stderr[:200])
    res = {}
    for chunk in re.split(r"\n\s*Function : ", out.stdout)[1:]:
        name = chunk.split("\n", 1)[0].strip()
        if "sparse" in name or "tile_ptr_kernel" in name:
            res[name] = collections.Counter(m.group(1).split(".")[0] for m in
                                            re.finditer(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Za-z0-9_.]*)", chunk))
    return res


def test_products_use_separate_multiply_and_add(sparse_kernels):
    for needle in PRODUCTS:
        fam = {k: v for k, v in sparse_kernels.items() if needle in k}
        assert len(fam) == 1, (needle, list(sparse_kernels))
        ops = next(iter(fam.values()))
        assert ops["DMUL"] >= 1 and ops["DADD"] >= 1, (needle, ops)
        assert ops["DFMA"] == 0, needle


def test_sparse_kernels_have_no_atomics_and_no_spills(sparse_kernels):
    assert len(sparse_kernels) >= 5                  # 3 products, toDense, rand, tile pointers
    for name, ops in sparse_kernels.items():
        for op in ("ATOM", "ATOMG", "ATOMS", "RED", "REDG", "REDS"):
            assert ops[op] == 0, (name, op)
        assert ops["LDL"] == 0 and ops["STL"] == 0, name
