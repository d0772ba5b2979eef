"""not-gpu: the C-ABI library loads and exports every symbol include/sg_b200.h declares (no compute calls)."""
import os
import re
import subprocess
import sys
import textwrap

from string_grouper_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "sg_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sg_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(lib, name), "libsg_b200.so does not export %s" % name
    assert sorted(_lib.SIGNATURES) == declared, set(_lib.SIGNATURES) ^ set(declared)


def test_pure_host_entry_points():
    lib = _lib.load()
    assert lib.sg_abi_version() == 3
    assert lib.sg_num_tiles(10_000, 3072) == 4 and lib.sg_num_tiles(0, 128) == 1
    assert lib.sg_tfidf_table_slots(3) == 2 ** 21 and lib.sg_tfidf_table_slots(5) == -1


def test_no_product_module_imports_the_oracle():
    pkg = os.path.join(ROOT, "string_grouper_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in re.sub(r'""".*?"""', "", src, flags=re.S).replace("# oracle", ""), fn


MISSING_DEVICE = textwrap.dedent('''
    import sys
    sys.path.insert(0, %r)
    import pandas as pd
    import torch
    assert not torch.cuda.is_available()
    import string_grouper_b200 as api
    from string_grouper_b200 import _lib
    try:
        api.match_strings(pd.Series(["foo inc", "foo inc."]))
    except _lib.SgB200Error:
        sys.exit(0)
    sys.exit("no SgB200Error without a CUDA device")
''')


def test_missing_device_fails_loudly():
    # a child process that sees no device, so that the check also runs on a machine with GPUs
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", MISSING_DEVICE % ROOT], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
