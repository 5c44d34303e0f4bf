"""The C-ABI library loads and exports every symbol include/hlynr.h, hlynr_post.h, hlynr_rollout.h and hlynr_policy.h declare
(no compute calls: CPU-safe)."""
import ctypes
import os
import re

from hlynr_intercept_b200 import _lib, abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "hlynr.h")).read() + open(os.path.join(ROOT, "include", "hlynr_post.h")).read() + \
        open(os.path.join(ROOT, "include", "hlynr_rollout.h")).read() + open(os.path.join(ROOT, "include", "hlynr_policy.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hlynr_[a-z_0-9]+)\s*\(", src)))


def test_header_symbols_listed_in_loader():
    assert _declared_symbols() == sorted(_lib.EXPORTS)


def test_library_loads_and_exports_everything():
    L = _lib.load()
    for name in _declared_symbols():
        assert hasattr(L, name), name
    assert L.hlynr_abi_version() == abi.ABI_VERSION
    assert L.hlynr_params_size() == ctypes.sizeof(abi.HlynrParams)
    assert L.hlynr_env_state_size() == ctypes.sizeof(abi.HlynrEnvState)


def test_info_fields_match_header():
    """abi.INFO_FIELDS lists the members of HlynrInfoSoA in the header's order, and abi.HlynrInfoSoA has exactly those."""
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "hlynr.h")).read(), flags=re.S)
    body = re.search(r"typedef struct HlynrInfoSoA \{(.*?)\} HlynrInfoSoA;", src, flags=re.S).group(1)
    header = re.findall(r"\*\s*(\w+)\s*;", body)
    assert header == [name for name, _, _ in abi.INFO_FIELDS]
    assert [name for name, _ in abi.HlynrInfoSoA._fields_] == header


def test_no_cpu_fallback_in_product():
    """The product package must not import, load or name the oracle."""
    pkg = os.path.join(ROOT, "hlynr_intercept_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "libhlynr_oracle" not in text, f
