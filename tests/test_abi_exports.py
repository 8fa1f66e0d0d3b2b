"""The C-ABI library builds, loads and exports every symbol include/b200lev.h declares
(no compute calls: this box has no GPU)."""
import ctypes
import os
import re

from conftest import ROOT


def _declared():
    text = open(os.path.join(ROOT, "include", "b200lev.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200lev_[a-z0-9_]+)\s*\(", text)))


def test_abi_v3_header_symbols_are_exported_and_bound():
    """ABI version 3 (the class weight of the OCD loss in the accumulation type, and its
    out-of-range target flag): every symbol the header declares is exported and bound, and the
    entry points version 2 retired are no longer exported."""
    import __graft_entry__ as entry
    from b200lev import _abi

    entry.build()
    names = _declared()
    assert len(names) >= 15
    lib = ctypes.CDLL(_abi.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in b200lev.h but not exported"
        assert n in _abi.SIGNATURES, f"{n} has no ctypes signature in _abi.py"
    assert set(_abi.SIGNATURES) == set(names)
    assert _abi.lib().b200lev_abi_version() == 3
    for n in ("b200lev_pack", "b200lev_final_packed", "b200lev_prefix_packed",
              "b200lev_workspace_ref_lens", "b200lev_workspace_hyp_lens", "b200lev_err_sum"):
        assert not hasattr(lib, n), f"{n} is still exported"


def test_product_refuses_cpu_tensors():
    """No CPU fallback: without CUDA tensors the
    product raises instead of computing."""
    import pytest
    import torch

    import b200lev.functional as F
    from b200lev import _abi

    if torch.cuda.is_available():
        pytest.skip("GPU present: host tensors are offloaded to it")
    with pytest.raises(_abi.B200LevError, match="no CPU fallback"):
        F.error_rate(torch.zeros(2, 2, dtype=torch.long), torch.zeros(2, 2, dtype=torch.long))
