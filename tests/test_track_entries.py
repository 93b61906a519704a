"""The one place that maps a track tensor's dtype (and, for search, the gallery's row type) to a C entry point:
every combination names an entry the header declares and the library exports (no GPU needed)."""
import types

import pytest
import torch

import seam_match_rcnn_b200 as pkg


@pytest.mark.parametrize("dtype,suffix", [(torch.float32, ""), (torch.float16, "_f16"), (torch.bfloat16, "_bf16")])
def test_track_dtype_selects_the_entry_point(dtype, suffix):
    lib = pkg.load_library()
    declared = set(pkg.declared_symbols())
    eng = types.SimpleNamespace(_lib=lib, _TRACK_SUFFIX=pkg.SeamEngine._TRACK_SUFFIX)
    seq = torch.empty((2, 1, 256), dtype=dtype)
    cases = [("aggregate", False, f"seam_aggregate{suffix}"),
             ("sharded_aggregate", False, f"seam_sharded_aggregate{suffix}"),
             ("search", False, f"seam_search{suffix}"),
             ("search", True, f"seam_search{suffix}_g16")]
    for op, rows_f16, name in cases:
        fn = pkg.SeamEngine._track_entry(eng, op, seq, rows_f16)
        assert fn.__name__ == name and name in declared
        assert fn.argtypes is not None and fn.argtypes == getattr(lib, f"seam_{op}{'_g16' if rows_f16 else ''}").argtypes


def test_other_track_dtypes_have_no_entry_point():
    eng = types.SimpleNamespace(_lib=pkg.load_library(), _TRACK_SUFFIX=pkg.SeamEngine._TRACK_SUFFIX)
    with pytest.raises(KeyError):
        pkg.SeamEngine._track_entry(eng, "aggregate", torch.empty((2, 1, 256), dtype=torch.float64))
