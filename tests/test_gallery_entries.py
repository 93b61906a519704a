"""Every (operation, track dtype, gallery row type) the engine can ask for resolves, through SeamEngine._track_entry, to
an entry point the header declares and the library exports; a bf16 gallery's _gbf16 entries are bound with exactly the
fp32 entries' argument types (no GPU needed)."""
import types

import pytest
import torch

import seam_match_rcnn_b200 as pkg
from seam_match_rcnn_b200.engine import ROW_SUFFIX

TRACKS = {torch.float32: "", torch.float16: "_f16", torch.bfloat16: "_bf16"}
# operations that read gallery rows, and whether they take tracks
GALLERY_OPS = {"search": True, "score_topk": False, "sharded_score_topk": False, "rank_of_target_prepared": False,
               "shard_target_margin": False, "shard_rank_count_prepared": False, "rank_fused_distances": False,
               "shard_fused_target": False, "shard_rank_fused_distances": False}


def _stub():
    return types.SimpleNamespace(_lib=pkg.load_library(), _TRACK_SUFFIX=pkg.SeamEngine._TRACK_SUFFIX)


def test_row_suffixes():
    assert ROW_SUFFIX == {torch.float32: "", torch.float16: "_g16", torch.bfloat16: "_gbf16"}


@pytest.mark.parametrize("op", sorted(GALLERY_OPS))
@pytest.mark.parametrize("rows", [torch.float32, torch.float16, torch.bfloat16])
def test_every_gallery_entry_is_declared_and_exported(op, rows):
    eng, declared = _stub(), set(pkg.declared_symbols())
    lib = eng._lib
    for tracks in (TRACKS if GALLERY_OPS[op] else [None]):
        seq = None if tracks is None else torch.empty((2, 1, 256), dtype=tracks)
        name = f"seam_{op}{'' if tracks is None else TRACKS[tracks]}{ROW_SUFFIX[rows]}"
        fn = pkg.SeamEngine._track_entry(eng, op, seq, ROW_SUFFIX[rows])
        assert fn.__name__ == name and name in declared and hasattr(lib, name)
        assert fn.argtypes is not None and fn.restype is not None
        fp32_twin = getattr(lib, f"seam_{op}{'' if tracks is None else TRACKS[tracks]}")
        if rows == torch.bfloat16:
            # the same parameter list as the fp32 entry, rows typed void*
            assert fn.argtypes == fp32_twin.argtypes
        if rows == torch.float32:
            assert fn is fp32_twin
        if rows == torch.float16 and op == "search":
            # a bool still says "fp16 rows", as it did before galleries had three row types
            assert pkg.SeamEngine._track_entry(eng, op, seq, True).__name__ == name


def test_bf16_preparation_takes_the_fp32_parameters():
    lib = pkg.load_library()
    assert "seam_prepare_gallery_bf16" in pkg.declared_symbols()
    assert lib.seam_prepare_gallery_bf16.argtypes == lib.seam_prepare_gallery.argtypes


def test_a_bool_row_argument_reads_as_before():
    eng = _stub()
    seq = torch.empty((2, 1, 256), dtype=torch.bfloat16)
    assert pkg.SeamEngine._track_entry(eng, "search", seq, False).__name__ == "seam_search_bf16"
    assert pkg.SeamEngine._track_entry(eng, "search", seq, True).__name__ == "seam_search_bf16_g16"
    assert pkg.SeamEngine._track_entry(eng, "search", seq).__name__ == "seam_search_bf16"
    with pytest.raises(AttributeError):
        pkg.SeamEngine._track_entry(eng, "aggregate", seq, "_gbf16")      # no gallery behind an aggregation


def test_prepared_gallery_row_type():
    def gal(dtype):
        g = torch.zeros((3, 256), dtype=dtype)
        return pkg.PreparedGallery(g=g, g16=g if dtype == torch.float16 else g.half(), cg=torch.zeros(3),
                                   gstat=torch.zeros(4))
    for dtype, f16, bf16 in ((torch.float32, False, False), (torch.float16, True, False),
                             (torch.bfloat16, False, True)):
        p = gal(dtype)
        assert (p.rows_f16, p.rows_bf16, p.row_suffix) == (f16, bf16, ROW_SUFFIX[dtype]) and p.G == 3
