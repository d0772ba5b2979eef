"""K2's host-side decisions (string_grouper_b200/_device.py: plan_k2, pick_tile, row_chunks, chunk_capacity,
select_mode) at their boundaries; no device needed."""
import pytest

from string_grouper_b200 import _device as D


def plan(n_rows=10_000, n_right=10_000, n_cols=5_000, nnz_right=100_000, threshold=0.8, **kw):
    return D.plan_k2(n_rows, n_right, n_cols, nnz_right, threshold, **kw)


def test_fixed_point_accumulator_and_its_fallbacks():
    p = plan()
    assert (p.acc, p.margin, p.margin_pf) == ("u16", D.CAND_MARGIN, D.U16_MARGIN_PER_FEATURE)
    assert p.thr_c == pytest.approx(0.8 - D.CAND_MARGIN)
    assert plan(nonneg=False).acc == "f32"
    assert plan(scale=1.0 + 1e-6).acc == "u16"
    assert plan(scale=1.0 + 2e-6).acc == "f32"
    assert plan(threshold=0.0515 + D.CAND_MARGIN).acc == "u16"
    assert plan(threshold=0.0485 + D.CAND_MARGIN).acc == "f32"         # thr_c < 0.05
    f = plan(acc="f32")
    assert (f.acc, f.margin_pf, f.refine) == ("f32", 0.0, False)
    assert plan(scale=2.0).margin == pytest.approx(2 * D.CAND_MARGIN)
    assert plan(threshold=0.001).thr_c == 0.0
    with pytest.raises(ValueError):
        plan(acc="f16")
    with pytest.raises(ValueError):
        plan(kernel="cols")


def test_tile_width_by_size_and_bucket_limit():
    # 16-bit accumulator: 128 columns from 400 000 right rows on when at least 150 000 left rows use the directory
    assert plan(n_rows=150_000, n_right=400_000).tile_w == 128
    assert plan(n_rows=150_000, n_right=399_999).tile_w == 256
    assert plan(n_rows=149_999, n_right=400_000).tile_w == 256
    assert plan(n_rows=150_000, n_right=400_000, acc="f32").tile_w == 128
    assert plan(n_rows=100, n_right=100).tile_w == 128                  # no wider than the right matrix needs
    p = plan(tile_w=1024, warps=16)
    assert (p.tile_w, p.warps) == (1024, 16)
    assert D.pick_tile(10_000, 1000, None, 2) == (896, 8)                # multiple of 128 u16 columns (256 bytes)


@pytest.mark.parametrize("entries_per_tile,want", [(1_000, 256), (1_001, 512), (2_000, 512), (2_001, 1024),
                                                  (4_000, 1024), (4_001, 2048)])
def test_tile_width_doubles_below_max_buckets(monkeypatch, entries_per_tile, want):
    monkeypatch.setattr(D, "MAX_BUCKETS", 20_000)
    # 5 000 right rows: 20 tiles of 256, 10 of 512, 5 of 1024; one directory entry per (feature + 1, tile)
    assert plan(n_right=5_000, n_cols=entries_per_tile - 1).tile_w == want


def test_tile_width_widening_stops_at_32768(monkeypatch):
    monkeypatch.setattr(D, "MAX_BUCKETS", 1)
    assert plan(n_right=10**6).tile_w == 32768


@pytest.mark.parametrize("nnz_right,n_right", [(1, 10), (10**5, 10**4), (10**7, 663_000), (10**9, 10**6),
                                               (4 * 10**7, 2 * 10**6)])
def test_tiles_per_group(nnz_right, n_right):
    p = plan(n_rows=n_right, n_right=n_right, nnz_right=nnz_right)
    assert p.tiles_per_group >= 64 and p.tiles_per_group % 64 == 0
    n_tiles = -(-n_right // p.tile_w)
    assert p.tiles_per_group == max(64, int(D.GROUP_BYTES // max(4 * nnz_right / n_tiles, 1)) // 64 * 64)


def test_tiles_per_group_value():
    # 10^7 postings over 5 180 tiles of 128 columns: 7 722 bytes per tile, 1 629 tiles per 12 MB -> 1 600
    assert plan(n_rows=663_000, n_right=663_000, nnz_right=10**7).tiles_per_group == 1600


def test_pruning_levels():
    p = D.PRUNE_FRAC
    assert plan().levels == (p, 0.75 * p, 0.5 * p, 0.25 * p, 0.0)
    assert plan(prune=0.9).levels == (0.9,)                 # the caller's level is kept
    assert plan(prune=0.0).levels == (0.0,)
    assert plan(threshold=0.001).levels == (p,)             # thr_c == 0: nothing to prune against


def test_pruning_levels_without_default_pruning(monkeypatch):
    monkeypatch.setattr(D, "PRUNE_FRAC", 0.0)
    assert plan().levels == (0.0,)


def test_whole_range_launch_and_sample():
    assert plan(n_rows=500_000, n_right=1_000_000).whole_range
    assert not plan(n_rows=500_000, n_right=1_000_001).whole_range
    assert plan(n_rows=65_535).sample_stride is None
    assert plan(n_rows=65_536).sample_stride == 64
    assert plan(n_rows=1_000_000).sample_stride == 1_000_000 // 8192
    assert plan(n_rows=1_000, n_right=2_000).cand_limit == pytest.approx(D.MAX_CAND_DENSITY * 2e6)


def test_tile_formulation_needs_its_stage_to_fit():
    fits = (256, 100_000, 232_448)
    t = plan(kernel="tiles", tile_fit=fits)
    assert (t.kernel, t.tile_w, t.warps, t.tiles_per_group, t.refine) == ("tiles", 256, 8, 0, False)
    assert (t.margin, t.margin_pf) == (D.TILE_MARGIN, D.TILE_MARGIN_PER_FEATURE)
    assert plan(kernel="tiles", tile_fit=(256, 232_449, 232_448)).kernel == "row"
    assert plan(kernel="tiles", tile_fit=(256, 232_448, 232_448)).kernel == "tiles"
    assert plan(kernel="tiles").kernel == "row"                               # blobs not built
    assert plan(kernel="tiles", acc="f32", tile_fit=fits).kernel == "row"     # fixed-point products only
    assert plan(kernel="row", tile_fit=fits).kernel == "row"
    assert plan().kernel == D.K2_KERNEL == "row"


def test_refine(monkeypatch):
    assert plan().refine
    monkeypatch.setattr(D, "REFINE", False)
    assert not plan().refine


def test_row_chunks(monkeypatch):
    monkeypatch.setattr(D, "CAND_CHUNK", 1000)
    assert D.row_chunks(10_001, None) == (1, 10_001)
    assert D.row_chunks(10_001, 0) == (1, 10_001)
    assert D.row_chunks(10_001, 769) == (1, 10_001)          # int(1.3 * 769) = 999
    assert D.row_chunks(10_001, 770) == (2, 5_001)           # 1001
    assert D.row_chunks(10_001, 10_000) == (13, 770)


def test_chunk_capacity():
    assert D.chunk_capacity(1000, 1000, None) == 96 * 1000 + (1 << 22)
    assert D.chunk_capacity(2 * 10**7, 2 * 10**7, None) == 1 << 30
    assert D.chunk_capacity(1000, 250, 10**6) == int(1.3 * 10**6 * 250 / 1000) + (1 << 22)
    assert D.chunk_capacity(1000, 1000, 0) == 1 << 22
    assert D.chunk_capacity(1000, 1000, 10**10) == 1 << 31


def test_select_mode(monkeypatch):
    cap = 4096
    assert D.select_mode(32, 10**6, cap) == "rows"            # warp network
    assert D.select_mode(3000, cap, cap) == "rows"            # every row fits one CTA
    assert D.select_mode(2048, cap + 1, cap) == "rows"        # long rows ranked in pieces
    assert D.select_mode(2049, cap + 1, cap) == "sort"
    assert D.select_mode(33, 10**6, 64) == "sort"
    monkeypatch.setattr(D, "SELECT_MODE", "sort")
    assert D.select_mode(20, 10, cap) == "sort"
