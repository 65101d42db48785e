"""Which tiling designs the fused step serves (`tiling_fused.serves`: 2..1024 alleles per guide, no --scale-by-acc) and which of
them shard over ranks (`supports`, `run.shards_over_ranks`: at most 32 alleles): host logic, no GPU."""
from functools import partial

import pytest

from crispr_bean_b200 import model as sm
from crispr_bean_b200.data_class import TilingSortingReporterScreenData
from crispr_bean_b200.run import shards_over_ranks
from crispr_bean_b200.synth import make_tiling_screen
from crispr_bean_b200.tiling_fused import WIDE_MAX_DRAWS, faster_than_site_kernels, serves, supports


@pytest.fixture(scope="module")
def data():
    scr = make_tiling_screen(n_guides=12, max_alleles=5, n_reps=2, seed=1)
    return TilingSortingReporterScreenData(scr, control_can_be_selected=True, allele_df_key="allele_counts")


@pytest.mark.parametrize("width,served,sharded", [(2, True, True), (32, True, True), (33, True, False), (1024, True, False),
                                                  (1025, False, False), (1, False, False)])
def test_served_and_sharded_widths(data, width, served, sharded):
    data.n_max_alleles = width
    acc = partial(sm.MultiMixtureNormalModel, scale_by_accessibility=True)
    assert serves(data) == served
    assert supports(data) == sharded
    assert shards_over_ranks(sm.MultiMixtureNormalModel, data) == sharded
    # --scale-by-acc: never the fused step, never sharded
    assert not serves(data, scale_by_accessibility=True)
    assert not supports(data, scale_by_accessibility=True)
    assert not shards_over_ranks(acc, data)


def test_wide_designs_go_to_the_fused_step_only_below_the_measured_crossover(data):
    G, R = data.n_guides, data.n_reps
    data.n_max_alleles = 32
    data.n_guides = 10 ** 6  # one lane per allele: always the fused step
    assert faster_than_site_kernels(data)
    data.n_guides = G
    for A in (33, 231, 1024):
        data.n_max_alleles = A
        assert faster_than_site_kernels(data) == (G * R * A <= WIDE_MAX_DRAWS)
    data.n_max_alleles = 231
    data.n_guides = WIDE_MAX_DRAWS // (R * 231)
    assert faster_than_site_kernels(data)
    data.n_guides += 1
    assert not faster_than_site_kernels(data)
    data.n_guides = G
