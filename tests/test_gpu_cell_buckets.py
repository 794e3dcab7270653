"""The cell search of the batched submits (assoc_cells_body: one thread per query, cell by cell over
the cell-ordered voxel buckets of map_assoc.cu pass 4) on single contexts, through
FORMGPU_SINGLE_CELL_SEARCH=1, so that it goes through every stage-2 oracle check of the
single-context sequences: neighbour ids, squared-distance bits, pair counts, novel sets."""
import pytest

import test_gpu_stages

pytestmark = pytest.mark.gpu


@pytest.fixture
def cell_search(monkeypatch):
    monkeypatch.setenv("FORMGPU_SINGLE_CELL_SEARCH", "1")


def test_cell_search_os1_64_sequence(cell_search):
    test_gpu_stages._run_sequence("os1-64", 8, remove_at={4: [1], 6: [0, 3]})


def test_cell_search_vlp16_sparse(cell_search):
    test_gpu_stages._run_sequence("vlp-16", 10, seq=2, remove_at={5: [2]})


def test_cell_search_os0_128(cell_search):
    test_gpu_stages._run_sequence("os0-128", 4, seq=1)


def test_cell_search_small_matching_distance(cell_search):
    test_gpu_stages._run_sequence("vlp-16", 5, overrides=dict(max_dist_matching=0.3, min_dist_map=0.05))


def test_cell_search_full_window_and_million_voxel_map(cell_search):
    import test_gpu_configs

    test_gpu_stages._run_sequence("os1-64", 64, seq=3, icp_iters=1, max_window=61, min_final_pairs=1000)
    test_gpu_configs.test_config4_stress_scans_against_million_voxel_map()
