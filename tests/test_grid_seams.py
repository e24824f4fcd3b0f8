"""CPU tier: every node count the kernels dispatch on, through the host lock-step build of the kernel
source (tests/emu), against the oracle (tests/grid_cases.py)."""
import pytest

from tests import grid_cases as gc
from tests.emu import emu


def backend(prob, params, aux, opts, want_curves):
    return emu.loglik_batch(prob, params, aux, opts, want_curves)


@pytest.fixture(scope="module")
def refs():
    """LSODA curves, each computed once for the module (the seam matrix and the mixed grids share them)."""
    return gc.References()


def test_every_node_count_and_seam_against_lsoda(refs):
    worst = gc.check_node_count_seams(backend, refs)
    for k in sorted(worst):
        print(k, f"{worst[k]:.2e}")


def test_reversed_profile_with_swapped_contacts():
    print(gc.check_reversal_with_swapped_contacts(backend))


def test_small_grids_inside_larger_kernels(refs):
    print(gc.check_mixed_grids(backend, refs))


def test_grids_the_library_refuses():
    assert gc.check_grid_refusals(backend)
