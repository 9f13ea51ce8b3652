"""The component layer on the real kernels, against the reference's own pipeline.

tests/golden/dropin_*.npz were written in the build container by running the reference's own
registry / builders / `Pipeline` / components (tests/golden/make_dropin_golden.py): the dataset
entering the first hot-path component (`in__*`) and the one leaving the last (`out__*`).  Here the
GPU components registered by `components.install()` (the same factories, the same kwargs the
reference's builder passes, the same order: [flatfield_correct,] stitch, find_buttons / find_beads)
run on the `in__` state the way `Pipeline.__call__` runs them (pipeline.py:19-22) and must
reproduce the `out__` state exactly -- values, dims, dtypes, coordinates -- and, for the chip cases,
the `valid` flags the reference's own three filters leave on that state.  /root/reference is not
needed (and does not exist) on the GPU box; centres are pinned to the ones the reference found.
tests/test_dropin_reference.py is the other half: the same layer inside the reference's real
Pipeline, on the CPU stand-in for the kernels.
"""
import pytest

from dropin_cases import replay_bead_case, replay_chip_case

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("case", ["chip_single", "chip_series", "chip_tiles", "chip_blank_float"])
def test_chip_components_reproduce_reference_pipeline(cuda_device, case):
    replay_chip_case(case)


@pytest.mark.parametrize("case", ["beads_single", "beads_flatfield_tiles", "beads_none"])
def test_bead_components_reproduce_reference_pipeline(cuda_device, case):
    replay_bead_case(case)
