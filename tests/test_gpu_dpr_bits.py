"""The dense refinement's outputs are those of the build before the sample loop evaluated its samples in pairs, bit for bit.

The sample loop runs a pair of samples as one straight-line body when every lane of the warp has both footprints in the
staged tile, and each sample through the general path otherwise.  Both paths spell out every float32 operation, so the
per-thread sums, and everything after them, must not move by a bit.  tests/golden/dpr_bits.npz holds the outputs of the
runs of tests/dpr_bits_cases.py as written by that earlier build (scripts/dpr_bits_golden.py); every array must be
byte-equal to it."""
import numpy as np
import pytest

from tests import dpr_bits_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def outputs(ctx1080, ctxvga):
    return dpr_bits_cases.run_all(ctx1080, ctxvga)


def test_outputs_are_the_golden_bits(outputs):
    golden = np.load(dpr_bits_cases.GOLDEN)
    assert sorted(golden.files) == sorted(outputs), "run set differs from the golden file"
    differ = [k for k in golden.files if golden[k].dtype != outputs[k].dtype or golden[k].tobytes() != outputs[k].tobytes()]
    assert not differ, f"{len(differ)} of {len(golden.files)} arrays differ from the golden bits: {differ[:8]}"


def test_runs_reach_the_general_path(outputs):
    """The case runs put samples outside the tile (left_roi is only set by the global-memory fetch), so the slow and the
    mixed pairs are exercised as well as the fast ones."""
    assert any(outputs[k].any() for k in outputs if k.endswith("/left_roi") and not k.startswith("bench"))
