"""CPU tests (no GPU) of the deep-list scenes in tests/deep_scenes.py and of the referee oracle on them.

The scene builders must produce the regimes tests/test_gpu_deep_backward.py names, read from the oracle's own
outputs: the exact n_contrib rungs around the blend backward's batch boundaries (BATCH = 256), tiles replayed to the
end of their list (m_len == n) or saturated before it (m_len < n), lists thousands deep, and 8x8 blocks of one tile
with long and short (or empty) hit lists side by side.  On the deepest scenes, the C referee's backward (T_i rebuilt
from fp32 final_T by division) is held to the float64 PyTorch restatement (cumulative products, autograd) at the
bars of tests/parity.py, as tests/test_oracle.py does for ordinary scenes."""
import numpy as np
import pytest

from tests import deep_scenes as D
from tests import parity
from tests.scenes import np_inputs


def _forward(scene):
    return parity.oracle_forward(scene["oracle_settings"], np_inputs(scene["gaussians"]))


@pytest.mark.parametrize("saturated", [False, True], ids=["to_the_end", "saturated"])
@pytest.mark.parametrize("K", D.LADDER)
def test_ladder_rungs(K, saturated):
    fo = _forward(D.ladder_scene(K, saturated))
    assert fo["fragile"].mean() <= parity.MAX_FRAGILE
    D.assert_ladder(fo, K, saturated)


def test_heavy_scene_is_thousands_deep():
    fo = _forward(D.heavy_scene())
    assert fo["fragile"].mean() <= 5e-3
    D.assert_heavy(fo)


@pytest.mark.parametrize("back", [False, True], ids=["front", "back"])
def test_deep_field_scene(back):
    scene = D.deep_field_scene(back=back)
    st = scene["oracle_settings"]
    assert st.image_width % 16 and st.image_height % 16 and st.scale_modifier != 1.0 and np.any(st.bg != 0)
    fo = _forward(scene)
    assert fo["fragile"].mean() <= parity.MAX_FRAGILE
    D.assert_deep_field(fo)


@pytest.mark.parametrize("other", [0, 24], ids=["empty", "short"])
@pytest.mark.parametrize("side", ["left", "right"])
def test_half_block_imbalance(side, other):
    fo = _forward(D.half_block_scene(side, other))
    assert fo["fragile"].mean() <= parity.MAX_FRAGILE
    D.assert_half_block(fo, side, other)


@pytest.mark.parametrize("name", ["heavy", "ladder513_saturated"])
def test_referee_backward_matches_float64_autograd(name):
    """The C referee's backward against float64 autograd through the PyTorch restatement, at the parity bars."""
    scene = D.heavy_scene() if name == "heavy" else D.ladder_scene(513, True)
    fo = _forward(scene)
    dL = D.seed_dL(fo, 17)
    gc = parity.oracle_backward(fo, dL)
    gt = D.f64_reference(scene, dL)
    names = parity.GRAD_NAMES + ("means2D",)
    out = parity.check_grads(fo, gt, {k: gc[k] for k in names})
    assert out["n"] > 0 and out["row_fail"] == 0.0
