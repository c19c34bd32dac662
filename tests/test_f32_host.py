"""Host-side argument checks of Handle.set_matrix_f32 (no GPU needed: they run before the C ABI is called)."""
import numpy as np
import pytest

from ccqppy_b200 import _capi


class _NoLibrary:
    """Stands in for a handle: any call that reached the C ABI would fail on it."""


@pytest.mark.parametrize("bad, exc", [
    (np.ones((4, 4), dtype=np.float64), TypeError),              # not float32
    (np.ones((4, 8), dtype=np.float32)[:, ::2], ValueError),     # columns not contiguous
    (np.ones((3, 4), dtype=np.float32), ValueError),             # wrong shape
    (np.ones(16, dtype=np.float32), ValueError),                 # not a matrix
])
def test_set_matrix_f32_rejects_what_it_cannot_pass_on(bad, exc):
    with pytest.raises(exc):
        _capi.Handle.set_matrix_f32(_NoLibrary(), bad, 4)


def test_set_matrix_f32_rejects_torch_inputs_too():
    torch = pytest.importorskip("torch")
    with pytest.raises(TypeError):
        _capi.Handle.set_matrix_f32(_NoLibrary(), torch.ones((4, 4), dtype=torch.float64), 4)
    with pytest.raises(ValueError):
        _capi.Handle.set_matrix_f32(_NoLibrary(), torch.ones((4, 4), dtype=torch.float32).t(), 4)
