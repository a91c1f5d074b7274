"""Which fold the plain M-best calls rank with (Periods._fold): the fp32 nomination sweep unless the instance or the
module names a fold mode; every named mode, the hierarchy included, keeps its meaning."""
import pytest

from pyperiod_b200 import Periods, _lib


@pytest.fixture
def module_mode():
    saved = _lib._module_fold_mode
    yield _lib.set_fold_mode
    _lib._module_fold_mode = saved


def test_plain_mbest_ranks_in_float_only_when_no_mode_is_named(module_mode):
    module_mode(None)
    assert not _lib.fold_mode_is_set() and _lib.default_fold_mode() == _lib.FOLD_HIERARCHICAL
    assert Periods()._fold(plain_mbest=True) == _lib.FOLD_NOMINATE_F32
    assert Periods()._fold() == _lib.FOLD_HIERARCHICAL                     # other sweeps keep the hierarchy
    assert Periods(dtype="fp32")._fold() == _lib.FOLD_NOMINATE_F32
    for name, mode in _lib.FOLD_NAMES.items():
        assert Periods(fold_mode=name)._fold(plain_mbest=True) == mode
        assert Periods(fold_mode=mode)._fold(plain_mbest=True) == mode
    for mode in _lib.FOLD_NAMES.values():                                  # module-wide, the hierarchy included
        module_mode(mode)
        assert _lib.fold_mode_is_set()
        assert Periods()._fold(plain_mbest=True) == mode
        assert Periods(fold_mode="direct")._fold(plain_mbest=True) == _lib.FOLD_DIRECT
    module_mode(None)
    assert Periods()._fold(plain_mbest=True) == _lib.FOLD_NOMINATE_F32
