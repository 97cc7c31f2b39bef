"""_mask_abi: how every wrapper turns a SparseMask into C ABI arguments.  No GPU and no library call."""
import pytest

from ccr_b200.engine import MASK_ADD, MASK_NONE, MASK_SET, SparseMask, _mask_abi


def test_nothing_to_apply_is_none():
    assert _mask_abi(None, 3, 10) is None
    assert _mask_abi(SparseMask.from_lists([[1], [], [2, 3]], 10, -1e6, MASK_NONE, "cpu"), 3, 10) is None
    assert _mask_abi(SparseMask.from_lists([[], [], []], 10, -1e6, MASK_SET, "cpu"), 3, 10) is None


def test_non_empty_mask_gives_pointers_and_counts():
    m = SparseMask.from_lists([[1], [], [9, 2, 3]], 10, 0.5, MASK_ADD, "cpu")
    assert _mask_abi(m, 3, 10) == (m.indptr.data_ptr(), m.cols.data_ptr(), m.vals.data_ptr(), 4, 3, MASK_ADD)


@pytest.mark.parametrize("mode", [MASK_NONE, MASK_SET])
@pytest.mark.parametrize("B,N", [(2, 10), (3, 11)])
def test_shape_mismatch_raises(mode, B, N):
    m = SparseMask.from_lists([[1], [], [2]], 10, -1e6, mode, "cpu")
    with pytest.raises(ValueError, match=rf"mask shape \(3, 10\) does not match \({B}, {N}\)"):
        _mask_abi(m, B, N)
