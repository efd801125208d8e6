"""Host-side plumbing of multi-column equi-join keys: key-count checks, str / list key normalisation and the runtime-filter
refusal all happen before the first batch reaches the device, so none of these tests needs a GPU."""

import pandas as pd
import pytest

from bodo_b200 import B200Error
from bodo_b200.physical import PhysicalJoin, merge
from bodo_b200.streaming.join import build_runtime_filter, init_join_state, runtime_join_filter
from bodo_b200.table import Table

NAMES_B = ("a", "b", "c", "d", "e")
NAMES_P = ("v", "w", "x", "y", "z")


@pytest.mark.parametrize("nk", [2, 3, 4])
def test_init_join_state_accepts_two_to_four_keys(nk):
    bk = tuple(range(nk - 1, -1, -1))  # non-leading, reversed logical positions
    pk = tuple(range(1, nk + 1))
    st = init_join_state(-1, bk, pk, NAMES_B, NAMES_P, False, False)
    assert st.build_key_inds == bk and st.probe_key_inds == pk and st.handle is None
    # the physical (keys-first) column order puts key position j at physical column j
    t = Table.from_pandas(pd.DataFrame({n: [1, 2] for n in NAMES_B}))
    phys = st._physical(t, st.build_key_inds)
    assert phys[:nk] == list(bk) and sorted(phys) == list(range(5))


@pytest.mark.parametrize("bk,pk", [((), ()), ((0, 1, 2, 3, 4), (0, 1, 2, 3, 4)), ((0, 1), (0,)), ((0,), (0, 1))])
def test_init_join_state_rejects_bad_key_counts(bk, pk):
    with pytest.raises(B200Error, match="between 1 and 4 equi-join keys"):
        init_join_state(-1, bk, pk, NAMES_B, NAMES_P, False, False)


def test_physical_join_and_merge_normalise_keys():
    j = PhysicalJoin(2, 0, NAMES_B, NAMES_P)
    assert j.state.build_key_inds == (2,) and j.state.probe_key_inds == (0,)
    j = PhysicalJoin([3, 1], (0, 4), NAMES_B, NAMES_P, how="outer")
    assert j.state.build_key_inds == (3, 1) and j.state.probe_key_inds == (0, 4) and j.state.build_outer and j.state.probe_outer
    left = pd.DataFrame({"x": [1], "y": [2]})
    right = pd.DataFrame({"u": [1], "w": [2]})
    with pytest.raises(B200Error, match="same length"):
        merge(left, right, left_on=["x", "y"], right_on=["u"])
    with pytest.raises(B200Error, match="between 1 and 4 equi-join keys"):
        merge(left, right, left_on=["x", "y", "x", "y", "x"], right_on=["u", "w", "u", "w", "u"])


def test_runtime_filters_refuse_multi_key_states():
    st = init_join_state(-1, (0, 1), (0, 1), NAMES_B, NAMES_P, False, False)
    with pytest.raises(B200Error, match="multi-column runtime join filters are not built yet"):
        build_runtime_filter(st)
    t = Table.from_pandas(pd.DataFrame({"v": [1, 2], "w": [3, 4]}))
    with pytest.raises(B200Error, match="multi-column runtime join filters are not built yet"):
        runtime_join_filter((st,), t, ((0, 1),))
    with pytest.raises(B200Error, match="multi-column runtime join filters are not built yet"):
        runtime_join_filter((st,), t, ((0,),))
    single = init_join_state(-1, (0,), (0,), NAMES_B, NAMES_P, False, False)
    with pytest.raises(B200Error, match="multi-column runtime join filters are not built yet"):
        runtime_join_filter((single,), t, ((0, 1),))
