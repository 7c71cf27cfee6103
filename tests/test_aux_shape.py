"""winterfell_b200.aux_shape reads (aux width, random elements, aux assertion values) off a flat AIR description: the shapes
dist.prove_air_aux_sharded gives its callbacks. Host-only."""
import numpy as np

import airs
import airs_aux
import winterfell_b200 as wf


def test_aux_shape_of_two_segment_airs():
    assert wf.aux_shape(airs.perm_rap(64)[0]) == (3, 2, 7)
    assert wf.aux_shape(airs.perm_rap(64, dyn_last_q=True)[0]) == (3, 2, 8)
    assert wf.aux_shape(airs_aux.perm_rap_lanes(64)[0]) == (9, 2, 21)
    assert wf.aux_shape(airs_aux.rap_sums(64)[0]) == (8, 1, 8)


def test_aux_shape_without_aux_segment_or_malformed():
    d = airs.mulfib2(64)[0]
    assert wf.aux_shape(d) == (0, 0, 0)
    assert wf.aux_shape(d[:5]) == (0, 0, 0)
    assert wf.aux_shape(airs.perm_rap(64)[0][:-3]) == (0, 0, 0)
    assert wf.aux_shape(np.zeros(0, dtype=np.uint64)) == (0, 0, 0)


def test_new_airs_pass_the_host_checks():
    # perm_rap_lanes(3) fits the 96-register aux program; a fourth lane does not
    assert wf.air_check(airs_aux.perm_rap_lanes(1 << 12)[0], 12, 8)[0] == 0
    assert wf.air_check(airs_aux.perm_rap_lanes(64, lanes=4)[0], 6, 8)[0] != 0
    assert wf.air_check(airs_aux.rap_sums(1 << 12)[0], 12, 8)[0] == 0


def test_lane_builder_columns_match_the_full_builder():
    from oracle import oracle as O
    n = 64
    for make in (airs_aux.perm_rap_lanes, airs_aux.rap_sums):
        _, _, b = make(n)
        for d in (1, 2, 3):
            rand = O.rand_elems((2, d), d)
            full = b(rand)
            for f in range(full.shape[0]):
                for c in range(1, full.shape[0] - f + 1):
                    assert (b.columns(rand, f, c) == full[f:f + c]).all()
