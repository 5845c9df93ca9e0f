"""The fp64 restatement of the grouped MCMC sampler (tests/mcmc_groups_ref.py), no GPU needed: with one group it is the C
restatement of the shipped sampler (oracle/fm_oracle.c, which the reference pins) bit for bit -- with no map and with an
explicit all-zero map -- and a real grouping moves the chain far from it.  Also the host mirror's checks of features$attr_group."""
import numpy as np
import pytest

from fmwr_b200 import _lib as L
from fmwr_b200 import api as A
from tests import mcmc_groups_cases as G
from tests.util import relerr


@pytest.mark.parametrize("layout", ["fields", "ragged"])
@pytest.mark.parametrize("task", [L.CLASSIFICATION, L.REGRESSION])
@pytest.mark.parametrize("enable_v", [0, 1])
def test_one_group_is_the_shipped_sampler(port, layout, task, enable_v):
    ds, _ = G.layout(layout)
    y, *init = G.problem(task, ds)
    strm = G.streams(ds["p"], 1)
    shipped = G.oracle_run(port, task, ds, y, init, enable_v, strm)
    for grp, ng in ((None, 1), (np.zeros(ds["p"], np.int32), 1)):
        mine = G.reference_run(port, task, ds, y, init, enable_v, L.COMPAT_REFERENCE, strm, grp, ng)
        assert mine[0] == shipped[0] and np.array_equal(mine[1], shipped[1]) and np.array_equal(mine[2], shipped[2]), (
            relerr(mine[0], shipped[0]), relerr(mine[1], shipped[1]), relerr(mine[2], shipped[2]))


@pytest.mark.parametrize("layout", G.LAYOUTS)
def test_grouping_moves_the_chain(port, layout):
    """negative control for the engine comparison: on its shapes, groups = fields ends far from the one-group chain"""
    ds, fields = G.layout(layout)
    y, *init = G.problem(L.REGRESSION, ds)
    grp, ng = G.group_map("fields", ds["p"], fields)
    strm = G.streams(ds["p"], ng)
    one = G.reference_run(port, L.REGRESSION, ds, y, init, 1, L.COMPAT_REFERENCE, strm, None, 1)
    grouped = G.reference_run(port, L.REGRESSION, ds, y, init, 1, L.COMPAT_REFERENCE, strm, grp, ng)
    assert relerr(grouped[1], one[1]) > 1e-3 and relerr(grouped[2], one[2]) > 1e-3, (relerr(grouped[1], one[1]), relerr(grouped[2], one[2]))


def test_host_mirror_checks_the_map():
    for bad, msg in ((np.zeros(4, np.int32), "one entry per column"), (np.array([0, 1, 0.5, 0, 1]), "one entry per column"),
                     (np.array([0, -1, 0, 0, 0]), "out of range"), (np.array([0, 5, 0, 0, 0]), "at most 65536 and the number of features")):
        with pytest.raises(ValueError, match=msg):
            A._attr_group(bad, 5)
    g, ng = A._attr_group([0, 2, 2, 0, 0], 5)
    assert g.dtype == np.int32 and list(g) == [0, 2, 2, 0, 0] and ng == 3
