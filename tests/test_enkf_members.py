"""EnsembleKalmanFilter refuses an ensemble of fewer than two members before any device work (the sample
covariance divides by M - 1), so this runs without a GPU."""
import numpy as np
import pandas as pd
import pytest


def test_one_member_filter_is_refused_and_leaves_the_model_alone(libtxh):
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    n = 200
    net = S.make_network(n, 3)
    d = S.model_dict(net, S.make_params(n, 3, well_posed=True))
    mdl = Muskingum(d, members=1)
    t = mdl.datetime
    o, i = mdl.o_t_next.copy(), mdl.i_t_next.copy()
    g = np.sort(np.random.default_rng(3).choice(n, size=4, replace=False))
    mdf = pd.DataFrame(np.ones((2, 4)), columns=[d["reach_ids"][j] for j in g],
                       index=pd.DatetimeIndex([t + mdl.timedelta * 6, t + mdl.timedelta * 12]))
    with pytest.raises(ValueError, match="at least 2 members"):
        EnsembleKalmanFilter(mdl, mdf, 1.0, 1e-2 * np.eye(4))
    assert mdl.datetime == t
    assert np.array_equal(mdl.o_t_next, o) and np.array_equal(mdl.i_t_next, i)
    assert mdl._dev is None                                   # no device state was created
