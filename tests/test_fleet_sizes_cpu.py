"""ChargingStationFleet(nevs=...) checks the per-station EV counts on the host, before it loads the
library or touches a device."""
import numpy as np
import pytest

import test_fleet_gpu as closed_loop_tests


class _DeviceWork(Exception):
    pass


@pytest.fixture
def no_device(monkeypatch):
    """Any step past the host-side checks raises _DeviceWork."""
    from chargingstation import fleet

    def refuse(*args, **kwargs):
        raise _DeviceWork()

    monkeypatch.setattr(fleet._native, "load", refuse)
    monkeypatch.setattr(fleet, "BiMPC", refuse)
    monkeypatch.setattr(fleet, "PriceSolver", refuse)
    return fleet.ChargingStationFleet


BAD = {
    "too short": [40, 40],
    "too long": [40, 40, 40, 40],
    "two-dimensional": [[40, 40, 40]],
    "zero": [40, 0, 40],
    "negative": [40, -3, 40],
    "float": [40.0, 9.0, 1.0],
    "fractional": [40, 9.5, 1],
    "bool": [True, True, True],
    "string": ["40", "9", "1"],
    "scalar": 40,
}


@pytest.mark.parametrize("nevs", list(BAD.values()), ids=list(BAD))
def test_bad_nevs_raise_before_device_work(no_device, nevs):
    consts = closed_loop_tests._consts(2, 8, 4, 40, 6, 1)
    with pytest.raises(AssertionError):
        no_device(consts, 3, nevs=nevs)


@pytest.mark.parametrize("nevs", [None, [1, 9, 40], np.array([500, 1, 2], dtype=np.int32),
                                  np.array([3, 3, 3], dtype=np.uint16)], ids=["default", "list", "int32", "uint16"])
def test_good_nevs_pass_the_host_checks(no_device, nevs):
    consts = closed_loop_tests._consts(2, 8, 4, 40, 6, 1)
    with pytest.raises(_DeviceWork):
        no_device(consts, 3, nevs=nevs)
