"""AT_B200_DEVICES: which engines the streamed regrid deals its chunks to (CPU only)."""

import re

import pytest
from conftest import REPO

from anemoi_transform_b200.device import DEVICES_ENV, fanout_devices, parse_devices


@pytest.mark.parametrize("value", [None, "", "  "])
def test_unset_keeps_the_single_engine(value):
    assert parse_devices(value, 8) is None


def test_unset_variable_selects_no_group(monkeypatch):
    monkeypatch.delenv(DEVICES_ENV, raising=False)
    assert fanout_devices() is None


@pytest.mark.parametrize("value,count,want", [("all", 1, [0]), ("all", 4, [0, 1, 2, 3]), (" ALL ", 2, [0, 1]), ("0,1", 2, [0, 1]), ("3", 4, [3]), ("2, 0", 4, [2, 0])])
def test_all_and_lists(value, count, want):
    assert parse_devices(value, count) == want


def test_a_repeated_ordinal_is_one_more_engine_on_that_device():
    assert parse_devices("0,0", 1) == [0, 0]
    assert parse_devices("1,0,1,1", 2) == [1, 0, 1, 1]


@pytest.mark.parametrize("value", ["x", "0;1", "0,,1", "0,", "-1", "1.0", "0x1", "all,0", "1 2", "٣"])
def test_malformed_values_raise_naming_the_variable(value):
    with pytest.raises(ValueError, match=DEVICES_ENV):
        parse_devices(value, 8)


@pytest.mark.parametrize("value,count", [("2", 2), ("0,8", 8), ("all", 0), ("0", 0)])
def test_ordinals_out_of_range_raise(value, count):
    with pytest.raises(ValueError, match=DEVICES_ENV):
        parse_devices(value, count)


def test_torchrun_processes_refuse_the_variable(monkeypatch):
    with pytest.raises(ValueError, match=f"{DEVICES_ENV}.*torchrun"):
        parse_devices("0,1", 8, local_world_size=2)
    assert parse_devices("0,1", 8, local_world_size=1) == [0, 1]
    assert parse_devices(None, 8, local_world_size=4) is None  # unset stays fine under torchrun
    monkeypatch.setenv(DEVICES_ENV, "all")
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "2")
    with pytest.raises(ValueError, match="torchrun"):
        fanout_devices()


def test_group_entry_points_are_declared_and_bound():
    from anemoi_transform_b200 import _cabi

    header = (REPO / "include" / "at_b200.h").read_text()
    for name in ("at_csr_replicate", "at_hostio_group_create", "at_hostio_group_destroy", "at_hostio_group_regrid", "at_hostio_group_regrid_grib", "at_hostio_group_wait"):
        assert re.search(rf"AT_API\s+int\s+{name}\s*\(", header), name
        assert name in _cabi.PROTOTYPES, name
    # the group entry points cite the call site they serve, like the others
    group_block = header[header.index("at_hostio_group_create") - 600 : header.index("at_hostio_group_wait")]
    assert "regrid.py:174-208" in group_block
