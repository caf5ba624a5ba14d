"""CPU test: a single image with fractional yaws (no integer column roll) may be split over several devices."""


def test_split_devices_accepts_fractional_tables(pkg):
    from p2p_b200 import panorama_to_plane_pitch as front

    Wp = 1000
    yaws = [0, 30, 33.3, 90]
    tables = [pkg.yaw_table(Wp, y) for y in yaws]
    assert any(t[2] is None for t in tables) and any(t[2] is not None for t in tables)
    assert front._split_devices([0, 1], tables, yaws, [60]) == [0, 1]
    assert front._split_devices([0, 0, 0], tables[1:3], yaws[1:3], [60, 120]) == [0, 0, 0]
    assert front._split_devices([0], tables, yaws, [60]) is None
    assert front._split_devices([0, 1], tables, yaws, []) is None
