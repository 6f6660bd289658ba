"""The committed LUT headers are exactly what tools/gen_tables.py derives from the reference's tile
data, kept as the snapshot tests/golden/tile_data.json."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TILE_DATA = os.path.join(ROOT, "tests", "golden", "tile_data.json")


def test_committed_tables_are_current(tmp_path):
    files = ["pgtg_b200/csrc/pgtg_tables.h", "oracle/pgtg_oracle_tables.h", "pgtg_b200/_names.py"]
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "gen_tables.py"), "--tile-data", TILE_DATA, "--out", str(tmp_path)],
                          stdout=subprocess.DEVNULL)
    for f in files:
        assert open(os.path.join(ROOT, f)).read() == open(os.path.join(tmp_path, f)).read(), f


def test_table_header_shapes():
    text = open(os.path.join(ROOT, "pgtg_b200", "csrc", "pgtg_tables.h")).read()
    assert text.count("0x") > 16 * 81  # 16 x 81 lane descriptors plus the bitmaps
    from pgtg_b200._names import MASK_NAMES, ROUTE_NAMES

    assert len(ROUTE_NAMES) == 20 and ROUTE_NAMES == sorted(ROUTE_NAMES)
    assert MASK_NAMES[:8] == ["blob", "small_blob", "chess_field", "reverse_chess_field", "top_half", "bottom_half", "left_half", "right_half"]
