#!/usr/bin/env python3
"""Generate the packed tile LUTs from the reference's literal tile data.

Reads the reference's pgtg/map_tiles_data.py (TILES :2, OBSTACLE_MASKS :1502, TRAFFIC_LANES :2220)
from the tree named by PGTG_REFERENCE and pgtg/constants.py (:18-36), checks every structural assumption the
kernels rely on, and emits two *differently shaped* derived tables:

  pgtg_b200/csrc/pgtg_tables.h   81-bit bitmaps + packed 64-bit lane descriptors (CUDA product)
  oracle/pgtg_oracle_tables.h    per-square feature words + lane lists (CPU oracle)

Both headers are committed; this script is the recipe that made them (`python tools/gen_tables.py`).
The tile data it reads is also kept as a JSON snapshot, tests/golden/tile_data.json
(`--write-tile-data FILE` writes it from a reference tree), so that tests/test_tables.py re-derives the
committed tables without the reference: `--tile-data FILE` reads the snapshot, `--out DIR` writes the
three files under DIR instead of into the repository.

Index conventions (shared by oracle and product, defined here once):
  tile type  e = N | E<<1 | S<<2 | W<<3          (exits list order [north,east,south,west])
  square bit  = lx*9 + ly                         (templates are indexed [x][y], parser.py:151-155)
  direction   up=0 down=1 left=2 right=3          (probe order, environment.py:891-902)
  route id    = rank of the route name in sorted() order (environment.py:861, 922, 989 sort names)
  mask id     0..7 = constants.OBSTACLE_MASK_NAMES order (the rng.choice index space,
              map_generator.py:430), 8..13 = traffic_light_{north,east,south,west,
              north_and_south,east_and_west} (append order at map_generator.py:436-468)
  obstacle    1 ice, 2 broken road, 3 sand, 4 traffic_light (constants.OBSTACLE_NAMES order + 1)
"""
import argparse
import json
import os
import sys
from types import SimpleNamespace

REF = os.environ.get("PGTG_REFERENCE", "/root/reference")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DIRS = ["up", "down", "left", "right"]
CARD = ["north", "east", "south", "west"]
TL_MASKS = [
    "traffic_light_north",
    "traffic_light_east",
    "traffic_light_south",
    "traffic_light_west",
    "traffic_light_north_and_south",
    "traffic_light_east_and_west",
]


def load_reference():
    sys.path.insert(0, os.path.join(REF, "pgtg"))
    import constants
    import map_tiles_data as d

    return constants, d


def _grid(squares):
    return [[set(c) for c in col] for col in squares]


def load_tile_data(path):
    """The same (constants, map_tiles_data) view as load_reference(), from a snapshot written by write_tile_data()."""
    with open(path) as f:
        s = json.load(f)
    constants = SimpleNamespace(
        TILE_WIDTH=s["TILE_WIDTH"], TILE_HEIGHT=s["TILE_HEIGHT"], OBSTACLE_NAMES=s["OBSTACLE_NAMES"],
        OBSTACLE_MASK_NAMES=s["OBSTACLE_MASK_NAMES"], DIRECTIONS_TO_INTS=s["DIRECTIONS_TO_INTS"],
        ACTIONS_TO_ACCELERATION={a: tuple(acc) for a, acc in s["ACTIONS_TO_ACCELERATION"]})
    d = SimpleNamespace(
        TILES={tuple(t["exits"]): _grid(t["squares"]) for t in s["TILES"]},
        OBSTACLE_MASKS={name: _grid(m) for name, m in s["OBSTACLE_MASKS"].items()},
        TRAFFIC_LANES={tuple(t["exits"]): _grid(t["squares"]) for t in s["TRAFFIC_LANES"]})
    return constants, d


def write_tile_data(path):
    """Snapshot of the reference data derive() reads: feature sets as sorted lists, tiles in tile-type order."""
    constants, d = load_reference()

    def tiles(table):
        return [dict(exits=[int(v) for v in exits], squares=[[sorted(c) for c in col] for col in t])
                for exits, t in sorted(table.items(), key=lambda kv: type_index(kv[0]))]

    s = dict(
        TILE_WIDTH=constants.TILE_WIDTH, TILE_HEIGHT=constants.TILE_HEIGHT, OBSTACLE_NAMES=list(constants.OBSTACLE_NAMES),
        OBSTACLE_MASK_NAMES=list(constants.OBSTACLE_MASK_NAMES), DIRECTIONS_TO_INTS=dict(constants.DIRECTIONS_TO_INTS),
        ACTIONS_TO_ACCELERATION=[[int(a), list(acc)] for a, acc in sorted(constants.ACTIONS_TO_ACCELERATION.items())],
        TILES=tiles(d.TILES),
        OBSTACLE_MASKS={name: [[sorted(c) for c in col] for col in m] for name, m in d.OBSTACLE_MASKS.items()},
        TRAFFIC_LANES=tiles(d.TRAFFIC_LANES))
    with open(path, "w") as f:
        json.dump(s, f, separators=(",", ":"), sort_keys=True)
        f.write("\n")


def type_index(exits):
    return exits[0] | exits[1] << 1 | exits[2] << 2 | exits[3] << 3


def bits81(pred):
    v = 0
    for x in range(9):
        for y in range(9):
            if pred(x, y):
                v |= 1 << (x * 9 + y)
    return v


def derive(tile_data=None):
    constants, d = load_tile_data(tile_data) if tile_data else load_reference()
    assert constants.TILE_WIDTH == 9 and constants.TILE_HEIGHT == 9
    assert constants.OBSTACLE_NAMES == ["ice", "broken road", "sand", "traffic_light"]
    mask_names = list(constants.OBSTACLE_MASK_NAMES) + TL_MASKS
    assert set(mask_names) == set(d.OBSTACLE_MASKS.keys()) and len(mask_names) == 14
    for a, acc in constants.ACTIONS_TO_ACCELERATION.items():
        assert acc == (a // 3 - 1, a % 3 - 1)
    assert constants.DIRECTIONS_TO_INTS == {"north": 0, "east": 1, "south": 2, "west": 3}

    # ---- wall / exit templates ------------------------------------------------------------
    wall = [0] * 16
    exit_line = [None] * 4
    tile_feat = [[[0] * 9 for _ in range(9)] for _ in range(16)]  # oracle: bit0 wall, bit1+d exit d
    assert len(d.TILES) == 16
    for exits, t in d.TILES.items():
        e = type_index(exits)
        assert len(t) == 9 and all(len(c) == 9 for c in t)
        for x in range(9):
            for y in range(9):
                assert t[x][y] <= {"wall", "exit north", "exit east", "exit south", "exit west"}
                f = 1 if "wall" in t[x][y] else 0
                for k, c in enumerate(CARD):
                    if "exit " + c in t[x][y]:
                        f |= 2 << k
                        assert "wall" not in t[x][y], "exit line on a wall"
                tile_feat[e][x][y] = f
        wall[e] = bits81(lambda x, y: "wall" in t[x][y])
        for k, c in enumerate(CARD):
            b = bits81(lambda x, y: ("exit " + c) in t[x][y])
            if exits[k]:
                assert b, "tile with exit has no exit marker"
                assert exit_line[k] in (None, b), "exit line differs between tile types"
                exit_line[k] = b
            else:
                assert b == 0
    # exit lines: 3 squares each, contiguous, never 4-adjacent to another line (A.1 claim)
    for k in range(4):
        assert bin(exit_line[k]).count("1") == 3

    # ---- obstacle masks -------------------------------------------------------------------
    masks = []
    for name in mask_names:
        m = d.OBSTACLE_MASKS[name]
        for x in range(9):
            for y in range(9):
                assert m[x][y] <= {"obstacle"}
        masks.append(bits81(lambda x, y: "obstacle" in m[x][y]))

    # ---- traffic lanes --------------------------------------------------------------------
    routes = set()
    for exits, t in d.TRAFFIC_LANES.items():
        for col in t:
            for s in col:
                for f in s:
                    if f.startswith("car_lane "):
                        r = f.split()[1]
                        if r != "all":
                            routes.add(r)
    routes = sorted(routes)
    assert len(routes) == 20
    rid = {r: i for i, r in enumerate(routes)}

    lane_desc = [[0] * 81 for _ in range(16)]  # packed u64 per square
    lane_list = [[[] for _ in range(81)] for _ in range(16)]  # oracle: [(route, dir)] sorted
    lane_all = [[0] * 81 for _ in range(16)]  # 0 none, 1+dir
    lane_any = [0] * 16
    native_spawner = [0] * 16  # bitmap
    assert (0, 0, 0, 0) not in d.TRAFFIC_LANES and len(d.TRAFFIC_LANES) == 15
    for exits, t in d.TRAFFIC_LANES.items():
        e = type_index(exits)
        for x in range(9):
            for y in range(9):
                sq = x * 9 + y
                feats = t[x][y]
                lanes, alls = [], []
                for f in feats:
                    if f == "car_spawner":
                        native_spawner[e] |= 1 << sq
                        continue
                    parts = f.split()
                    assert parts[0] == "car_lane" and len(parts) == 3 and parts[2] in DIRS, f
                    if parts[1] == "all":
                        alls.append(DIRS.index(parts[2]))
                    else:
                        lanes.append((rid[parts[1]], DIRS.index(parts[2])))
                    # the reference matches by substring (environment.py:915-932); prove that
                    # substring matching equals exact token matching on this vocabulary
                    for r in routes + ["all"]:
                        assert (r in f) == (parts[1] == r), (r, f)
                    for dd in DIRS:
                        assert (dd in f) == (parts[2] == dd), (dd, f)
                assert len(alls) <= 1, "more than one 'all' lane on a square"
                if alls:
                    assert lanes, "tile-entry square without a route lane"
                lanes.sort()
                assert len(lanes) <= 6
                # (route, dir) pairs are unique => at most one lane matches a car's (route, dir)
                assert len(set(lanes)) == len(lanes)
                lane_list[e][sq] = lanes
                lane_all[e][sq] = (alls[0] + 1) if alls else 0
                if lanes or alls:
                    lane_any[e] |= 1 << sq
                v = lane_all[e][sq] | (len(lanes) << 3)
                for i, (r, dd) in enumerate(lanes):
                    v |= (r | dd << 5) << (6 + 7 * i)
                lane_desc[e][sq] = v
    # tile-entry squares: one per present exit, inward direction, fixed local coordinates
    entry_sq = {"right": None, "left": None, "down": None, "up": None}
    for e in range(1, 16):
        for sq in range(81):
            a = lane_all[e][sq]
            if a:
                name = DIRS[a - 1]
                assert entry_sq[name] in (None, sq)
                entry_sq[name] = sq
    for e in range(16):
        n = bin(native_spawner[e]).count("1")
        assert n == (1 if bin(e).count("1") == 1 else 0)
    return dict(
        wall=wall, exit_line=exit_line, masks=masks, mask_names=mask_names, routes=routes,
        lane_desc=lane_desc, lane_list=lane_list, lane_all=lane_all, lane_any=lane_any,
        native_spawner=native_spawner, entry_sq=entry_sq, tile_feat=tile_feat,
    )


def w3(v):
    return "{0x%08xu, 0x%08xu, 0x%08xu}" % (v & 0xFFFFFFFF, (v >> 32) & 0xFFFFFFFF, v >> 64)


HEADER = """// GENERATED by tools/gen_tables.py from the reference's literal tile data
// (pgtg/map_tiles_data.py: TILES :2, OBSTACLE_MASKS :1502, TRAFFIC_LANES :2220). Do not edit.
// Conventions: tile type e = N|E<<1|S<<2|W<<3; square bit = lx*9+ly; dir up0 down1 left2 right3;
// route id = rank in sorted route names; mask id 0..7 = OBSTACLE_MASK_NAMES order, 8..13 lights.
"""


def emit_cuda(t, path):
    o = [HEADER, "#pragma once\n#include <stdint.h>\n"]
    o.append("#define PGTG_NUM_ROUTES 20\n#define PGTG_NUM_MASKS 14\n")
    o.append("// 81-bit bitmaps as 3 x u32 (bit = lx*9+ly)")
    o.append("#define PGTG_TAB_WALL {%s}" % ", ".join(w3(v) for v in t["wall"]))
    o.append("#define PGTG_TAB_EXIT_LINE {%s}" % ", ".join(w3(v) for v in t["exit_line"]))
    o.append("#define PGTG_TAB_MASK {%s}" % ", ".join(w3(v) for v in t["masks"]))
    o.append("#define PGTG_TAB_LANE_ANY {%s}" % ", ".join(w3(v) for v in t["lane_any"]))
    o.append("#define PGTG_TAB_NATIVE_SPAWNER {%s}" % ", ".join(
        str(v.bit_length() - 1 if v else 255) for v in t["native_spawner"]))
    o.append("// tile-entry squares ('car_lane all <dir>'), index = dir (up,down,left,right)")
    o.append("#define PGTG_TAB_ENTRY_SQ {%s}" % ", ".join(str(t["entry_sq"][d]) for d in DIRS))
    o.append("// per (type, square): all_dir+1 (3b) | n_lanes (3b) | 6 x (route 5b | dir 2b)")
    rows = []
    for e in range(16):
        rows.append("{" + ", ".join("0x%xull" % v for v in t["lane_desc"][e]) + "}")
    o.append("#define PGTG_TAB_LANE_DESC {\\\n%s}" % ",\\\n".join(rows))
    o.append("#define PGTG_ROUTE_NAMES {%s}" % ", ".join('"%s"' % r for r in t["routes"]))
    o.append("#define PGTG_MASK_NAMES {%s}" % ", ".join('"%s"' % r for r in t["mask_names"]))
    with open(path, "w") as f:
        f.write("\n".join(o) + "\n")


def emit_oracle(t, path):
    o = [HEADER, "#pragma once\n"]
    o.append("/* per (type, x, y): bit0 wall, bit1..4 'exit north/east/south/west' */")
    o.append("static const unsigned char ORA_TILE[16][9][9] = {")
    for e in range(16):
        o.append(" {" + ",".join("{" + ",".join(str(v) for v in col) + "}" for col in t["tile_feat"][e]) + "},")
    o.append("};")
    o.append("/* per (mask, x, y): 1 = 'obstacle' */")
    o.append("static const unsigned char ORA_MASK[14][9][9] = {")
    for m in t["masks"]:
        o.append(" {" + ",".join("{" + ",".join(str((m >> (x * 9 + y)) & 1) for y in range(9)) + "}" for x in range(9)) + "},")
    o.append("};")
    o.append("/* per (type, x, y): n lanes, then up to 6 (route, dir) sorted by route name; all = 0 none, 1+dir */")
    o.append("typedef struct { unsigned char n, all, spawner; unsigned char route[6], dir[6]; } ora_lane_sq;")
    o.append("static const ora_lane_sq ORA_LANES[16][9][9] = {")
    for e in range(16):
        cols = []
        for x in range(9):
            sqs = []
            for y in range(9):
                sq = x * 9 + y
                ll = t["lane_list"][e][sq]
                r = [str(a) for a, _ in ll] + ["0"] * (6 - len(ll))
                dd = [str(b) for _, b in ll] + ["0"] * (6 - len(ll))
                sp = (t["native_spawner"][e] >> sq) & 1
                sqs.append("{%d,%d,%d,{%s},{%s}}" % (len(ll), t["lane_all"][e][sq], sp, ",".join(r), ",".join(dd)))
            cols.append("{" + ",".join(sqs) + "}")
        o.append(" {" + ",\n  ".join(cols) + "},")
    o.append("};")
    o.append("static const char* const ORA_ROUTE_NAMES[20] = {%s};" % ", ".join('"%s"' % r for r in t["routes"]))
    with open(path, "w") as f:
        f.write("\n".join(o) + "\n")


def emit_python(t, path):
    with open(path, "w") as f:
        f.write('"""GENERATED by tools/gen_tables.py -- name tables for the host side. Do not edit."""\n')
        f.write("ROUTE_NAMES = %r\n" % (t["routes"],))
        f.write("MASK_NAMES = %r\n" % (t["mask_names"],))
        f.write("OBSTACLE_NAMES = ['ice', 'broken road', 'sand', 'traffic_light']\n")
        f.write("DIR_NAMES = %r\n" % (DIRS,))
        f.write("CARDINALS = %r\n" % (CARD,))


OUTPUTS = ["pgtg_b200/csrc/pgtg_tables.h", "oracle/pgtg_oracle_tables.h", "pgtg_b200/_names.py"]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--tile-data", help="read the tile data from this JSON snapshot instead of the reference tree")
    ap.add_argument("--write-tile-data", metavar="FILE", help="write the reference tree's tile data to FILE and exit")
    ap.add_argument("--out", default=ROOT, help="directory the generated files are written under (default: the repository)")
    args = ap.parse_args()
    if args.write_tile_data:
        write_tile_data(args.write_tile_data)
        return
    t = derive(args.tile_data)
    paths = [os.path.join(args.out, p) for p in OUTPUTS]
    for p in paths:
        os.makedirs(os.path.dirname(p), exist_ok=True)
    emit_cuda(t, paths[0])
    emit_oracle(t, paths[1])
    emit_python(t, paths[2])
    print("routes:", t["routes"])
    print("entry squares:", {k: divmod(v, 9) for k, v in t["entry_sq"].items()})
    print("exit lines:", [[divmod(i, 9) for i in range(81) if (b >> i) & 1] for b in t["exit_line"]])
    print("native spawners:", {e: divmod(v.bit_length() - 1, 9) for e, v in enumerate(t["native_spawner"]) if v})
    print("lane counts:", [bin(v).count("1") for v in t["lane_any"]])


if __name__ == "__main__":
    main()
