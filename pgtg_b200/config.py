"""Host-side mirror of `PGTGEnv.__init__` (reference pgtg/environment.py:302-359).

`make_config(**kwargs)` takes the reference's keyword arguments (same names, same defaults),
performs the argument checks the reference performs (warnings at environment.py:366-412,
ValueErrors of generate_map at map_generator.py:92-154) and freezes everything into the POD
`pgtg_config` of include/pgtg_b200.h. Quantities the reference derives with Python/numpy
semantics -- banker's `round()`, `cumsum()/cdf[-1]`, `patience_level * 10` -- are computed here, on
the host, with the same operations, so device code only ever compares against finished doubles.
"""
from __future__ import annotations

import ctypes as C
import json
import warnings
from dataclasses import dataclass, field
from typing import Any

import numpy as np

from ._names import CARDINALS, MASK_NAMES, OBSTACLE_NAMES, ROUTE_NAMES

ABI_VERSION = 2
MAX_CHANNELS = 16
MAX_RULES = 8
NUM_PROFILES = 5
NUM_ROUTE_IDS = 20
MAX_TILES = 256
# observation planes as stored by the ticks: int8 cells [N, C, P, P], or bits (env i at bit i * C*P*P; pgtg_set_obs_format)
OBSERVATION_FORMATS = ("int8", "bits")
LEVELS_MAX = 1 << 24  # largest num_levels (the pool of a 16x16-tile map is then 8 GB of descriptors)
LEVEL_SAMPLING = ("uniform", "env_index")

# pgtg_channel
CH_ZERO, CH_WALLS, CH_GOALS, CH_TRAFFIC, CH_ICE, CH_BROKEN, CH_SAND = range(7)
CH_LIGHT_GREEN, CH_LIGHT_YELLOW, CH_LIGHT_RED = 7, 8, 9
CH_SUBGOAL, CH_FINAL_GOAL, CH_START, CH_USED_SUBGOAL, CH_CAR_SPAWNER = 10, 11, 12, 13, 14

RNG_PHILOX, RNG_TAPE, RNG_NUMPY = 0, 1, 2
STREAM_MAP, STREAM_CAR, STREAM_ICE, STREAM_BROKEN, STREAM_SAND = range(5)
DRAW_DOUBLE, DRAW_INDEX = 0, 1

AGENT_DIRECTIONS = ["south_to_north", "west_to_east", "north_to_south", "east_to_west", "stationary", "near_goal"]

DEFAULT_FEATURES = [
    "walls", "goals", "ice", "broken road", "sand", "traffic",
    "traffic_light_green", "traffic_light_yellow", "traffic_light_red",
]

# DRIVER_BEHAVIORS (environment.py:64-109), profile order = DriverProfile declaration order
# (:38-44): conservative, normal, aggressive, elderly, reckless.
PROFILE_NAMES = ["conservative", "normal", "aggressive", "elderly", "reckless"]
DRIVER_BEHAVIORS = {
    #                yellow_stop red_violation min_follow patience speed reaction_delay
    "conservative": (0.95, 0.01, 2, 0.9, 0.8, 0.1),
    "normal": (0.75, 0.05, 1, 0.7, 1.0, 0.15),
    "aggressive": (0.3, 0.15, 0, 0.3, 1.3, 0.05),
    "elderly": (0.98, 0.001, 3, 0.95, 0.6, 0.3),
    "reckless": (0.1, 0.3, 0, 0.1, 1.5, 0.1),
}

# _add_default_rules (environment.py:517-567)
DEFAULT_RULES = [
    {
        "name": "four_way_intersection_brake",
        "tile_type": "1111",
        "velocity_range": [0.5, 10.0],
        "min_traffic": 1,
        "min_matching_traffic": 1,
        "maneuvers": [
            {"agent": "west_to_east", "traffic": ["north_to_south", "south_to_north"]},
            {"agent": "east_to_west", "traffic": ["north_to_south", "south_to_north"]},
            {"agent": "north_to_south", "traffic": ["west_to_east", "east_to_west"]},
            {"agent": "south_to_north", "traffic": ["west_to_east", "east_to_west"]},
        ],
    },
    {
        "name": "t_intersection_brake",
        "tile_type": "1110",
        "velocity_range": [0.5, 10.0],
        "min_traffic": 1,
        "min_matching_traffic": 1,
        "maneuvers": [
            {"agent": "south_to_north", "traffic": ["west_to_east", "east_to_west"]},
            {"agent": "west_to_east", "traffic": ["south_to_north"]},
        ],
    },
]


class PgtgRule(C.Structure):
    _fields_ = [
        ("tile_type", C.c_int32),
        ("min_traffic", C.c_int32),
        ("min_matching_traffic", C.c_int32),
        ("reserved", C.c_int32),
        ("vel_lo", C.c_double),
        ("vel_hi", C.c_double),
        ("weight", (C.c_uint8 * NUM_ROUTE_IDS) * 6),
    ]


class PgtgConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("num_envs", C.c_int32),
        ("env_id_base", C.c_int64),
        ("seed", C.c_uint64),
        ("rng_mode", C.c_int32),
        ("fixed_map", C.c_int32),
        ("map_w", C.c_int32),
        ("map_h", C.c_int32),
        ("edges_to_keep", C.c_int32),
        ("border_connections", C.c_int32),
        ("start_mode", C.c_int32),
        ("goal_mode", C.c_int32),
        ("start_x", C.c_int32),
        ("start_y", C.c_int32),
        ("start_dir", C.c_int32),
        ("goal_x", C.c_int32),
        ("goal_y", C.c_int32),
        ("goal_dir", C.c_int32),
        ("min_start_goal_distance", C.c_int32),
        ("num_levels", C.c_int32),
        ("obstacle_probability", C.c_double),
        ("obstacle_cdf", C.c_double * 4),
        ("num_channels", C.c_int32),
        ("channel_kind", C.c_int32 * MAX_CHANNELS),
        ("sliding", C.c_int32),
        ("window_k", C.c_int32),
        ("use_next_subgoal_direction", C.c_int32),
        ("sum_subgoals_reward", C.c_double),
        ("final_goal_bonus", C.c_double),
        ("crash_penalty", C.c_double),
        ("traffic_light_violation_penalty", C.c_double),
        ("standing_still_penalty", C.c_double),
        ("already_visited_position_penalty", C.c_double),
        ("ice_probability", C.c_double),
        ("street_damage_probability", C.c_double),
        ("sand_probability", C.c_double),
        ("traffic_density", C.c_double),
        ("light_green", C.c_int32),
        ("light_yellow", C.c_int32),
        ("light_red", C.c_int32),
        ("ignore_traffic_collisions", C.c_int32),
        ("profile_cdf", C.c_double * NUM_PROFILES),
        ("drv_yellow_stop", C.c_double * NUM_PROFILES),
        ("drv_red_violation", C.c_double * NUM_PROFILES),
        ("drv_patience_threshold", C.c_double * NUM_PROFILES),
        ("drv_push_probability", C.c_double * NUM_PROFILES),
        ("drv_speed_multiplier", C.c_double * NUM_PROFILES),
        ("drv_reaction_delay", C.c_double * NUM_PROFILES),
        ("drv_min_following", C.c_int32 * NUM_PROFILES),
        ("separate_reward_cost", C.c_int32),
        ("num_rules", C.c_int32),
        ("level_sampling", C.c_int32),
        ("rules", PgtgRule * MAX_RULES),
        ("max_episode_steps", C.c_int32),
        ("write_final_obs", C.c_int32),
        ("max_cars", C.c_int32),
        ("start_level", C.c_int32),
    ]


class PgtgTile(C.Structure):
    _fields_ = [("exits", C.c_uint8), ("obstacle_type", C.c_uint8), ("obstacle_mask", C.c_uint8), ("reserved", C.c_uint8)]


@dataclass
class MapPlan:
    """A fixed map plan (reference MapPlan, map_generator.py:10-40)."""

    width: int
    height: int
    tiles: list  # tiles[y][x] = {"exits": [n,e,s,w], "obstacle_type": str|None, "obstacle_mask": str|None}
    start: tuple
    goal: tuple

    @classmethod
    def from_dict(cls, data: dict) -> "MapPlan":
        # MapPlan.from_dict (map_generator.py:20-29): KeyError when start/goal are missing
        return cls(data["width"], data["height"], data["map"], tuple(data["start"]), tuple(data["goal"]))

    @classmethod
    def from_json(cls, path: str) -> "MapPlan":
        # json_file_to_map_plan (parser.py:227-241)
        if not path.endswith(".json"):
            path = path + ".json"
        with open(path) as f:
            return cls.from_dict(json.load(f))

    def to_dict(self) -> dict:
        return {"width": self.width, "height": self.height, "map": self.tiles, "start": list(self.start), "goal": list(self.goal)}

    def packed_tiles(self):
        arr = (PgtgTile * (self.width * self.height))()
        for y in range(self.height):
            for x in range(self.width):
                t = self.tiles[y][x]
                ex = t["exits"]
                arr[y * self.width + x].exits = int(ex[0]) | int(ex[1]) << 1 | int(ex[2]) << 2 | int(ex[3]) << 3
                ot = t.get("obstacle_type")
                if ot is not None:
                    if ot not in OBSTACLE_NAMES:
                        raise ValueError(f"Unknown obstacle type: {ot}")  # parser.py:205 assert
                    if t.get("obstacle_mask") is None:
                        raise ValueError(f"The tile at ({x},{y}) has a obstacle type without a obstacle mask")
                    arr[y * self.width + x].obstacle_type = 1 + OBSTACLE_NAMES.index(ot)
                    arr[y * self.width + x].obstacle_mask = MASK_NAMES.index(t["obstacle_mask"])
        return arr


@dataclass
class HostConfig:
    """Everything the Python host needs next to the POD."""

    pod: PgtgConfig
    kwargs: dict
    observation_keys: list  # ordered keys of obs["map"]
    window: int
    map_plan: MapPlan | None = None
    rules: list = field(default_factory=list)
    observation_format: str = "int8"  # how the ticks store the observation planes: int8 cells or bits (pgtg_set_obs_format)


def _validate_generate_map_args(width, height, start_position, goal_position, min_dist):
    """Reject what generate_map rejects (map_generator.py:92-154), with its messages. A position is "random", a border
    tile (x, y) or a border tile with the side it opens to (x, y, side); -1 counts from the far edge."""
    for name, pos in (("start_position", start_position), ("goal_position", goal_position)):
        if isinstance(pos, str):
            if pos != "random":
                raise ValueError(f"{name} must be a tuple or the string 'random'.")
            continue
        if not isinstance(pos, tuple):
            continue
        # the map borders this tile lies on: coordinate 0 / -1 or the last index of its axis
        on = {"west": pos[0] == 0, "east": pos[0] in (-1, width - 1), "north": pos[1] == 0, "south": pos[1] in (-1, height - 1)}
        if not any(on.values()):
            raise ValueError(f"{name} must specify a tile on the map border.")
        if len(pos) == 3 and pos[2] in on and not on[pos[2]]:
            raise ValueError(f"The direction in {name} is not a map border.")
    both_exact = all(isinstance(p, tuple) and len(p) == 3 for p in (start_position, goal_position))
    if both_exact and start_position == goal_position:
        raise ValueError("start_position and goal_position can't be the same tile and direction.")
    if min_dist is not None:
        if "random" not in (start_position, goal_position):  # (the reference lets one fixed end pass)
            raise ValueError(
                "minimum_distance_between_start_and_goal can only be used if start_position and goal_position are 'random'."
            )
        if min_dist > width + height - 2:
            raise ValueError("minimum_distance_between_start_and_goal can't be larger than width + height - 2.")


def _position_fields(position, width, height):
    """-> (mode, x, y, dir) with -1 coordinates resolved (map_generator.py:503-533)."""
    if position == "random":
        return 2, 0, 0, 0
    x = position[0] if position[0] != -1 else width - 1
    y = position[1] if position[1] != -1 else height - 1
    if len(position) == 2:
        return 1, x, y, 0
    return 0, x, y, CARDINALS.index(position[2])


def observation_layout(features: list[str]) -> list[tuple[str, int]]:
    """Ordered (key, plane kind) pairs of obs["map"] for a feature list.

    Follows get_observation (environment.py:1387-1445): "walls", "goals" and "traffic" are
    special-cased; a literal "traffic_light" entry expands to the three phase planes; every other
    name is matched literally against the squares' feature strings -- which is why the default
    "traffic_light_green/yellow/red" planes are always zero (no square carries those strings).
    The reference's key order for the literal planes is set-iteration order (hash-randomised);
    this layout fixes it to the order of `features`.
    """
    out: dict[str, int] = {}
    literal = {
        "wall": CH_WALLS, "subgoal": CH_SUBGOAL, "final goal": CH_FINAL_GOAL, "start": CH_START,
        "used subgoal": CH_USED_SUBGOAL, "ice": CH_ICE, "broken road": CH_BROKEN, "sand": CH_SAND,
        "car_spawner": CH_CAR_SPAWNER,
    }
    for name in features:
        if name == "walls":
            out[name] = CH_WALLS
        elif name == "goals":
            out[name] = CH_GOALS
        elif name == "traffic":
            out[name] = CH_TRAFFIC
        elif name == "traffic_light":
            for key, kind in (("traffic_light_green", CH_LIGHT_GREEN), ("traffic_light_yellow", CH_LIGHT_YELLOW), ("traffic_light_red", CH_LIGHT_RED)):
                out.setdefault(key, kind)
        elif name.startswith("car_lane"):
            raise NotImplementedError(f"observation plane for literal lane feature {name!r} is not supported")
        else:
            # the generic loop runs after the special cases and overwrites their keys (:1441-1445)
            out[name] = literal.get(name, CH_ZERO)
    return list(out.items())


def rule_to_pod(rule: dict) -> PgtgRule:
    """TrafficRule.from_dict (environment.py:141-159) flattened."""
    r = PgtgRule()
    tt = rule["tile_type"]
    r.tile_type = -1
    if isinstance(tt, str) and len(tt) == 4 and set(tt) <= {"0", "1"}:
        r.tile_type = int(tt[0]) | int(tt[1]) << 1 | int(tt[2]) << 2 | int(tt[3]) << 3
    r.min_traffic = int(rule["min_traffic"])
    r.min_matching_traffic = int(rule["min_matching_traffic"])
    r.vel_lo = float(rule["velocity_range"][0])
    r.vel_hi = float(rule["velocity_range"][1])
    for m in rule["maneuvers"]:
        if m["agent"] not in AGENT_DIRECTIONS:
            continue  # can never equal get_agent_direction()'s result
        a = AGENT_DIRECTIONS.index(m["agent"])
        for route in set(m["traffic"]):
            if route in ROUTE_NAMES:
                r.weight[a][ROUTE_NAMES.index(route)] += 1
    return r


def make_config(
    map_path: str | None = None,
    *,
    random_map_width: int = 4,
    random_map_height: int = 4,
    random_map_percentage_of_connections: float = 0.5,
    random_map_start_position: Any = (0, -1, "west"),
    random_map_goal_position: Any = (-1, 0, "east"),
    random_map_minimum_distance_between_start_and_goal: int | None = None,
    random_map_obstacle_probability: float = 0.0,
    random_map_ice_probability_weight: float = 1,
    random_map_broken_road_probability_weight: float = 1,
    random_map_sand_probability_weight: float = 1,
    random_map_traffic_light_probability_weight: float = 1,
    render_mode: str | None = None,
    features_to_include_in_observation: list[str] | None = None,
    use_sliding_observation_window: bool = False,
    sliding_observation_window_size: int = 4,
    use_next_subgoal_direction: bool = False,
    sum_subgoals_reward: int = 100,
    final_goal_bonus: int = 0,
    crash_penalty: int = 100,
    traffic_light_violation_penalty: int = 50,
    standing_still_penalty: int = 0,
    already_visited_position_penalty: int = 0,
    ice_probability: float = 0.1,
    street_damage_probability: float = 0.1,
    sand_probability: float = 0.2,
    traffic_density: float = 0.0,
    traffic_light_phases_duration: tuple = (10, 3, 10),
    ignore_traffic_collisions: bool = False,
    max_allowed_deviation: int | None = 10,
    conservative_driver_percentage: float = 0.25,
    normal_driver_percentage: float = 0.35,
    aggressive_driver_percentage: float = 0.20,
    elderly_driver_percentage: float = 0.15,
    reckless_driver_percentage: float = 0.05,
    separate_reward_cost: bool = False,
    # --- vector-env additions -----------------------------------------------------------------
    num_envs: int = 1,
    max_episode_steps: int | None = None,
    seed: int = 0,
    env_id_base: int = 0,
    rng_mode: int | str = RNG_PHILOX,
    final_observation: bool = False,
    map_plan: MapPlan | dict | None = None,
    traffic_rules: list | None = None,
    num_levels: int = 0,
    start_level: int = 0,
    level_sampling: str = "uniform",
    observation_format: str = "int8",
) -> HostConfig:
    kwargs = dict(locals())
    features = list(DEFAULT_FEATURES if features_to_include_in_observation is None else features_to_include_in_observation)
    if render_mode is not None:
        raise NotImplementedError("rendering (pgtg/graphic.py) is out of scope for the batched simulator")

    # the reference's "unobservable obstacle" warnings (environment.py:366-412)
    if random_map_obstacle_probability > 0:
        for weight, feat, text in [
            (random_map_ice_probability_weight, "ice", "The ice obstacle is used in the map generation but not included in the observation. An agent will not be able to learn to avoid it."),
            (random_map_broken_road_probability_weight, "broken road", "The broken road obstacle is used in the map generation but not included in the observation. An agent will not be able to learn to avoid it."),
            (random_map_sand_probability_weight, "sand", "The sand obstacle is used in the map generation but not included in the observation. An agent will not be able to learn to avoid it."),
            (random_map_traffic_light_probability_weight, "traffic_light_green", "The traffic light obstacle is used in the map generation but green traffic lights are not included in the observation. An agent will not be able to learn to avoid it."),
            (random_map_traffic_light_probability_weight, "traffic_light_yellow", "The traffic light obstacle is used in the map generation but yellow traffic lights are not included in the observation. An agent will not be able to learn to avoid it."),
            (random_map_traffic_light_probability_weight, "traffic_light_red", "The traffic light obstacle is used in the map generation but red traffic lights are not included in the observation. An agent will not be able to learn to avoid it."),
        ]:
            if weight > 0 and feat not in features:
                warnings.warn(text)
    if traffic_density > 0 and "traffic" not in features:
        warnings.warn("Traffic is generated but not included in the observation. An agent will not be able to learn to avoid it.")

    c = PgtgConfig()
    c.abi_version = ABI_VERSION
    if num_envs < 1:
        raise ValueError("num_envs must be >= 1")
    c.num_envs = int(num_envs)
    c.env_id_base = int(env_id_base)
    c.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    if isinstance(rng_mode, str):
        rng_mode = {"philox": RNG_PHILOX, "tape": RNG_TAPE, "numpy": RNG_NUMPY}[rng_mode]
    c.rng_mode = int(rng_mode)
    if c.rng_mode == RNG_NUMPY and (int(seed) + int(env_id_base) < 0 or int(seed) + int(env_id_base) + int(num_envs) >= 2 ** 64):
        raise ValueError("numpy rng mode needs seeds in [0, 2**64)")

    plan = None
    if map_plan is not None:
        plan = map_plan if isinstance(map_plan, MapPlan) else MapPlan.from_dict(map_plan)
    elif map_path is not None:
        plan = MapPlan.from_json(map_path)
    if plan is not None:
        c.fixed_map = 1
        W, H = plan.width, plan.height
    else:
        W, H = int(random_map_width), int(random_map_height)
        start, goal = random_map_start_position, random_map_goal_position
        if isinstance(start, list):
            start = tuple(start)
        if isinstance(goal, list):
            goal = tuple(goal)
        _validate_generate_map_args(W, H, start, goal, random_map_minimum_distance_between_start_and_goal)
        c.start_mode, c.start_x, c.start_y, c.start_dir = _position_fields(start, W, H)
        c.goal_mode, c.goal_x, c.goal_y, c.goal_dir = _position_fields(goal, W, H)
        d = random_map_minimum_distance_between_start_and_goal
        c.min_start_goal_distance = -1 if d is None else int(d)
        # len(removable_edges) counts directed edges (map_generator.py:227, 242); Python round()
        n_removable = 2 * (W * (H - 1) + H * (W - 1))
        c.edges_to_keep = round(n_removable * random_map_percentage_of_connections)
        c.border_connections = round((2 * W + 2 * H - 2) * random_map_percentage_of_connections)  # :362-364
        c.obstacle_probability = float(random_map_obstacle_probability)
        weights = [random_map_ice_probability_weight, random_map_broken_road_probability_weight,
                   random_map_sand_probability_weight, random_map_traffic_light_probability_weight]
        wsum = sum(weights)  # map_generator.py:396-411
        if random_map_obstacle_probability > 0:
            if not wsum > 0:
                raise ValueError("obstacle probability weights must sum to a positive number")
            p = np.array([w / wsum for w in weights], dtype=np.float64)
            cdf = p.cumsum()
            cdf /= cdf[-1]  # Generator.choice(p=...) internals
            c.obstacle_cdf[:] = cdf.tolist()
    if W < 1 or H < 1 or W * H > MAX_TILES:
        raise ValueError(f"map of {W}x{H} tiles is outside the supported range (1..{MAX_TILES} tiles)")
    c.map_w, c.map_h = W, H

    layout = observation_layout(features)
    if len(layout) > MAX_CHANNELS:
        raise ValueError(f"at most {MAX_CHANNELS} observation planes are supported")
    c.num_channels = len(layout)
    for i, (_, kind) in enumerate(layout):
        c.channel_kind[i] = kind
    c.sliding = int(bool(use_sliding_observation_window))
    c.window_k = int(sliding_observation_window_size)
    c.use_next_subgoal_direction = int(bool(use_next_subgoal_direction))
    window = 9 if not use_sliding_observation_window else 1 + 2 * int(sliding_observation_window_size)

    c.sum_subgoals_reward = float(sum_subgoals_reward)
    c.final_goal_bonus = float(final_goal_bonus)
    c.crash_penalty = float(crash_penalty)
    c.traffic_light_violation_penalty = float(traffic_light_violation_penalty)
    c.standing_still_penalty = float(standing_still_penalty)
    c.already_visited_position_penalty = float(already_visited_position_penalty)
    c.ice_probability = float(ice_probability)
    c.street_damage_probability = float(street_damage_probability)
    c.sand_probability = float(sand_probability)
    c.traffic_density = float(traffic_density)
    c.light_green, c.light_yellow, c.light_red = (int(v) for v in traffic_light_phases_duration)
    if c.light_green + c.light_yellow + c.light_red <= 0:
        raise ValueError("traffic_light_phases_duration must sum to a positive number")
    c.ignore_traffic_collisions = int(bool(ignore_traffic_collisions))

    # driver profile percentages, normalised as at environment.py:493-508
    pct = [conservative_driver_percentage, normal_driver_percentage, aggressive_driver_percentage,
           elderly_driver_percentage, reckless_driver_percentage]
    total = sum(pct)
    pct = [v / total for v in pct] if total > 0 else [0.0, 1.0, 0.0, 0.0, 0.0]
    cdf = np.array(pct, dtype=np.float64).cumsum()
    cdf /= cdf[-1]
    c.profile_cdf[:] = cdf.tolist()
    for i, name in enumerate(PROFILE_NAMES):
        ys, rv, mf, pl, sm, rd = DRIVER_BEHAVIORS[name]
        c.drv_yellow_stop[i] = ys
        c.drv_red_violation[i] = rv
        c.drv_min_following[i] = mf
        c.drv_patience_threshold[i] = pl * 10   # environment.py:954
        c.drv_push_probability[i] = 1.0 - pl    # environment.py:956
        c.drv_speed_multiplier[i] = sm
        c.drv_reaction_delay[i] = rd
    c.separate_reward_cost = int(bool(separate_reward_cost))

    rules = list(DEFAULT_RULES if traffic_rules is None else traffic_rules)
    names = [r["name"] for r in rules]
    if len(set(names)) != len(names):
        raise ValueError("Rule names must be unique.")
    if len(rules) > MAX_RULES:
        raise ValueError(f"at most {MAX_RULES} traffic rules are supported")
    c.num_rules = len(rules)
    for i, r in enumerate(rules):
        c.rules[i] = rule_to_pod(r)

    # level sets (Procgen's num_levels / start_level): a finite pool of generated maps, built once per handle
    if num_levels:
        if c.rng_mode != RNG_PHILOX:
            raise ValueError("num_levels needs rng_mode='philox'")
        if plan is not None:
            raise ValueError("num_levels cannot be combined with map_path / map_plan")
        if not 1 <= int(num_levels) <= LEVELS_MAX:
            raise ValueError(f"num_levels must be in 1..{LEVELS_MAX}")
        if not 0 <= int(start_level) <= 2 ** 31 - 1:
            raise ValueError("start_level must be in 0..2**31 - 1")
        if level_sampling not in LEVEL_SAMPLING:
            raise ValueError(f"level_sampling must be one of {LEVEL_SAMPLING}")
        c.num_levels, c.start_level, c.level_sampling = int(num_levels), int(start_level), LEVEL_SAMPLING.index(level_sampling)
    if observation_format not in OBSERVATION_FORMATS:
        raise ValueError(f"observation_format must be one of {OBSERVATION_FORMATS}")
    c.max_episode_steps = 0 if not max_episode_steps else int(max_episode_steps)
    c.write_final_obs = int(bool(final_observation))
    # car capacity: lane squares per tile <= 32 (crossing), count = int(n_spawnable * density)
    if traffic_density > 0:
        c.max_cars = max(1, int(32 * W * H * min(float(traffic_density), 1.0)))
    else:
        c.max_cars = 1
    return HostConfig(pod=c, kwargs=kwargs, observation_keys=[k for k, _ in layout], window=window, map_plan=plan, rules=rules,
                      observation_format=observation_format)


def direction_lut(radius: int) -> np.ndarray:
    """Host-generated direction table, evaluated with the host libm exactly as the reference does.

    Entry (dy + R) * (2R + 1) + (dx + R):
      bits 0-2  compass octant index into [N, NE, E, SE, S, SW, W, NW] of atan2(dy, dx)
                (_get_subgoal_compass_directions, environment.py:1069-1088);
      bits 3-5  remapped index of atan2(-dy, dx) (get_observation, environment.py:1486-1502).
    """
    import math

    n = 2 * radius + 1
    lut = np.zeros((n, n), dtype=np.uint8)
    PI_8 = math.pi / 8
    remap = {0: 2, 1: 1, 2: 0, 3: 7, 4: 6, 5: 5, 6: 4, 7: 3}
    for dy in range(-radius, radius + 1):
        for dx in range(-radius, radius + 1):
            angle = math.atan2(dy, dx)
            if -PI_8 <= angle < PI_8:
                o = 2
            elif PI_8 <= angle < 3 * PI_8:
                o = 3
            elif 3 * PI_8 <= angle < 5 * PI_8:
                o = 4
            elif 5 * PI_8 <= angle < 7 * PI_8:
                o = 5
            elif angle >= 7 * PI_8 or angle < -7 * PI_8:
                o = 6
            elif -7 * PI_8 <= angle < -5 * PI_8:
                o = 7
            elif -5 * PI_8 <= angle < -3 * PI_8:
                o = 0
            else:
                o = 1
            angle2 = math.atan2(-dy, dx)
            idx = int(((angle2 + math.pi) / (math.pi / 4)) % 8)
            lut[dy + radius, dx + radius] = o | remap[idx] << 3
    return lut
