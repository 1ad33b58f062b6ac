"""ctypes mirror of include/tron_b200.h (types and constants only; loads nothing).

Field order and types must match the header exactly; tests/test_abi.py checks sizes/offsets against
values compiled from the header with gcc.
"""
import ctypes as C

ABI_VERSION = 4

# status
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_ALIGN = 0, -1, -2, -3, -4
# tiles (tron/map.py:9-17)
TILE_WALL, TILE_EMPTY, TILE_P1_BODY, TILE_P1_HEAD, TILE_P2_BODY, TILE_P2_HEAD, TILE_P1_SLIDE, TILE_P2_SLIDE = (
    -1, 0, 1, 2, 3, 4, 5, 6)
# dtypes
U8, I32, I64, BF16, F32, I8 = 0, 1, 2, 3, 4, 5
# encodings
ENC_NONE, ENC_LUT1, ENC_POPUP3, ENC_POPUP3_CONST = 0, 1, 2, 3
LAYOUT_TILE8 = 0
LAYOUT_BITS10 = 1
LAYOUT_TRAIL = 2
LAYOUT_BITS = 3
OPT_SPARSE_MIN_CELLS = 1
OPT_TILE_BYTES = 2
OPT_ENCODE_VARIANT = 3
OPT_BITS_CTAS_PER_SM = 4
OPT_TILE_CTAS_PER_SM = 5
SLIDE_NONE, SLIDE_TAPE, SLIDE_ICE, SLIDE_TEMPER = 0, 1, 2, 3
SPAWN_UNIFORM, SPAWN_FAIR = 0, 1
POLICY_UNIFORM, POLICY_FREE_EPS = 0, 1
STATS_SLOTS, STATS_FIELDS = 64, 8
(STAT_EPISODES, STAT_P1_WINS, STAT_P2_WINS, STAT_DRAWS, STAT_EP_TICKS, STAT_BAD_ACTION,
 STAT_ENV_STEPS) = range(7)

DEFAULT_LUT = (1, -1, -2, -3, 10, -10)  # tron/map.py:67-81


class Reward(C.Structure):
    _fields_ = [("step_base", C.c_float), ("step_per_tick", C.c_float), ("win", C.c_float),
                ("lose", C.c_float), ("draw", C.c_float)]


# Named reward policies (see tron_reward_t in the header for the citations).
REWARD_POLICIES = {
    "survivor": (0.0, 1.0, 100.0, -25.0, 0.0),         # DQN.py:224-241 as coded: step index k
    "survivor_readme": (1.0, 0.0, 100.0, -25.0, 0.0),  # README.md:97-111
    "basic": (0.0, 0.0, 100.0, -25.0, 0.0),            # README.md:47, no code in the reference
    "ddqn": (-1.0, 0.0, 100.0, -100.0, 0.0),           # DDQN.py:289-305
    "acktr1": (-1.0, 0.0, 10.0, -10.0, 0.0),           # ACKTR.py:316 + config.py:37
    "acktr2": (-1.0, 0.0, 10.0, -20.0, 0.0),           # config.py:39
    "acktr3": (-1.0, 0.0, 20.0, -10.0, 0.0),           # config.py:41
}


class StepArgs(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("n_envs", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
        ("layout", C.c_int32), ("state", C.c_void_p),
        ("actions", C.c_void_p), ("action_dtype", C.c_int32),
        ("obs", C.c_void_p), ("obs_dtype", C.c_int32), ("obs_enc", C.c_int32),
        ("lut", C.c_int8 * 6), ("pad0", C.c_int8 * 2), ("const_plane", C.c_float),
        ("reward", C.c_void_p), ("reward_table", Reward),
        ("done", C.c_void_p), ("winner", C.c_void_p), ("ep_len_out", C.c_void_p),
        ("auto_reset", C.c_int32), ("spawn", C.c_void_p), ("spawn_mode", C.c_int32),
        ("seed", C.c_uint64), ("counter", C.c_uint64), ("env_id_base", C.c_uint64), ("counter_dev", C.c_void_p),
        ("slide_mode", C.c_int32), ("slide_rate", C.c_float), ("slide_tape", C.c_void_p),
        ("slide_params", C.c_void_p),
        ("stats", C.c_void_p),
        ("policy", C.c_int32), ("policy_epsilon", C.c_float),
        ("n_ticks", C.c_int32), ("obs_every_tick", C.c_int32),
        ("obs_terminal", C.c_void_p), ("extra", C.c_void_p),
        ("obs_prev", C.c_int32), ("pad1", C.c_int32),
    ]


class ReplayRing(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("frame_elems", C.c_int32), ("frame_dtype", C.c_int32),
        ("pad0", C.c_int32), ("capacity", C.c_int64),
        ("state", C.c_void_p), ("next_state", C.c_void_p), ("action", C.c_void_p),
        ("reward", C.c_void_p), ("done", C.c_void_p),
    ]


class ReplayFrames(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("frame_elems", C.c_int32), ("frame_dtype", C.c_int32),
        ("n_slots", C.c_int32), ("rows", C.c_int64),
        ("frames", C.c_void_p), ("terminal", C.c_void_p), ("action", C.c_void_p),
        ("reward", C.c_void_p), ("done", C.c_void_p),
    ]


class ReplayStates(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("n_slots", C.c_int32), ("slot_bytes", C.c_int64),
        ("states", C.c_void_p), ("action", C.c_void_p), ("counter", C.c_void_p), ("slide_params", C.c_void_p),
    ]


def new_step_args(**kw):
    a = StepArgs()
    a.struct_size = C.sizeof(StepArgs)
    a.n_ticks = 1
    for k, v in kw.items():
        if k == "lut":
            for i, x in enumerate(v):
                a.lut[i] = int(x)
        elif k == "reward_table":
            a.reward_table = v if isinstance(v, Reward) else Reward(*v)
        else:
            setattr(a, k, v)
    return a


def cells_per_env(width, height):
    return (width + 2) * (height + 2)


def enc_planes(enc):
    return {ENC_NONE: 0, ENC_LUT1: 1, ENC_POPUP3: 3, ENC_POPUP3_CONST: 4}[enc]


def dtype_size(dt):
    return {U8: 1, I8: 1, BF16: 2, I32: 4, F32: 4, I64: 8}[dt]


def trail_bulk_ok(width, height, enc, dtype):
    """does the trail layout's bulk-store observation kernel (template rows in shared memory, step_trail.cu) cover this
    configuration?  It renders terminal frames; the element-store kernel it falls back to does not."""
    row = 2 * enc_planes(enc) * cells_per_env(width, height) * dtype_size(dtype)
    if row == 0:
        return False
    grp = 1
    while (grp * row) % 16:
        grp *= 2
    while grp < 16 and grp * row < 8192:
        grp *= 2
    return ((grp * row + 15) & ~15) <= 200 * 1024


def state_bytes(n_envs, width, height, layout=LAYOUT_TILE8):
    per = 32 if layout == LAYOUT_BITS10 else 48 if layout == LAYOUT_BITS else cells_per_env(width, height)
    if layout == LAYOUT_TRAIL:  # 64 hot bytes (header + 12 list words) + the cold tail of the lists + the bitmap of the cells it names
        per = 64 + ((4 * max(0, width * height - 12) + 15) & ~15)
        if width * height > 12:
            per += (4 * width * ((height + 31) >> 5) + 15) & ~15
    grid = (n_envs * per + 255) & ~255
    meta = (8 * n_envs + 255) & ~255
    return grid + meta + 8 * n_envs


# Every symbol the header declares; tests check that the built library exports each one.
EXPORTED_SYMBOLS = (
    "tron_abi_version", "tron_status_string", "tron_device_count",
    "tron_state_bytes", "tron_state_offsets", "tron_cells_per_env", "tron_enc_planes",
    "tron_dtype_size", "tron_build_plane_tables", "tron_set_option",
    "tron_reset", "tron_reset_ex", "tron_step", "tron_observe", "tron_step_many", "tron_export_grid",
    "tron_import_grid", "tron_random_actions", "tron_select_actions", "tron_advance_counter", "tron_minimax_actions", "tron_pop_up",
    "replay_push", "replay_gather", "replay_sample_indices", "replay_sample_gather", "replay_frames_sample_gather",
    "replay_states_sample_gather",
    "tron_host_env_create", "tron_host_env_destroy", "tron_host_env_reset", "tron_host_env_step",
    "tron_host_env_step_begin", "tron_host_env_step_wait",
    "tron_host_env_state", "tron_host_alloc", "tron_host_free", "tron_host_copy_bandwidth",
    "tron_debug_violations",
)
