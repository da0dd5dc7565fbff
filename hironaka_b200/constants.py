"""Constants of the C-ABI (mirror of include/hironaka_b200.h; tests/test_capi_cpu.py checks
that the two stay identical)."""

HK_VERSION = 106

HK_OK = 0
HK_ERR_BAD_ARG = -1
HK_ERR_UNSUPPORTED = -2
HK_ERR_ALIGN = -3

HK_MAX_DIM = 10
HK_MAX_POINTS = 1024
HK_MAX_GAME_WORDS = 4096

HK_DTYPE_I32 = 0
HK_DTYPE_F32 = 1

HK_OP_SHIFT = 1 << 0
HK_OP_REPOSITION = 1 << 1
HK_OP_NEWTON = 1 << 2
HK_OP_RESCALE = 1 << 3
HK_OP_DEDUPE = 1 << 4

HK_F_NOOP_INVALID = 1 << 0
HK_F_FREEZE_ENDED = 1 << 1
HK_F_ACT_DISCRETE = 1 << 2
HK_F_ROLE_AGENT = 1 << 3
HK_F_OBS_RESCALE = 1 << 4
HK_F_OBS_SORT_COORD0 = 1 << 5
HK_F_OBS_SORT_LEX = 1 << 6
HK_F_ACT_U8 = 1 << 7
HK_F_HOST_ALL_COORD = 1 << 8
HK_F_HOST_ZEILLINGER = 1 << 9
HK_F_AGENT_FIRST = 1 << 10
HK_F_AGENT_LAST = 1 << 11
HK_F_OBS_SORT_LEX_FIRST = 1 << 12
HK_F_STORE_ALL = 1 << 13
HK_F_ACT_PACKED = 1 << 14
HK_F_RESCALE_EPS = 1 << 15
HK_F_ACT_NIBBLE = 1 << 16
HK_F_HOST_RANDOM = 1 << 17
HK_F_AGENT_RANDOM = 1 << 18

# status of a root after hk_search_depth and hk_search_value (HISTORY: hk_search_value only)
HK_SEARCH_RESOLVED = 0
HK_SEARCH_MAX_DEPTH = 1
HK_SEARCH_MAX_NODES = 2
HK_SEARCH_CAPACITY = 3
HK_SEARCH_INT32_BOUND = 4
HK_SEARCH_HISTORY = 5

# the two semantics of the reference
TORCH_SEMANTICS = HK_F_NOOP_INVALID | HK_F_FREEZE_ENDED  # hironaka/src/_torch_ops.py:90-93
JAX_SEMANTICS = 0                                          # hironaka/src/_jax_ops.py:76-90
