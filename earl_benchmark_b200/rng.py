"""Bit-exact replicas of the host RNG streams the reference samples goals / initial states from.

The generators run natively in libearl_b200.so (csrc/mt19937.hpp); this module only wraps them.
Reference call sites (SURVEY.md Appendix D):
  random.sample(task_list, 1)    earl_benchmark/envs/tabletop_manipulation.py:66   -> PyRandom.tabletop_goal_rows
  np.random.uniform(-2.5, 2.5)   earl_benchmark/envs/tabletop_manipulation.py:115-117 -> NumpyLegacyRandom.uniform
  np.random.randint(0, n)        earl_benchmark/envs/sawyer_peg.py:147,151; envs/kitchen.py:123 -> .randint
  SawyerPegV2.reset_model draws  earl_benchmark/envs/sawyer_peg.py:192-229        -> NumpyLegacyRandom.peg_reset_draws
"""
import ctypes as C

import numpy as np

from . import _lib

# 'rc_r-rc_k-rc_g-rc_b' with target_colors ['r','g','b','k'] (tabletop_manipulation.py:35,66-74):
# task index -> row of goal_states
TABLETOP_TASK_TO_ROW = np.array([0, 3, 1, 2], dtype=np.uint8)


def _limbs(seed):
    seed = abs(int(seed))
    out = []
    while True:
        out.append(seed & 0xFFFFFFFF)
        seed >>= 32
        if seed == 0:
            break
    return np.array(out, dtype=np.uint32)


class _Stream:
    _kind = 0

    def __init__(self, seed):
        limbs = _limbs(seed)
        if self._kind == 1 and len(limbs) != 1:
            raise ValueError("legacy numpy seeds are 32-bit")
        self._h = _lib.lib().earl_rng_create(self._kind, limbs.ctypes.data, len(limbs))
        if not self._h:
            raise RuntimeError("earl_rng_create failed")

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        try:
            if h:
                _lib.lib().earl_rng_destroy(h)
        except Exception:  # interpreter shutdown
            pass

    def next_u32(self):
        return int(_lib.lib().earl_rng_next_u32(self._h))


class PyRandom(_Stream):
    """CPython `random.seed(seed)` stream."""
    _kind = 0

    def randbelow(self, n, count):
        out = np.empty(count, np.int32)
        _lib.lib().earl_rng_py_randbelow(self._h, int(n), count, out.ctypes.data)
        return out

    def tabletop_goal_rows(self, count, task_to_row=TABLETOP_TASK_TO_ROW):
        """`count` successive get_next_goal() draws, as rows of goal_states."""
        t = np.ascontiguousarray(task_to_row, np.uint8)
        out = np.empty(count, np.uint8)
        _lib.lib().earl_rng_tabletop_goal_rows(self._h, t.ctypes.data, len(t), count, out.ctypes.data)
        return out


class NumpyLegacyRandom(_Stream):
    """Legacy `np.random.seed(seed)` stream (RandomState / randomkit)."""
    _kind = 1

    def randint(self, n, count):
        out = np.empty(count, np.int32)
        _lib.lib().earl_rng_np_randint(self._h, int(n), count, out.ctypes.data)
        return out

    def uniform(self, low, high, count):
        out = np.empty(count, np.float64)
        _lib.lib().earl_rng_np_uniform(self._h, float(low), float(high), count, out.ctypes.data)
        return out

    def peg_reset_draws(self, count, wide_init=False, reset_at_goal=False):
        """`count` successive SawyerPegV2._draw_one() draws (goal row, peg position), replayed natively:
        (rows int32 [count], pos float64 [count,3])."""
        rows = np.empty(count, np.int32)
        pos = np.empty((count, 3), np.float64)
        _lib.lib().earl_rng_peg_reset_draws(self._h, int(bool(wide_init)), int(bool(reset_at_goal)), count, rows.ctypes.data,
                                            pos.ctypes.data)
        return rows, pos
