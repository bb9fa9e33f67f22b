"""Host mirror of `twisterl.twisterl.env` (rust/src/python_interface/env.rs, pyenv.rs).

Every state operation is a kernel launch on the device batch behind the object (`EnvBatch`, n = 1 for
the scalar classes); there is no CPU implementation of the env dynamics in this package.  Methods
that only describe the env (`num_actions`, `obs_shape`, `difficulty`, `twists`) need no device.
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _lib

_live_specs: "weakref.WeakValueDictionary[int, PyBaseEnv]" = weakref.WeakValueDictionary()


class EnvBatch:
    """n envs in structure-of-arrays form on the device (twr_envs): the Env trait applied to all n."""

    def __init__(self, spec: _lib.EnvSpec, n: int, engine: _lib.Engine | None = None):
        self.engine = engine or _lib.default_engine()
        self.spec = _lib.EnvSpec(spec.kind, spec.width, spec.height, spec.difficulty, spec.depth_slope, spec.max_depth)
        self.n = int(n)
        self.cells = spec.width * spec.height
        h = C.c_void_p()
        _lib.check(_lib.load().twr_envs_create(self.engine._h, C.byref(self.spec), self.n, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self.engine, "_h", None):
            _lib.load().twr_envs_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_difficulty(self, d: int):
        _lib.check(_lib.load().twr_envs_set_difficulty(self._h, int(d)))

    def set_state(self, states):
        a = np.ascontiguousarray(states, dtype=np.int64).reshape(self.n, self.cells)
        _lib.check(_lib.load().twr_envs_set_state(self._h, _lib.ptr(a)))

    def set_cell(self, env: int, cell: int, value: int):
        _lib.check(_lib.load().twr_envs_set_cell(self._h, int(env), int(cell), int(value)))

    def reset(self, env_id_base: int = 0, collect_id: int = 0):
        _lib.check(_lib.load().twr_envs_reset(self._h, int(env_id_base), int(collect_id)))

    def step(self, actions):
        a = np.ascontiguousarray(actions, dtype=np.int32).reshape(self.n)
        _lib.check(_lib.load().twr_envs_step(self._h, _lib.ptr(a)))

    def _q(self, name, shape, dtype):
        out = np.zeros(shape, dtype=dtype)
        _lib.check(getattr(_lib.load(), "twr_envs_" + name)(self._h, _lib.ptr(out)))
        return out

    def get_state(self): return self._q("get_state", (self.n, self.cells), np.int64)
    def observe(self): return self._q("observe", (self.n, self.cells), np.int32)
    def masks(self): return self._q("masks", (self.n, _lib.MAX_ACTIONS), np.uint8).astype(bool)
    def reward(self): return self._q("reward", (self.n,), np.float32)
    def is_final(self): return self._q("is_final", (self.n,), np.uint8).astype(bool)
    def success(self): return self._q("success", (self.n,), np.uint8).astype(bool)
    def depth(self): return self._q("depth", (self.n,), np.int32)


class PyBaseEnv:
    """`env.PyBaseEnv` (python_interface/env.rs:39-114).  Subclasses fill `_spec`."""

    _spec: _lib.EnvSpec

    def _init_spec(self, spec: _lib.EnvSpec):
        self._spec = spec
        self._batch: EnvBatch | None = None
        _live_specs[C.addressof(spec)] = self

    # -- description (no device needed)
    def num_actions(self) -> int:
        return 4

    def obs_shape(self) -> list[int]:
        n = self._spec.width * self._spec.height
        return [n, n]

    @property
    def difficulty(self) -> int:
        return int(self._spec.difficulty)

    @difficulty.setter
    def difficulty(self, d: int) -> None:
        d = int(d)
        if d < 0:
            raise OverflowError("can't convert negative int to unsigned")
        if self._spec.kind == _lib.ENV_GRIDWORLD:
            d = min(d, self._spec.width + self._spec.height)      # lib.rs:92-94
        self._spec.difficulty = d
        if self._batch is not None:
            self._batch.set_difficulty(d)

    def twists(self):
        return ([], [])                                           # rl/env.rs:59 default

    def __extract_env__(self) -> int:
        """Address of this env's `twr_env_spec` -- the device-side stand-in for the reference's
        `&Box<dyn Env>` pointer (python_interface/env.rs:109-113)."""
        return C.addressof(self._spec)

    # -- state (device batch of one)
    def _b(self) -> EnvBatch:
        if self._batch is None:
            self._batch = EnvBatch(self._spec, 1)
        return self._batch

    def set_state(self, state) -> None: self._b().set_state([list(state)])
    def reset(self) -> None:
        b = self._b()
        self._resets = getattr(self, "_resets", 0) + 1
        b.reset(env_id_base=0xE0000000 | (id(self) & 0xFFFFFF), collect_id=self._resets)
    def step(self, action: int) -> None: self._b().step([int(action)])
    def masks(self) -> list[bool]: return [bool(x) for x in self._b().masks()[0][: self.num_actions()]]
    def is_final(self) -> bool: return bool(self._b().is_final()[0])
    def reward(self) -> float: return float(self._b().reward()[0])
    def observe(self) -> list[int]: return [int(x) for x in self._b().observe()[0]]


def spec_from_env(env) -> _lib.EnvSpec:
    """What `get_env` does in the reference (python_interface/env.rs:163-177): ask the object for its
    native env.  Objects without a device implementation are rejected -- there is no CPU fallback."""
    try:
        addr = env.__extract_env__()
    except AttributeError:
        raise TypeError("Object must implement __extract_env__ method") from None
    owner = _live_specs.get(int(addr))
    if owner is None or owner is not env:
        raise RuntimeError("this environment has no device implementation (only Puzzle and GridWorld run on the "
                           "B200 engine; there is no CPU fallback for arbitrary Env objects)")
    s = owner._spec
    return _lib.EnvSpec(s.kind, s.width, s.height, s.difficulty, s.depth_slope, s.max_depth)


class Puzzle(PyBaseEnv):
    """`env.Puzzle(width, height, difficulty, depth_slope, max_depth)` (python_interface/env.rs:117-160).  Boards of up to
    25 cells (the 24-puzzle, 5x5, among them) run on the device; a larger board raises RuntimeError at its first use."""

    def __init__(self, width: int, height: int, difficulty: int, depth_slope: int, max_depth: int, add_perms: bool = False):
        for v in (width, height, difficulty, depth_slope, max_depth):
            if int(v) < 0:
                raise OverflowError("can't convert negative int to unsigned")
        kind = _lib.ENV_PUZZLE_WIDE if int(width) * int(height) > 16 else _lib.ENV_PUZZLE
        self._init_spec(_lib.EnvSpec(kind, int(width), int(height), int(difficulty), int(depth_slope), int(max_depth)))
        # Opt-in twist set (docs/twists.md: "gate toggles through config ... an `add_perms` flag"): the reference's Puzzle
        # declares no twists (Env::twists default, rl/env.rs:59), and neither does this one unless asked to
        self._add_perms = bool(add_perms)

    def twists(self):
        """`Env::twists` (rl/env.rs:33,59).  With `add_perms=True` on a square board: {identity, main-diagonal transpose}
        -- cell i and tile label v both move to their transposed index, left<->up and right<->down trade places
        (SURVEY.md section 8a row T: `twist(step(s, a)) == step(twist(s), A(a))`, the solved board is a fixed point)."""
        w, h = self._spec.width, self._spec.height
        if not getattr(self, "_add_perms", False) or w != h:
            return ([], [])
        n = w * h
        t = [(i % w) * w + (i // w) for i in range(n)]
        return ([list(range(n * n)), [t[i] * n + t[v] for i in range(n) for v in range(n)]], [[0, 1, 2, 3], [1, 0, 3, 2]])

    def get_state(self) -> list[int]: return [int(x) for x in self._b().get_state()[0]]
    def solved(self) -> bool: return bool(self._b().success()[0])

    def get_position(self, x: int, y: int) -> int:
        return self.get_state()[y * self._spec.width + x]

    def set_position(self, x: int, y: int, val: int) -> None:
        # envs/puzzle.rs:71-73: pokes one cell, zero_location and depth untouched (twr_envs_set_cell)
        if not (0 <= int(x) < self._spec.width and 0 <= int(y) < self._spec.height):
            raise IndexError("index out of bounds")                # the reference panics on state[y*width + x]
        self._b().set_cell(0, int(y) * self._spec.width + int(x), int(val))

    def display(self) -> None:
        st, w = self.get_state(), self._spec.width
        out = []
        for i, v in enumerate(st):                               # envs/puzzle.rs:56-69
            out.append("   " if v == 0 else (f"  {v} " if v < 10 else f" {v} "))
            if (i + 1) % w == 0:
                out.append("\n")
        print("".join(out), end="")


class GridWorld(PyBaseEnv):
    """`grid_world.GridWorld(width, height, max_steps, difficulty)` (examples/grid_world/src/lib.rs:166-211).  Boards of
    3 to 64 cells (up to 8x8, or 4x16, 1x64, ...) run on the device; a larger board raises RuntimeError at its first use."""

    def __init__(self, width: int, height: int, max_steps: int, difficulty: int):
        for v in (width, height, max_steps, difficulty):
            if int(v) < 0:
                raise OverflowError("can't convert negative int to unsigned")
        d = min(int(width) + int(height), int(difficulty))       # lib.rs:36
        self._init_spec(_lib.EnvSpec(_lib.ENV_GRIDWORLD, int(width), int(height), d, 0, int(max_steps)))

    def get_state(self) -> list[int]: return [int(x) for x in self._b().get_state()[0]]
    def at_goal(self) -> bool: return bool(self._b().success()[0])

    def at_trap(self) -> bool:
        # the agent overwrites the trap cell in the board encoding (lib.rs:74-81)
        return 3 not in self.get_state()

    def get_positions(self):
        st, w = self.get_state(), self._spec.width
        pos = lambda v: ((st.index(v) % w, st.index(v) // w) if v in st else None)
        a = pos(1)
        g = pos(2) or a
        t = pos(3) or a
        return (a, g, t)


class PyEnv(PyBaseEnv):
    """`env.PyEnv(py_obj)` (python_interface/pyenv.rs:21-173): wraps an arbitrary Python env object.
    Scalar calls delegate to the wrapped object; it cannot run on the device, so collectors reject it."""

    def __new__(cls, pyenv=None, *a, **k):
        self = super().__new__(cls)
        self._obj = pyenv
        self._difficulty = 1
        return self

    def __init__(self, *a, **k):
        pass

    def num_actions(self): return int(self._obj.num_actions())
    def obs_shape(self): return list(self._obj.obs_shape())

    @property
    def difficulty(self): return self._difficulty

    @difficulty.setter
    def difficulty(self, d): self._difficulty = int(d)

    def twists(self):
        return self._obj.twists() if hasattr(self._obj, "twists") else ([], [])

    def set_state(self, state): self._obj.set_state(list(state))
    def reset(self): self._obj.reset(self._difficulty)
    def step(self, action): self._obj.next(int(action))
    def masks(self): return [bool(m) for m in self._obj.masks()]
    def is_final(self): return bool(self._obj.is_final())
    def reward(self): return float(self._obj.value())
    def observe(self): return [int(o) for o in self._obj.observe()]

    def __extract_env__(self) -> int:
        raise RuntimeError("PyEnv-wrapped Python environments cannot run on the B200 engine and this package has "
                           "no CPU fallback; port the env to a device kernel (see DESIGN.md)")
