"""ctypes binding of the C ABI in include/mapf_b200.h (csrc/libmapf_b200.so).

The hot path has no CPU fallback: a missing library, a missing CUDA device or a failing call raises."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB_PATH = os.environ.get("MAPF_B200_LIB", os.path.join(CSRC, "libmapf_b200.so"))  # override: tuning experiments

MAPF_OK, MAPF_ERR_INVALID, MAPF_ERR_KEY, MAPF_ERR_UNSUPPORTED, MAPF_ERR_CUDA, MAPF_ERR_NO_DEVICE = 0, -1, -2, -3, -4, -5
MAPF_SOC, MAPF_MAKESPAN = 0, 1
OPT_AUTO_RESET = 1
OPT_SHARE_SM = 2
OPT_COMPACT = 4
FLAG_DONE, FLAG_COLLISION = 1, 2
POLICY_RANDOM, POLICY_JOINT, POLICY_AGENTS, POLICY_GROUPS, POLICY_TABLE = 0, 1, 2, 3, 4
VTABLE_EMPTY = (1 << 64) - 1     # key of a free value-table slot
VTABLE_REFUSED = 1 << 63         # bit of a value table's count word: a store was dropped for lack of room
NO_CONFLICT = 0xFF  # conflict byte of an episode that did not end in a collision
EPISODE_TIMEOUT, EPISODE_COLLISION, EPISODE_GOAL, EPISODE_TERMINAL_START = 0, 1, 2, 3

EXPORTS = ["mapf_ctx_create", "mapf_ctx_destroy", "mapf_ctx_info", "mapf_ctx_moves", "mapf_ctx_reward_table", "mapf_decode_states",
           "mapf_encode_states", "mapf_count_rows", "mapf_scan_scratch_bytes", "mapf_scan_rows", "mapf_count_scan_rows",
           "mapf_count_scan_range", "mapf_expand",
           "mapf_count_range", "mapf_expand_range", "mapf_checksum", "mapf_step", "mapf_rollout", "mapf_step_host", "mapf_step_host_resident",
           "mapf_evaluate_scratch_bytes", "mapf_evaluate", "mapf_evaluate_groups",
           "mapf_rtdp_backup", "mapf_vtable_store", "mapf_vtable_lookup", "mapf_evaluate_table",
           "mapf_backup", "mapf_backup_range", "mapf_greedy", "mapf_greedy_bcast", "mapf_count_predecessors", "mapf_predecessors",
           "mapf_projected_words", "mapf_project_states", "mapf_parse_map_text", "mapf_parse_scen_text", "mapf_ctx_create_from_text", "mapf_ctx_grid",
           "mapf_group_create", "mapf_group_destroy", "mapf_group_size", "mapf_group_step", "mapf_last_error",
           "mapf_version"]


class MapfSpec(C.Structure):
    _fields_ = [("height", C.c_int32), ("width", C.c_int32), ("obstacles", C.c_void_p), ("n_agents", C.c_int32),
                ("start_rc", C.c_void_p), ("goal_rc", C.c_void_p), ("fail_prob", C.c_double),
                ("reward_of_clash", C.c_double), ("reward_of_goal", C.c_double), ("reward_of_living", C.c_double),
                ("criterion", C.c_int32)]


class MapfInfo(C.Structure):
    _fields_ = [("n_agents", C.c_int32), ("n_cells", C.c_int32), ("state_words", C.c_int32),
                ("moves_in_smem", C.c_int32), ("n_actions", C.c_int64), ("n_states", C.c_uint64 * 2),
                ("start_state", C.c_uint64 * 2), ("goal_state", C.c_uint64 * 2), ("max_row_len", C.c_int64),
                ("device", C.c_int32), ("sm_count", C.c_int32)]


class MapfVtable(C.Structure):
    _fields_ = [("keys", C.c_void_p), ("values", C.c_void_p), ("actions", C.c_void_p), ("capacity", C.c_int64),
                ("count", C.c_void_p)]


class NativeError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("mapf_b200 error %d: %s" % (code, text))
        self.code = code
        self.text = text


_lib = None
_lock = threading.Lock()


def build(verbose=False):
    """Compile csrc/ for sm_100a (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", CSRC], capture_output=True, text=True)
    if verbose or out.returncode:
        print(out.stdout + out.stderr)
    if out.returncode:
        raise RuntimeError("building libmapf_b200.so failed")
    return LIB_PATH


def lib():
    """Load the shared library (once).  Raises if it has not been built: there is no fallback path."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing: build it with `make -C %s` (or `python -c 'import __graft_entry__ as g; "
                               "g.build()'`); gym_mapf_b200 has no CPU fallback" % (LIB_PATH, CSRC))
        L = C.CDLL(LIB_PATH)
        vp, i64, u64, u32, i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_uint32, C.c_int32
        L.mapf_ctx_create.argtypes = [C.POINTER(MapfSpec), i32, C.POINTER(vp)]
        L.mapf_ctx_destroy.argtypes = [vp]
        L.mapf_ctx_destroy.restype = None
        L.mapf_ctx_info.argtypes = [vp, C.POINTER(MapfInfo)]
        L.mapf_ctx_moves.argtypes = [vp, vp, vp, vp, vp]
        L.mapf_ctx_reward_table.argtypes = [vp, vp]
        L.mapf_decode_states.argtypes = [vp, vp, i64, vp, vp]
        L.mapf_encode_states.argtypes = [vp, vp, i64, vp, vp]
        L.mapf_count_rows.argtypes = [vp, vp, vp, i64, vp, vp]
        L.mapf_scan_scratch_bytes.argtypes = [i64]
        L.mapf_scan_scratch_bytes.restype = i64
        L.mapf_scan_rows.argtypes = [vp, vp, i64, vp, vp, vp]
        L.mapf_count_scan_rows.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp]
        L.mapf_count_scan_range.argtypes = [vp, C.POINTER(u64 * 2), i64, vp, vp, vp, vp]
        L.mapf_expand.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp, vp, vp]
        L.mapf_count_range.argtypes = [vp, C.POINTER(u64 * 2), i64, vp, vp]
        L.mapf_expand_range.argtypes = [vp, C.POINTER(u64 * 2), i64, vp, vp, vp, vp, vp, vp]
        L.mapf_checksum.argtypes = [vp, i64, i64, vp, vp, vp, vp, vp, vp]
        L.mapf_step.argtypes = [vp, vp, vp, i64, vp, u64, u64, i64, u32, vp, vp, vp, vp, vp, vp]
        L.mapf_rollout.argtypes = [vp, vp, vp, i64, i64, vp, u64, u64, i64, u32, vp, vp, vp, vp, vp, vp]
        L.mapf_step_host.argtypes = [vp, vp, vp, i64, vp, u64, u64, i64, u32, vp, vp, vp, vp, vp]
        L.mapf_step_host_resident.argtypes = [vp, vp, vp, i64, vp, u64, u64, i64, u32, vp, vp, vp, vp, vp]
        L.mapf_evaluate_scratch_bytes.argtypes = []
        L.mapf_evaluate_scratch_bytes.restype = i64
        L.mapf_evaluate.argtypes = [vp, i32, vp, i64, i64, i64, C.c_double, u64, u64, i64, vp, vp, vp, vp, vp]
        L.mapf_evaluate_groups.argtypes = [vp, vp, vp, i64, i64, i64, C.c_double, u64, u64, i64, vp, vp, vp, vp, vp, vp]
        vtp = C.POINTER(MapfVtable)
        L.mapf_rtdp_backup.argtypes = [vp, vp, i64, vp, vp, i64, vtp, C.c_double, vp, vp, vp]
        L.mapf_vtable_store.argtypes = [vp, vp, i64, vp, vp, vtp, vp]
        L.mapf_vtable_lookup.argtypes = [vp, vp, i64, vp, vp, i64, vtp, vp, vp, vp]
        L.mapf_evaluate_table.argtypes = [vp, vtp, vp, vp, i64, i64, i64, C.c_double, u64, u64, i64, vp, vp, vp, vp, vp,
                                          vp]
        L.mapf_backup.argtypes = [vp, vp, vp, i64, vp, i64, C.c_double, vp, vp]
        L.mapf_backup_range.argtypes = [vp, C.POINTER(u64 * 2), i64, vp, i64, C.c_double, vp, vp]
        L.mapf_greedy.argtypes = [vp, vp, i64, vp, vp, vp]
        L.mapf_greedy_bcast.argtypes = [vp, vp, i64, i64, C.POINTER(vp), i32, vp, vp]
        L.mapf_count_predecessors.argtypes = [vp, vp, i64, vp, vp]
        L.mapf_predecessors.argtypes = [vp, vp, i64, vp, vp, vp]
        L.mapf_projected_words.argtypes = [vp, i32]
        L.mapf_project_states.argtypes = [vp, vp, i64, vp, i32, vp, vp]
        L.mapf_parse_map_text.argtypes = [C.c_char_p, i64, i32, C.POINTER(i32), C.POINTER(i32), vp, i64]
        L.mapf_parse_scen_text.argtypes = [C.c_char_p, i64, i32, vp, vp, C.POINTER(i32)]
        L.mapf_ctx_create_from_text.argtypes = [C.c_char_p, i64, C.c_char_p, i64, i32, C.c_double, C.c_double, C.c_double,
                                                C.c_double, i32, i32, C.POINTER(vp)]
        L.mapf_ctx_grid.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), vp, vp, vp]
        L.mapf_group_create.argtypes = [C.POINTER(vp), C.POINTER(i64), i32, C.POINTER(vp)]
        L.mapf_group_destroy.argtypes = [vp]
        L.mapf_group_destroy.restype = None
        L.mapf_group_size.argtypes = [vp]
        L.mapf_group_size.restype = i64
        L.mapf_group_step.argtypes = [vp, vp, vp, vp, u64, u64, i64, u32, vp, vp, vp, vp, vp, vp]
        L.mapf_last_error.restype = C.c_char_p
        L.mapf_version.restype = C.c_char_p
        _lib = L
        return _lib


def check(rc):
    if rc != MAPF_OK:
        text = lib().mapf_last_error().decode("utf8", "replace")
        if rc == MAPF_ERR_KEY:
            raise KeyError(text)  # the reference's KeyError for a start/goal on an obstacle (mapf_env.py:369)
        raise NativeError(rc, text)


def _ptr(t):
    """Device (or host) address of a torch tensor / numpy array; None -> NULL."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


class Engine:
    """One immutable device context (mapf_ctx) for one env spec on one CUDA device."""

    def __init__(self, obstacles, n_agents, starts, goals, fail_prob, r_clash, r_goal, r_living, makespan, device=0):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("gym_mapf_b200 needs a CUDA device (B200, sm_100a): there is no CPU fallback")
        obstacles = np.ascontiguousarray(obstacles, dtype=np.uint8)
        start_rc = np.ascontiguousarray(np.array(starts, dtype=np.int32).reshape(-1))
        goal_rc = np.ascontiguousarray(np.array(goals, dtype=np.int32).reshape(-1))
        spec = MapfSpec(obstacles.shape[0], obstacles.shape[1], obstacles.ctypes.data, int(n_agents),
                        start_rc.ctypes.data, goal_rc.ctypes.data, float(fail_prob), float(r_clash), float(r_goal),
                        float(r_living), MAPF_MAKESPAN if makespan else MAPF_SOC)
        self.device_index = torch.device(device).index if not isinstance(device, int) else device
        if self.device_index is None:
            self.device_index = torch.cuda.current_device()
        self.torch_device = torch.device("cuda", self.device_index)
        h = C.c_void_p()
        check(lib().mapf_ctx_create(C.byref(spec), self.device_index, C.byref(h)))
        self._adopt(h)

    @classmethod
    def from_text(cls, map_text, scen_text, n_agents, fail_prob, r_clash, r_goal, r_living, makespan, device=0):
        """Context straight from the CONTENTS of a MovingAI .map and .scen file (bytes or str): the map is parsed on the
        device (mapf_ctx_create_from_text)."""
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("gym_mapf_b200 needs a CUDA device (B200, sm_100a): there is no CPU fallback")
        self = object.__new__(cls)
        self.device_index = torch.device(device).index if not isinstance(device, int) else device
        if self.device_index is None:
            self.device_index = torch.cuda.current_device()
        self.torch_device = torch.device("cuda", self.device_index)
        map_b = map_text.encode("utf8") if isinstance(map_text, str) else bytes(map_text)
        scen_b = scen_text.encode("utf8") if isinstance(scen_text, str) else bytes(scen_text)
        h = C.c_void_p()
        check(lib().mapf_ctx_create_from_text(map_b, len(map_b), scen_b, len(scen_b), int(n_agents), float(fail_prob),
                                              float(r_clash), float(r_goal), float(r_living),
                                              MAPF_MAKESPAN if makespan else MAPF_SOC, self.device_index, C.byref(h)))
        self._adopt(h)
        return self

    def grid(self):
        """(obstacles uint8[H, W], starts, goals) the context was built from (mapf_ctx_grid)."""
        h, w = C.c_int32(), C.c_int32()
        check(lib().mapf_ctx_grid(self._h, C.byref(h), C.byref(w), None, None, None))
        obstacles = np.zeros((h.value, w.value), np.uint8)
        start_rc = np.zeros(2 * self.n, np.int32)
        goal_rc = np.zeros(2 * self.n, np.int32)
        check(lib().mapf_ctx_grid(self._h, None, None, _ptr(obstacles), _ptr(start_rc), _ptr(goal_rc)))
        pairs = lambda a: tuple((int(a[2 * i]), int(a[2 * i + 1])) for i in range(self.n))  # noqa: E731
        return obstacles, pairs(start_rc), pairs(goal_rc)

    def _adopt(self, h):
        self._h = h
        info = MapfInfo()
        check(lib().mapf_ctx_info(self._h, C.byref(info)))
        self.n = info.n_agents
        self.L = info.n_cells
        self.words = info.state_words
        self.moves_in_smem = bool(info.moves_in_smem)
        self.nA = info.n_actions
        self.nS = info.n_states[0] | (info.n_states[1] << 64)
        self.s0 = info.start_state[0] | (info.start_state[1] << 64)
        self.goal_state = info.goal_state[0] | (info.goal_state[1] << 64)
        self.max_row_len = info.max_row_len
        self.sm_count = info.sm_count
        self._moves = None
        self._mapf_step = lib().mapf_step  # hot call: skip the attribute lookups

    def close(self):
        if getattr(self, "_h", None):
            lib().mapf_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass

    # ---- helpers
    def _check_batch(self, states, actions, uniforms=None):
        """Cheap host-side validation of a (states, actions[, uniforms]) batch: wrong dtypes, shapes or devices would
        otherwise be read as garbage by the kernels.  (Value ranges are not checked here -- that would need a device
        synchronisation; the kernels clamp out-of-range states and actions instead of faulting.)"""
        import torch
        B = states.shape[0]
        if states.dtype is not torch.int64 or tuple(states.shape) != self.state_shape(B) or not states.is_contiguous():
            raise ValueError("states must be a contiguous int64 tensor of shape %s" % (self.state_shape(B),))
        if actions.dtype is not torch.int32 or tuple(actions.shape) != (B,) or not actions.is_contiguous():
            raise ValueError("actions must be a contiguous int32 tensor of shape (%d,)" % B)
        if states.device != self.torch_device or actions.device != self.torch_device:
            raise ValueError("states and actions must live on %s" % self.torch_device)
        if uniforms is not None and (uniforms.dtype is not torch.float64 or tuple(uniforms.shape) != (B, self.n)
                                     or not uniforms.is_contiguous() or uniforms.device != self.torch_device):
            raise ValueError("uniforms must be a contiguous float64 tensor of shape (%d, %d) on %s" % (B, self.n, self.torch_device))

    def _check_tensor(self, name, t, dtype, shape=None, optional=False):
        """dtype / shape / device / contiguity of one device tensor handed to the library as a raw pointer."""
        if t is None:
            if optional:
                return
            raise ValueError("%s is required" % name)
        if t.dtype is not dtype or not t.is_contiguous() or t.device != self.torch_device or \
                (shape is not None and tuple(t.shape) != tuple(shape)):
            raise ValueError("%s must be a contiguous %s tensor%s on %s (got %s %s on %s)" % (
                name, dtype, "" if shape is None else " of shape %s" % (tuple(shape),), self.torch_device, t.dtype,
                tuple(t.shape), t.device))

    def _stream(self):
        import torch
        return torch.cuda.current_stream(self.device_index).cuda_stream

    def state_shape(self, B):
        return (B,) if self.words == 1 else (B, 2)

    def new_states(self, B):
        import torch
        return torch.empty(self.state_shape(B), dtype=torch.int64, device=self.torch_device)

    def states_from_ints(self, values):
        """Python ints -> state tensor on the device."""
        import torch
        m = (1 << 64) - 1
        if self.words == 1:
            arr = np.array([int(v) for v in values], dtype=np.uint64).view(np.int64)
        else:
            arr = np.array([[int(v) & m, (int(v) >> 64) & m] for v in values], dtype=np.uint64).view(np.int64)
            arr = arr.reshape(-1, 2)
        return torch.from_numpy(arr).to(self.torch_device)

    def states_to_ints(self, t):
        arr = t.detach().cpu().numpy().view(np.uint64)
        if self.words == 1:
            return [int(x) for x in arr]
        return [int(lo) | (int(hi) << 64) for lo, hi in arr.reshape(-1, 2)]

    # ---- table read-back
    def moves(self):
        """(k[L,5], dest[L,5,3], prob[L,5,3], cells_rc[L,2]) -- single_agent_movements for every (cell, action)."""
        if self._moves is None:
            k = np.zeros((self.L, 5), np.uint8)
            dest = np.zeros((self.L, 5, 3), np.int32)
            prob = np.zeros((self.L, 5, 3), np.float64)
            rc = np.zeros((self.L, 2), np.int32)
            check(lib().mapf_ctx_moves(self._h, _ptr(k), _ptr(dest), _ptr(prob), _ptr(rc)))
            self._moves = (k, dest, prob, rc)
        return self._moves

    # ---- bulk encodings
    def decode(self, states):
        import torch
        B = states.shape[0]
        self._check_tensor("states", states, torch.int64, self.state_shape(B))
        cells = torch.empty((B, self.n), dtype=torch.int32, device=self.torch_device)
        check(lib().mapf_decode_states(self._h, _ptr(states), B, _ptr(cells), self._stream()))
        return cells

    def encode(self, cells):
        import torch
        B = cells.shape[0]
        self._check_tensor("cells", cells, torch.int32, (B, self.n))
        states = self.new_states(B)
        check(lib().mapf_encode_states(self._h, _ptr(cells), B, _ptr(states), self._stream()))
        return states

    # ---- P[s][a] rows
    def _scan(self, row_len):
        import torch
        B = row_len.shape[0]
        row_ptr = torch.empty(B + 1, dtype=torch.int64, device=self.torch_device)
        scratch = torch.empty(int(lib().mapf_scan_scratch_bytes(B)) // 8 + 1, dtype=torch.int64, device=self.torch_device)
        check(lib().mapf_scan_rows(self._h, _ptr(row_len), B, _ptr(row_ptr), _ptr(scratch), self._stream()))
        return row_ptr

    def _scan_buffers(self, B):
        import torch
        row_ptr = torch.empty(B + 1, dtype=torch.int64, device=self.torch_device)
        scratch = torch.empty(int(lib().mapf_scan_scratch_bytes(B)) // 8 + 1, dtype=torch.int64, device=self.torch_device)
        return row_ptr, scratch

    def _alloc_records(self, total):
        import torch
        dev = self.torch_device
        return (self.new_states(total), torch.empty(total, dtype=torch.float64, device=dev),
                torch.empty(total, dtype=torch.float64, device=dev), torch.empty(total, dtype=torch.uint8, device=dev))

    def transitions(self, states, actions):
        """CSR expansion of P[states[b]][actions[b]] -> (row_ptr, next_state, prob, reward, flags), all on device."""
        import torch
        B = states.shape[0]
        self._check_batch(states, actions)
        row_ptr, scratch = self._scan_buffers(B)
        check(lib().mapf_count_scan_rows(self._h, _ptr(states), _ptr(actions), B, None, _ptr(row_ptr),
                                         _ptr(scratch), self._stream()))
        total = int(row_ptr[-1].item())
        ns, prob, reward, flags = self._alloc_records(total)
        check(lib().mapf_expand(self._h, _ptr(states), _ptr(actions), B, _ptr(row_ptr), _ptr(ns), _ptr(prob),
                                _ptr(reward), _ptr(flags), self._stream()))
        return row_ptr, ns, prob, reward, flags

    def table_range(self, s_begin, n_states):
        """The slab [s_begin, s_begin + n_states) x [0, nA) of the full table, rows in (s, a) order."""
        import torch
        sb = (C.c_uint64 * 2)(s_begin & ((1 << 64) - 1), s_begin >> 64)
        B = n_states * self.nA
        row_ptr, scratch = self._scan_buffers(B)
        check(lib().mapf_count_scan_range(self._h, C.byref(sb), n_states, None, _ptr(row_ptr), _ptr(scratch),
                                          self._stream()))
        total = int(row_ptr[-1].item())
        ns, prob, reward, flags = self._alloc_records(total)
        check(lib().mapf_expand_range(self._h, C.byref(sb), n_states, _ptr(row_ptr), _ptr(ns), _ptr(prob), _ptr(reward),
                                      _ptr(flags), self._stream()))
        return row_ptr, ns, prob, reward, flags

    def checksum(self, ns, prob, reward, flags, index_base=0, out=None):
        import torch
        if out is None:
            out = torch.zeros(8, dtype=torch.int64, device=self.torch_device)
        check(lib().mapf_checksum(self._h, prob.shape[0], index_base, _ptr(ns), _ptr(prob), _ptr(reward), _ptr(flags),
                                  _ptr(out), self._stream()))
        return out

    # ---- step / rollout
    def step(self, states, actions, uniforms=None, seed=0, step_index=0, env_offset=0, auto_reset=False, out=None,
             share_sm=False, compact=False):
        """`share_sm`: one resident CTA per SM (MAPF_OPT_SHARE_SM), for env pools that are stepped concurrently on
        separate streams.  `compact` (MAPF_OPT_COMPACT): the result is
        (next_states, reward_code u8[B], prob, flags u8[B]) -- reward = reward_table()[code], flags = done | collision << 1."""
        B = states.shape[0]
        self._check_batch(states, actions, uniforms)
        if compact:
            return self._step_compact(states, actions, uniforms, seed, step_index, env_offset, auto_reset, out, share_sm)
        if out is None:
            import torch
            dev = self.torch_device
            out = (self.new_states(B), torch.empty(B, dtype=torch.float64, device=dev),
                   torch.empty(B, dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.bool, device=dev),
                   torch.empty(B, dtype=torch.bool, device=dev))
        ns, reward, prob, done, coll = out
        rc = self._mapf_step(self._h, states.data_ptr(), actions.data_ptr(), B,
                             None if uniforms is None else uniforms.data_ptr(), seed, step_index, env_offset,
                             (OPT_AUTO_RESET if auto_reset else 0) | (OPT_SHARE_SM if share_sm else 0), ns.data_ptr(),
                             reward.data_ptr(), prob.data_ptr(), done.data_ptr(), coll.data_ptr(), self._stream())
        if rc:
            check(rc)
        return out

    def reward_table(self):
        """f64[64]: every reward a step can return, indexed by the code of the compact result layout."""
        if getattr(self, "_reward_table", None) is None:
            t = np.zeros(64, np.float64)
            check(lib().mapf_ctx_reward_table(self._h, _ptr(t)))
            self._reward_table = t
        return self._reward_table

    def _step_compact(self, states, actions, uniforms, seed, step_index, env_offset, auto_reset, out, share_sm):
        import torch
        B, dev = states.shape[0], self.torch_device
        if out is None:
            out = (self.new_states(B), torch.empty(B, dtype=torch.uint8, device=dev),
                   torch.empty(B, dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.uint8, device=dev))
        ns, code, prob, flags = out
        opts = OPT_COMPACT | (OPT_AUTO_RESET if auto_reset else 0) | (OPT_SHARE_SM if share_sm else 0)
        check(self._mapf_step(self._h, states.data_ptr(), actions.data_ptr(), B,
                              None if uniforms is None else uniforms.data_ptr(), seed, step_index, env_offset, opts,
                              ns.data_ptr(), code.data_ptr(), prob.data_ptr(), flags.data_ptr(), None, self._stream()))
        return out

    def rollout(self, states, actions, T, uniforms=None, seed=0, step_index=0, env_offset=0, auto_reset=True, out=None):
        import torch
        B = states.shape[0]
        dev = self.torch_device
        T = int(T)
        self._check_tensor("states", states, torch.int64, self.state_shape(B))
        self._check_tensor("actions", actions, torch.int32, (T, B), optional=True)
        self._check_tensor("uniforms", uniforms, torch.float64, (T, B, self.n), optional=True)
        if out is None:
            out = (torch.empty((T,) + self.state_shape(B), dtype=torch.int64, device=dev),
                   torch.empty((T, B), dtype=torch.float64, device=dev),
                   torch.empty((T, B), dtype=torch.float64, device=dev),
                   torch.empty((T, B), dtype=torch.bool, device=dev), torch.empty((T, B), dtype=torch.bool, device=dev))
        ns, reward, prob, done, coll = out
        check(lib().mapf_rollout(self._h, _ptr(states), _ptr(actions), T, B, _ptr(uniforms), seed, step_index,
                                 env_offset, OPT_AUTO_RESET if auto_reset else 0, _ptr(ns), _ptr(reward), _ptr(prob),
                                 _ptr(done), _ptr(coll), self._stream()))
        return out

    def step_host(self, states, actions, out, uniforms=None, seed=0, step_index=0, env_offset=0, auto_reset=False,
                  compact=False):
        """Host-buffer step (numpy arrays or pinned CPU tensors in, the five results written into `out`).  `compact`:
        `out` = (next_states, reward_code u8[B], prob, flags u8[B]), 18 instead of 26 bytes per env over the host link."""
        B = actions.shape[0]
        if compact:
            ns, code, prob, flags = out
            check(lib().mapf_step_host(self._h, _ptr(states), _ptr(actions), B, _ptr(uniforms), seed, step_index, env_offset,
                                       OPT_COMPACT | (OPT_AUTO_RESET if auto_reset else 0), _ptr(ns), _ptr(code), _ptr(prob),
                                       _ptr(flags), None))
            return out
        ns, reward, prob, done, coll = out
        check(lib().mapf_step_host(self._h, _ptr(states), _ptr(actions), B, _ptr(uniforms), seed, step_index, env_offset,
                                   OPT_AUTO_RESET if auto_reset else 0, _ptr(ns), _ptr(reward), _ptr(prob), _ptr(done),
                                   _ptr(coll)))
        return out

    def step_host_resident(self, states_dev, actions, out, uniforms=None, seed=0, step_index=0, env_offset=0,
                           auto_reset=False, compact=False):
        """`step_host` for envs whose states stay on the device (the reference's env keeps `self.s`; `step` receives
        only the action): `states_dev` (device tensor) is advanced in place, only `actions` crosses the host link on
        the way in.  `out` as for `step_host`; results are bit-identical to it."""
        import torch
        B = actions.shape[0]
        self._check_tensor("states_dev", states_dev, torch.int64, self.state_shape(B))
        torch.cuda.current_stream(self.device_index).synchronize()  # the call runs on the context's own streams
        opts = (OPT_COMPACT if compact else 0) | (OPT_AUTO_RESET if auto_reset else 0)
        if compact:
            ns, code, prob, flags = out
            check(lib().mapf_step_host_resident(self._h, _ptr(states_dev), _ptr(actions), B, _ptr(uniforms), seed, step_index,
                                                env_offset, opts, _ptr(ns), _ptr(code), _ptr(prob), _ptr(flags), None))
            return out
        ns, reward, prob, done, coll = out
        check(lib().mapf_step_host_resident(self._h, _ptr(states_dev), _ptr(actions), B, _ptr(uniforms), seed, step_index,
                                            env_offset, opts, _ptr(ns), _ptr(reward), _ptr(prob), _ptr(done), _ptr(coll)))
        return out

    # ---- closed-loop policy evaluation -----------------------------------------------------------------------
    def evaluate(self, policy, n_episodes, max_steps, gamma=1.0, seed=0, step_index=0, episode_offset=0, out=None):
        """`n_episodes` episodes from the start state under `policy`, each cut at its first done or after `max_steps`
        steps, in one launch (mapf_evaluate).  Episode e draws what env `episode_offset + e` of `step` draws from
        `step_index` on.  `policy`: None (uniformly random joint actions, as `rollout` draws them), an int32[nS] tensor
        of joint actions indexed by the joint state, or an integer [n_agents, L] tensor of per-agent actions indexed by
        the agent's cell, a `GroupPolicy` (see `evaluate_groups`) or a `TablePolicy` (see `evaluate_table`).  Returns (returns f64[E], lengths i32[E],
        outcomes u8[E]) with outcomes EPISODE_*."""
        import torch
        from .envs.vec_env import GroupPolicy, TablePolicy
        if isinstance(policy, TablePolicy):
            return self.evaluate_table(policy, n_episodes, max_steps, gamma=gamma, seed=seed, step_index=step_index,
                                       episode_offset=episode_offset, out=out)
        if isinstance(policy, GroupPolicy):
            return self.evaluate_groups(policy, n_episodes, max_steps, gamma=gamma, seed=seed, step_index=step_index,
                                        episode_offset=episode_offset, out=out)
        E = int(n_episodes)
        if E < 0:
            raise ValueError("n_episodes must be >= 0 (got %d)" % E)
        if policy is None:
            kind, table, n_entries = POLICY_RANDOM, None, 0
        elif not isinstance(policy, torch.Tensor) or policy.dim() not in (1, 2):
            raise ValueError("policy must be None, an int32[nS] tensor or an integer [n_agents, L] tensor")
        elif policy.dim() == 1:
            self._check_tensor("policy", policy, torch.int32)
            if policy.shape[0] < self.nS:
                raise ValueError("a joint-state policy needs nS = %d entries (got %d)" % (self.nS, policy.shape[0]))
            kind, table, n_entries = POLICY_JOINT, policy, policy.shape[0]
        else:
            if policy.dtype.is_floating_point or policy.dtype.is_complex or policy.dtype is torch.bool or \
                    tuple(policy.shape) != (self.n, self.L) or policy.device != self.torch_device:
                raise ValueError("a per-agent policy must be an integer tensor of shape (%d, %d) on %s (got %s %s on %s)"
                                 % (self.n, self.L, self.torch_device, policy.dtype, tuple(policy.shape), policy.device))
            kind, table, n_entries = POLICY_AGENTS, policy, policy.numel()
        if table is not None and table.numel() > 0:
            hi = self.nA if kind == POLICY_JOINT else 5
            lo_v, hi_v = torch.aminmax(table)
            if int(lo_v) < 0 or int(hi_v) >= hi:
                raise ValueError("policy entries must lie in [0, %d) (got [%d, %d])" % (hi, int(lo_v), int(hi_v)))
        if kind == POLICY_AGENTS:
            table = table.to(torch.uint8).contiguous()
        dev = self.torch_device
        if out is None:
            out = (torch.empty(E, dtype=torch.float64, device=dev), torch.empty(E, dtype=torch.int32, device=dev),
                   torch.empty(E, dtype=torch.uint8, device=dev))
        ret, length, outcome = out
        self._check_tensor("returns", ret, torch.float64, (E,))
        self._check_tensor("lengths", length, torch.int32, (E,))
        self._check_tensor("outcomes", outcome, torch.uint8, (E,))
        scratch = torch.empty((int(lib().mapf_evaluate_scratch_bytes()) + 7) // 8, dtype=torch.int64, device=dev)
        check(lib().mapf_evaluate(self._h, kind, _ptr(table), n_entries, E, int(max_steps), float(gamma), int(seed),
                                  int(step_index), int(episode_offset), _ptr(scratch), _ptr(ret), _ptr(length),
                                  _ptr(outcome), self._stream()))
        return out

    def evaluate_groups(self, policy, n_episodes, max_steps, gamma=1.0, seed=0, step_index=0, episode_offset=0, out=None,
                        conflicts=None):
        """`evaluate` for a `GroupPolicy` (mapf_evaluate_groups): each group of agents acts by its own table, indexed by
        the group's local state.  `conflicts` (u8[E] device tensor, optional) receives, for every episode that ends in a
        collision, the pair i | j << 4 (i < j) of its last step's clash -- agents of different groups first -- and
        NO_CONFLICT for every other episode."""
        import torch
        E = int(n_episodes)
        if E < 0:
            raise ValueError("n_episodes must be >= 0 (got %d)" % E)
        if policy.n_agents != self.n or policy.n_cells != self.L or policy.tables[0].device != self.torch_device:
            raise ValueError("the GroupPolicy is for %d agents on %d cells on %s; this env has %d agents on %d cells on %s"
                             % (policy.n_agents, policy.n_cells, policy.tables[0].device, self.n, self.L,
                                self.torch_device))
        tables = policy.tables[0].contiguous() if len(policy.tables) == 1 else torch.cat(policy.tables)
        group_of = (C.c_int32 * self.n)(*policy.group_of())
        dev = self.torch_device
        if out is None:
            out = (torch.empty(E, dtype=torch.float64, device=dev), torch.empty(E, dtype=torch.int32, device=dev),
                   torch.empty(E, dtype=torch.uint8, device=dev))
        ret, length, outcome = out
        self._check_tensor("returns", ret, torch.float64, (E,))
        self._check_tensor("lengths", length, torch.int32, (E,))
        self._check_tensor("outcomes", outcome, torch.uint8, (E,))
        if conflicts is not None:
            self._check_tensor("conflicts", conflicts, torch.uint8, (E,))
        scratch = torch.empty((int(lib().mapf_evaluate_scratch_bytes()) + 7) // 8, dtype=torch.int64, device=dev)
        check(lib().mapf_evaluate_groups(self._h, group_of, _ptr(tables), tables.numel(), E, int(max_steps),
                                         float(gamma), int(seed), int(step_index), int(episode_offset), _ptr(scratch),
                                         _ptr(ret), _ptr(length), _ptr(outcome), _ptr(conflicts), self._stream()))
        return out

    def evaluate_table(self, policy, n_episodes, max_steps, gamma=1.0, seed=0, step_index=0, episode_offset=0, out=None,
                       conflicts=None):
        """`evaluate_groups` for a `TablePolicy` (mapf_evaluate_table): in a state that is a key of the policy's value
        table an episode takes the action stored with it, anywhere else the fallback GroupPolicy's action.  Same draws,
        outputs and `conflicts` as `evaluate_groups`."""
        import torch
        E = int(n_episodes)
        if E < 0:
            raise ValueError("n_episodes must be >= 0 (got %d)" % E)
        if policy.table.engine is not self:
            raise ValueError("the TablePolicy's value table belongs to another env")
        group_of, tables = self._group_args(policy.fallback.groups, policy.fallback.tables, "fallback GroupPolicy")
        dev = self.torch_device
        if out is None:
            out = (torch.empty(E, dtype=torch.float64, device=dev), torch.empty(E, dtype=torch.int32, device=dev),
                   torch.empty(E, dtype=torch.uint8, device=dev))
        ret, length, outcome = out
        self._check_tensor("returns", ret, torch.float64, (E,))
        self._check_tensor("lengths", length, torch.int32, (E,))
        self._check_tensor("outcomes", outcome, torch.uint8, (E,))
        if conflicts is not None:
            self._check_tensor("conflicts", conflicts, torch.uint8, (E,))
        scratch = torch.empty((int(lib().mapf_evaluate_scratch_bytes()) + 7) // 8, dtype=torch.int64, device=dev)
        check(lib().mapf_evaluate_table(self._h, C.byref(policy.table.c_struct()), group_of, _ptr(tables),
                                        tables.numel(), E, int(max_steps), float(gamma), int(seed), int(step_index),
                                        int(episode_offset), _ptr(scratch), _ptr(ret), _ptr(length), _ptr(outcome),
                                        _ptr(conflicts), self._stream()))
        return out

    # ---- RTDP over a value table (one-word states) -------------------------------------------------------------
    def _group_args(self, groups, tables, what):
        """(group_of as a C array, the per-group tables concatenated) of a GroupPolicy's or GroupValues' tensors."""
        import torch
        n = sum(len(g) for g in groups)
        if n != self.n or any(t.numel() != self.L ** len(g) for g, t in zip(groups, tables)) or \
                tables[0].device != self.torch_device:
            raise ValueError("the %s is for %d agents with tables of %s entries on %s; this env has %d agents on %d cells "
                             "on %s" % (what, n, [t.numel() for t in tables], tables[0].device, self.n, self.L,
                                        self.torch_device))
        group_of = [0] * n
        for gid, g in enumerate(groups):
            for a in g:
                group_of[a] = gid
        flat = tables[0].contiguous() if len(tables) == 1 else torch.cat(tables)
        return (C.c_int32 * n)(*group_of), flat

    def _check_keys(self, states):
        import torch
        if self.words != 1:
            raise ValueError("value tables are keyed by one-word states; this env's states take two words")
        self._check_tensor("states", states, torch.int64, (states.shape[0],))

    def rtdp_backup(self, states, heuristic, table, gamma):
        """(v f64[B], a i32[B]) (mapf_rtdp_backup): v[b] = max over actions of the Bellman backup of states[b], every
        successor valued by `table` when it is a key and by `heuristic` (GroupValues) otherwise; a[b] = the first
        action attaining it.  `table` is only read."""
        import torch
        self._check_keys(states)
        B = states.shape[0]
        group_of, hv = self._group_args(heuristic.groups, heuristic.values, "GroupValues")
        v = torch.empty(B, dtype=torch.float64, device=self.torch_device)
        a = torch.empty(B, dtype=torch.int32, device=self.torch_device)
        check(lib().mapf_rtdp_backup(self._h, _ptr(states), B, group_of, _ptr(hv), hv.numel(),
                                     C.byref(table.c_struct()), float(gamma), _ptr(v), _ptr(a), self._stream()))
        return v, a

    def vtable_store(self, states, v, a, table):
        """Stores (states[b], v[b], a[b]) in `table`, overwriting present keys; the states must be distinct
        (mapf_vtable_store)."""
        import torch
        self._check_keys(states)
        B = states.shape[0]
        self._check_tensor("v", v, torch.float64, (B,))
        self._check_tensor("a", a, torch.int32, (B,))
        check(lib().mapf_vtable_store(self._h, _ptr(states), B, _ptr(v), _ptr(a), C.byref(table.c_struct()),
                                      self._stream()))

    def vtable_lookup(self, states, heuristic, table):
        """(value_of(states) f64[B], the stored action or -1 i32[B]) (mapf_vtable_lookup)."""
        import torch
        self._check_keys(states)
        B = states.shape[0]
        group_of, hv = self._group_args(heuristic.groups, heuristic.values, "GroupValues")
        v = torch.empty(B, dtype=torch.float64, device=self.torch_device)
        a = torch.empty(B, dtype=torch.int32, device=self.torch_device)
        check(lib().mapf_vtable_lookup(self._h, _ptr(states), B, group_of, _ptr(hv), hv.numel(),
                                       C.byref(table.c_struct()), _ptr(v), _ptr(a), self._stream()))
        return v, a

    # ---- rows next to the hot path (SURVEY.md 8f) ----------------------------------------------------------
    def backup(self, states, actions, V, gamma, out=None):
        """Q[b] = sum over P[states[b]][actions[b]], in order, of p * (r + gamma * V[s2]) -- no table is written."""
        import torch
        B = states.shape[0]
        self._check_batch(states, actions)
        self._check_tensor("V", V, torch.float64, (V.shape[0],))
        Q = out if out is not None else torch.empty(B, dtype=torch.float64, device=self.torch_device)
        self._check_tensor("Q", Q, torch.float64, (B,))
        check(lib().mapf_backup(self._h, _ptr(states), _ptr(actions), B, _ptr(V), V.shape[0], float(gamma), _ptr(Q),
                                self._stream()))
        return Q

    def backup_range(self, s_begin, n_states, V, gamma, out=None):
        """The same for the slab [s_begin, s_begin + n_states) x all actions: Q[n_states, nA]."""
        import torch
        sb = (C.c_uint64 * 2)(s_begin & ((1 << 64) - 1), s_begin >> 64)
        self._check_tensor("V", V, torch.float64, (V.shape[0],))
        Q = out if out is not None else torch.empty((n_states, self.nA), dtype=torch.float64, device=self.torch_device)
        self._check_tensor("Q", Q, torch.float64, (n_states, self.nA))
        check(lib().mapf_backup_range(self._h, C.byref(sb), n_states, _ptr(V), V.shape[0], float(gamma), _ptr(Q),
                                      self._stream()))
        return Q

    def greedy(self, Q):
        """(max over actions, first argmax) of a Q[n_states, nA] slab."""
        import torch
        n_states = Q.shape[0]
        V = torch.empty(n_states, dtype=torch.float64, device=self.torch_device)
        pi = torch.empty(n_states, dtype=torch.int32, device=self.torch_device)
        check(lib().mapf_greedy(self._h, _ptr(Q), n_states, _ptr(V), _ptr(pi), self._stream()))
        return V, pi

    def greedy_bcast(self, Q, s_begin, peer_ptrs):
        """Greedy step of a SHARDED sweep with the exchange fused in: V of state s_begin + i goes straight into every
        rank's value vector (`peer_ptrs`: device addresses of all ranks' vectors, e.g. a symmetric-memory handle's
        buffer_ptrs).  Returns the policy of the shard."""
        import torch
        n_states = Q.shape[0]
        pi = torch.empty(n_states, dtype=torch.int32, device=self.torch_device)
        arr = (C.c_void_p * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        check(lib().mapf_greedy_bcast(self._h, _ptr(Q), n_states, int(s_begin), arr, len(peer_ptrs), _ptr(pi),
                                      self._stream()))
        return pi

    def predecessors(self, states):
        """CSR (row_ptr, pred_states) of MapfEnv.predecessors for every state."""
        import torch
        B = states.shape[0]
        self._check_tensor("states", states, torch.int64, self.state_shape(B))
        row_len = torch.empty(B, dtype=torch.int64, device=self.torch_device)
        check(lib().mapf_count_predecessors(self._h, _ptr(states), B, _ptr(row_len), self._stream()))
        row_ptr = self._scan(row_len)
        pred = self.new_states(int(row_ptr[-1].item()))
        check(lib().mapf_predecessors(self._h, _ptr(states), B, _ptr(row_ptr), _ptr(pred), self._stream()))
        return row_ptr, pred

    def project(self, states, agents):
        """The states as the sub-env of `agents` (get_local_view) numbers them: int64[B] or int64[B, 2]."""
        import torch
        B = states.shape[0]
        self._check_tensor("states", states, torch.int64, self.state_shape(B))
        agents = np.ascontiguousarray(agents, dtype=np.int32)
        words = lib().mapf_projected_words(self._h, len(agents))
        if words < 0:
            check(words)
        out = torch.empty((B,) if words == 1 else (B, 2), dtype=torch.int64, device=self.torch_device)
        check(lib().mapf_project_states(self._h, _ptr(states), B, _ptr(agents), len(agents), _ptr(out), self._stream()))
        return out


def parse_map_text(map_text, device=0):
    """uint8[H, W] obstacle mask (1 = '@') of a MovingAI .map file's CONTENTS, parsed on the device
    (mapf_parse_map_text; reference utils.py:33-37 + grid.py:17-25).  KeyError for an unknown cell character."""
    data = map_text.encode("utf8") if isinstance(map_text, str) else bytes(map_text)
    h, w = C.c_int32(), C.c_int32()
    out = np.zeros(max(1, len(data)), np.uint8)
    check(lib().mapf_parse_map_text(data, len(data), int(device), C.byref(h), C.byref(w), _ptr(out), out.size))
    return out[:h.value * w.value].reshape(h.value, w.value).copy()


def parse_scen_text(scen_text, n_agents):
    """(starts, goals) of a .scen file's CONTENTS by the library's host parser (mapf_parse_scen_text; reference
    utils.py:8-30).  Needs no GPU."""
    data = scen_text.encode("utf8") if isinstance(scen_text, str) else bytes(scen_text)
    n_agents = int(n_agents)
    start_rc = np.zeros(2 * max(1, n_agents), np.int32)
    goal_rc = np.zeros(2 * max(1, n_agents), np.int32)
    found = C.c_int32()
    check(lib().mapf_parse_scen_text(data, len(data), n_agents, _ptr(start_rc), _ptr(goal_rc), C.byref(found)))
    pairs = lambda a: tuple((int(a[2 * i]), int(a[2 * i + 1])) for i in range(found.value))  # noqa: E731
    return pairs(start_rc), pairs(goal_rc)


class Group:
    """A heterogeneous env batch (mapf_group): counts[i] envs of engines[i], concatenated; one launch steps them all."""

    def __init__(self, engines, counts):
        if len(engines) != len(counts) or not engines:
            raise ValueError("one env count per engine")
        self.engines = list(engines)
        self.counts = [int(c) for c in counts]
        self.n, self.words = engines[0].n, engines[0].words
        self.torch_device = engines[0].torch_device
        self.device_index = engines[0].device_index
        arr = (C.c_void_p * len(engines))(*[e._h for e in engines])
        cnt = (C.c_int64 * len(counts))(*self.counts)
        h = C.c_void_p()
        check(lib().mapf_group_create(arr, cnt, len(engines), C.byref(h)))
        self._h = h
        self.size = int(lib().mapf_group_size(self._h))

    def close(self):
        if getattr(self, "_h", None):
            lib().mapf_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass

    def step(self, states, actions, uniforms=None, seed=0, step_index=0, env_offset=0, auto_reset=False, out=None):
        import torch
        B, dev = self.size, self.torch_device
        shape = (B,) if self.words == 1 else (B, 2)
        if states.dtype is not torch.int64 or tuple(states.shape) != shape or not states.is_contiguous() or states.device != dev:
            raise ValueError("states must be a contiguous int64 tensor of shape %s on %s" % (shape, dev))
        if actions.dtype is not torch.int32 or tuple(actions.shape) != (B,) or not actions.is_contiguous() or actions.device != dev:
            raise ValueError("actions must be a contiguous int32 tensor of shape (%d,) on %s" % (B, dev))
        if uniforms is not None and (uniforms.dtype is not torch.float64 or tuple(uniforms.shape) != (B, self.n)
                                     or not uniforms.is_contiguous() or uniforms.device != dev):
            raise ValueError("uniforms must be a contiguous float64 tensor of shape (%d, %d) on %s" % (B, self.n, dev))
        if out is None:
            out = (torch.empty(shape, dtype=torch.int64, device=dev), torch.empty(B, dtype=torch.float64, device=dev),
                   torch.empty(B, dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.bool, device=dev),
                   torch.empty(B, dtype=torch.bool, device=dev))
        ns, reward, prob, done, coll = out
        check(lib().mapf_group_step(self._h, _ptr(states), _ptr(actions), _ptr(uniforms), seed, step_index, env_offset,
                                    OPT_AUTO_RESET if auto_reset else 0, _ptr(ns), _ptr(reward), _ptr(prob), _ptr(done),
                                    _ptr(coll), torch.cuda.current_stream(self.device_index).cuda_stream))
        return out
