"""ctypes binding of include/gcrl_b200.h (the drop-in C ABI)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libgcrl_b200.so"


def library_path() -> str:
    return os.environ.get("GCRL_B200_LIB", os.path.join(_HERE, _LIB_NAME))


class GcrlError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"gcrl_b200 error {code}: {msg}")
        self.code = code


OK, ERR_INVALID, ERR_UNDERFILLED, ERR_CUDA, ERR_CAPACITY = 0, 1, 2, 3, 4
HER_FUTURE, HER_FINAL, HER_EPISODE = 0, 1, 2          # GCRL_HER_* goal-selection strategies

c_i32, c_i64, c_u64, c_f32, c_f64 = C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_double
vp = C.c_void_p
pp = C.POINTER(C.c_void_p)


class AgentConfig(C.Structure):
    """struct gcrl_agent_config (include/gcrl_b200.h)."""
    _fields_ = [("algo", c_i32), ("state_dim", c_i32), ("act_dim", c_i32), ("hidden_dim", c_i32),
                ("layer_count", c_i32), ("max_batch", c_i32), ("gamma", c_f32), ("tau", c_f32),
                ("grad_clip", c_f32), ("policy_noise", c_f32), ("noise_clamp", c_f32),
                ("weight_decay", c_f32), ("precision", c_i32), ("reserved", c_i32)]


class SacConfig(C.Structure):
    """struct gcrl_sac_config (include/gcrl_b200.h)."""
    _fields_ = [("algo", c_i32), ("state_dim", c_i32), ("act_dim", c_i32), ("hidden_dim", c_i32),
                ("layer_count", c_i32), ("max_batch", c_i32), ("n_critics", c_i32), ("drop_top", c_i32),
                ("gamma", c_f32), ("tau", c_f32), ("grad_clip", c_f32), ("weight_decay", c_f32),
                ("entropy_coef", c_f32), ("target_entropy", c_f32), ("alpha_lr", c_f32), ("precision", c_i32)]


# name -> (restype, argtypes); every symbol include/gcrl_b200.h declares
SIGNATURES = {
    "gcrl_abi_version": (C.c_int, []),
    "gcrl_last_error": (C.c_char_p, []),
    "gcrl_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "gcrl_kernel_launches": (c_u64, []),
    # HER buffer
    "gcrl_her_create": (C.c_int, [pp, C.c_int, c_i64, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, c_u64]),
    "gcrl_her_destroy": (C.c_int, [vp]),
    "gcrl_her_push_episode": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_her_set_threshold": (C.c_int, [vp, C.c_float]),
    "gcrl_her_set_goal_selection": (C.c_int, [vp, C.c_int, C.c_int]),
    "gcrl_her_set_n_step": (C.c_int, [vp, C.c_int, C.c_float]),
    "gcrl_her_get_draw_epoch": (c_u64, [vp]),
    "gcrl_her_set_draw_epoch": (C.c_int, [vp, c_u64]),
    "gcrl_her_index_tables": (C.c_int, [vp, pp, C.POINTER(c_i64), pp, C.POINTER(c_i64)]),
    "gcrl_her_len": (c_i64, [vp]),
    "gcrl_her_total_entries": (c_i64, [vp]),
    "gcrl_her_live_transitions": (c_i64, [vp]),
    "gcrl_her_clear": (C.c_int, [vp]),
    "gcrl_her_live_episodes": (c_i64, [vp]),
    "gcrl_her_get_episode": (C.c_int, [vp, c_i64, C.POINTER(C.c_int), vp, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_her_sample": (C.c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_her_sample_dev_idx": (C.c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_her_sample_host": (C.c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_pyrandom_randint": (C.c_int, [vp, C.POINTER(C.c_int), c_i64, vp, vp, vp]),
    "gcrl_pyrandom_sample_range": (C.c_int, [vp, C.POINTER(C.c_int), c_i64, c_i64, vp]),
    # normaliser
    "gcrl_norm_create": (C.c_int, [pp, C.c_int, C.c_int, c_f64, c_f64]),
    "gcrl_norm_destroy": (C.c_int, [vp]),
    "gcrl_norm_update": (C.c_int, [vp, vp, c_i64, C.c_int, vp]),
    "gcrl_norm_update_dev": (C.c_int, [vp, vp, c_i64, C.c_int, vp]),
    "gcrl_norm_batch_moments": (C.c_int, [vp, vp, c_i64, C.c_int, vp, vp]),
    "gcrl_norm_update_moments": (C.c_int, [vp, vp, C.c_int, vp]),
    "gcrl_norm_apply": (C.c_int, [vp, vp, c_i64, C.c_int, vp, vp]),
    "gcrl_norm_apply_dev_f32": (C.c_int, [vp, vp, c_i64, C.c_int, vp, c_i64, c_i64, vp]),
    "gcrl_norm_get_state": (C.c_int, [vp, vp, vp, C.POINTER(c_f64), C.POINTER(c_f64), vp]),
    "gcrl_norm_set_state": (C.c_int, [vp, vp, vp, c_f64, c_f64, vp]),
    # agents
    "gcrl_agent_create": (C.c_int, [pp, C.c_int, C.POINTER(AgentConfig)]),
    "gcrl_agent_destroy": (C.c_int, [vp]),
    "gcrl_agent_num_layers": (C.c_int, [vp, C.c_int]),
    "gcrl_agent_layer_shape": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "gcrl_agent_set_layer": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp]),
    "gcrl_agent_get_layer": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp]),
    "gcrl_agent_get_adam_layer": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp]),
    "gcrl_agent_set_adam_layer": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp]),
    "gcrl_agent_get_adam_step": (C.c_int, [vp, C.c_int, C.POINTER(C.c_int)]),
    "gcrl_agent_set_adam_step": (C.c_int, [vp, C.c_int, C.c_int]),
    "gcrl_agent_hard_update": (C.c_int, [vp, vp]),
    "gcrl_agent_soft_update": (C.c_int, [vp, C.c_int, c_f64, vp]),
    "gcrl_agent_reset_optim": (C.c_int, [vp, vp]),
    "gcrl_agent_update_batch": (C.c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp, c_f64, c_f64, C.c_int, vp, vp]),
    "gcrl_agent_update_from_buffer": (C.c_int, [vp, vp, c_i64, vp, vp, c_f64, c_f64, C.c_int, vp, vp]),
    "gcrl_agent_update_many": (C.c_int, [vp, vp, c_i64, C.c_int, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_agent_update_many_replay": (C.c_int, [vp, vp, c_i64, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_agent_read_metrics": (C.c_int, [vp, vp, vp]),
    "gcrl_agent_act": (C.c_int, [vp, c_i64, vp, vp, vp]),
    "gcrl_agent_q": (C.c_int, [vp, c_i64, vp, vp, vp, vp]),
    "gcrl_agent_update_phase": (C.c_int, [vp, C.c_int, vp, c_i64, vp, vp, vp, vp, vp, vp, vp, c_f64, c_f64,
                                         C.c_int, vp]),
    "gcrl_agent_dp_export": (C.c_int, [vp, vp, C.POINTER(C.c_int)]),
    "gcrl_agent_dp_connect": (C.c_int, [vp, C.c_int, C.c_int, vp]),
    "gcrl_agent_dp_barrier": (C.c_int, [vp, vp]),
    "gcrl_agent_grad_buffer": (C.c_int, [vp, C.c_int, pp, C.POINTER(c_i64)]),
    "gcrl_agent_metrics_buffer": (C.c_int, [vp, pp]),
    "gcrl_agent_param_buffers": (C.c_int, [vp, C.c_int, pp, C.POINTER(c_i64), pp, C.POINTER(c_i64)]),
    # SAC / TQC
    "gcrl_sac_create": (C.c_int, [pp, C.c_int, C.POINTER(SacConfig)]),
    "gcrl_sac_create_quantile": (C.c_int, [pp, C.c_int, C.POINTER(SacConfig), C.c_int, C.c_int]),
    "gcrl_sac_destroy": (C.c_int, [vp]),
    "gcrl_sac_set_actor_linear": (C.c_int, [vp, C.c_int, vp, vp, vp]),
    "gcrl_sac_get_actor_linear": (C.c_int, [vp, C.c_int, vp, vp, vp]),
    "gcrl_sac_set_actor_bn": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp]),
    "gcrl_sac_get_actor_bn": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp]),
    "gcrl_sac_set_critic_layer": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "gcrl_sac_get_critic_layer": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "gcrl_sac_hard_update": (C.c_int, [vp, vp]),
    "gcrl_sac_set_log_alpha": (C.c_int, [vp, c_f32, vp]),
    "gcrl_sac_get_log_alpha": (C.c_int, [vp, C.POINTER(c_f32), vp]),
    "gcrl_sac_update_batch": (C.c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp, vp, c_f64, c_f64, C.c_int, vp, vp]),
    "gcrl_sac_update_from_buffer": (C.c_int, [vp, vp, c_i64, vp, vp, vp, c_f64, c_f64, C.c_int, vp, vp]),
    "gcrl_sac_update_many": (C.c_int, [vp, vp, c_i64, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_sac_update_many_replay": (C.c_int, [vp, vp, c_i64, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_sac_act": (C.c_int, [vp, c_i64, vp, vp, vp, vp]),
    "gcrl_sac_update_phase": (C.c_int, [vp, C.c_int, vp, c_i64, vp, vp, vp, vp, vp, vp, vp, vp, c_f64, c_f64, C.c_int,
                                        vp]),
    "gcrl_sac_set_sync_bn": (C.c_int, [vp, C.c_int, C.c_int]),
    "gcrl_sac_update_segment": (C.c_int, [vp, C.c_int, vp, c_i64, vp, vp, vp, vp, vp, vp, vp, vp, c_f64, c_f64, C.c_int,
                                          C.POINTER(C.c_int), vp]),
    "gcrl_sac_dp_buffer": (C.c_int, [vp, C.c_int, pp, C.POINTER(c_i64)]),
    "gcrl_sac_read_metrics": (C.c_int, [vp, C.c_int, vp, vp]),
    # uniform / prioritised replay
    "gcrl_replay_create": (C.c_int, [pp, C.c_int, c_i64, C.c_int, C.c_int, C.c_int, c_f64]),
    "gcrl_replay_destroy": (C.c_int, [vp]),
    "gcrl_replay_push": (C.c_int, [vp, c_i64, vp, vp]),
    "gcrl_replay_len": (c_i64, [vp]),
    "gcrl_replay_total": (c_i64, [vp]),
    "gcrl_replay_sample": (C.c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_replay_sample_prioritized": (C.c_int, [vp, c_i64, vp, c_f64, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gcrl_replay_update_priorities": (C.c_int, [vp, c_i64, vp, vp, vp]),
    "gcrl_replay_get_priorities": (C.c_int, [vp, vp, vp]),
    "gcrl_replay_set_priorities": (C.c_int, [vp, vp, c_i64, vp]),
    "gcrl_replay_get_rows": (C.c_int, [vp, c_i64, c_i64, vp, vp]),
    "gcrl_replay_last_sample_info": (C.c_int, [vp, C.POINTER(c_f32), C.POINTER(C.c_int), vp]),
    "gcrl_replay_last_positions": (C.c_int, [vp, c_i64, vp, vp]),
    "gcrl_replay_last_tables": (C.c_int, [vp, vp, vp, vp]),
    "gcrl_agent_per_buffers": (C.c_int, [vp, pp, pp]),
    "gcrl_sac_per_buffers": (C.c_int, [vp, pp, pp]),
    # diagnostics
    "gcrl_agent_time_critic_kernel": (C.c_int, [vp, c_i64, C.c_int, C.POINTER(c_f32), vp]),
    "gcrl_split_tf32": (C.c_int, [C.c_int, vp, vp, vp, c_i64, vp]),
    "gcrl_dense_layer_presplit": (C.c_int, [C.c_int, C.c_int, c_i64, C.c_int, C.c_int, vp, C.c_int, vp, vp, C.c_int, vp, vp,
                                            C.c_int, vp, C.c_int, vp]),
    "gcrl_dense_layer_ensemble": (C.c_int, [C.c_int, C.c_int, C.c_int, c_i64, C.c_int, C.c_int, pp, C.c_int, pp, pp,
                                            C.c_int, pp, pp, C.c_int, pp, C.c_int, vp]),
    "gcrl_dense_wgrad": (C.c_int, [C.c_int, C.c_int, c_i64, C.c_int, C.c_int, vp, C.c_int, vp, C.c_int, vp, C.c_int, c_i64,
                                   vp, c_i64, C.c_int, C.POINTER(C.c_int), vp]),
    "gcrl_dense_layer": (C.c_int, [C.c_int, C.c_int, C.c_int, c_i64, C.c_int, C.c_int, vp, C.c_int, vp, C.c_int, vp,
                                   vp, C.c_int, vp, C.c_int, vp]),
    "gcrl_quantile_critic_loss": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, c_i64, vp, vp, C.c_int, c_i64, vp, vp,
                                            vp, vp, c_f32, c_f32, vp, vp, C.c_int, vp, vp, vp, vp, vp]),
}


def _load():
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: the CUDA extension is not built. Run ./build.sh (or "
            "`python -c 'import __graft_entry__ as g; g.build()'`) -- there is no CPU fallback.")
    dll = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(dll, name)          # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if dll.gcrl_abi_version() != 5:
        raise ImportError("libgcrl_b200.so ABI version mismatch")
    return dll


lib = _load()


def check(code):
    if code != OK:
        msg = lib.gcrl_last_error().decode("utf-8", "replace")
        if code == ERR_UNDERFILLED:
            raise AssertionError(msg)          # reference: assert at src/buffer.py:122
        if code == ERR_INVALID:
            raise ValueError(msg)
        raise GcrlError(code, msg)


def device_count() -> int:
    n = C.c_int(0)
    check(lib.gcrl_device_count(C.byref(n)))
    return n.value


def require_cuda():
    if device_count() < 1:
        raise GcrlError(ERR_CUDA, "no CUDA device: gcrl_b200 has no CPU fallback")


def np_ptr(arr):
    return vp(arr.ctypes.data)      # the caller keeps `arr` alive for the duration of the call


def current_stream(device_index):
    import torch
    return vp(torch.cuda.current_stream(device_index).cuda_stream)


# -- CPython `random` mirror (csrc/pyrandom.cu): exact draws from the interpreter's global stream ------------
# The generator words of the last state tuple this module produced, kept as a uint32 array: converting a
# random.getstate() tuple (625 Python ints) costs ~55 us, recognising one we made ourselves ~10 us (by value)
# or nothing (same object).  The array is advanced in place by the C mirror, so the cache is dropped before
# every call and re-armed with the tuple of the new state afterwards.
_mt_cache = None      # (state tuple, its 624 words as uint32 array, pos)


def _words_of(state):
    """(uint32[624] array -- owned by the caller from here on, pos, gauss) for a random.getstate() tuple."""
    import numpy as np
    global _mt_cache
    cached, _mt_cache = _mt_cache, None
    if cached is not None and (cached[0] is state or cached[0] == state):
        return cached[1], C.c_int(cached[2]), state[2]
    version, internal, gauss = state
    if version != 3 or len(internal) != 625:
        raise RuntimeError("unexpected random.getstate() layout")
    return np.array(internal[:-1], dtype=np.uint32), C.c_int(internal[-1]), gauss


def _state_of(mt, pos, gauss):
    """The random.setstate() tuple of advanced words; remembers the pair."""
    global _mt_cache
    words = mt.tolist()
    words.append(pos.value)
    state = (3, tuple(words), gauss)
    _mt_cache = (state, mt, pos.value)
    return state


# Direct view of the interpreter's global generator.  random._inst is a _random.Random (CPython: PyObject_HEAD, then
# `int index; uint32_t state[624];`, Modules/_randommodule.c), so the C mirror can advance the very words the
# interpreter draws from, in place: no getstate() (625 Python ints, ~18 us), no tuple of the advanced state (~20 us),
# no setstate() (~5 us) per call.  The layout is VERIFIED against getstate() on a scratch generator and on the global
# one before it is trusted (and re-checked whenever random._inst is replaced); any mismatch falls back to the
# state-tuple path below.  The two entry points run through a PyDLL handle: the GIL stays held while the words move.
_direct = None        # None: not probed yet; False: layout check failed; else (instance, address)
_pydll = None


def _probe_direct():
    import random
    global _direct, _pydll
    try:
        def view(inst):
            addr = id(inst)
            index = C.c_int.from_address(addr + 16).value
            words = (C.c_uint32 * 624).from_address(addr + 20)
            return index, tuple(words)

        scratch = random.Random(0x5EED1234)
        for inst, draws in ((scratch, 700), (random._inst, 0)):      # the global generator is only LOOKED at
            for step in range(3):
                for _ in range(draws if step else 0):
                    inst.random()                                     # across a 624-word refill on the scratch one
                version, internal, _g = inst.getstate()
                index, words = view(inst)
                if version != 3 or len(internal) != 625 or internal[-1] != index or internal[:-1] != words:
                    raise RuntimeError("layout mismatch")
        if _pydll is None:
            _pydll = C.PyDLL(library_path())
            for name in ("gcrl_pyrandom_randint", "gcrl_pyrandom_sample_range"):
                fn = getattr(_pydll, name)
                fn.restype, fn.argtypes = SIGNATURES[name]
        _direct = (random._inst, id(random._inst))
    except Exception:   # noqa: BLE001  (another interpreter / layout: the portable path is always correct)
        _direct = False


def _direct_ptrs():
    """(words pointer, index pointer) into the interpreter's global generator, or None."""
    import random
    if os.environ.get("GCRL_PYRANDOM_PORTABLE") == "1":
        return None
    if _direct is None or (_direct and _direct[0] is not random._inst):
        _probe_direct()
    if not _direct:
        return None
    addr = _direct[1]
    return vp(addr + 20), C.cast(addr + 16, C.POINTER(C.c_int))


def py_randint_seq(lo, hi):
    """[random.randint(lo[i], hi[i]) for i in range(len(lo))], consuming the global stream identically."""
    import random

    import numpy as np
    lo = np.ascontiguousarray(lo, np.int32)
    hi = np.ascontiguousarray(hi, np.int32)
    out = np.empty(lo.shape, np.int32)
    ptrs = _direct_ptrs()
    if ptrs is not None:
        check(_pydll.gcrl_pyrandom_randint(ptrs[0], ptrs[1], lo.size, np_ptr(lo), np_ptr(hi), np_ptr(out)))
        return out
    mt, pos, gauss = _words_of(random.getstate())
    check(lib.gcrl_pyrandom_randint(np_ptr(mt), C.byref(pos), lo.size, np_ptr(lo), np_ptr(hi), np_ptr(out)))
    random.setstate(_state_of(mt, pos, gauss))
    return out


def py_sample_range_from(state, n, k):
    """(positions, state_after) of random.sample(range(n), k) started from ``state`` (a random.getstate()
    tuple); the interpreter's global generator is not touched."""
    import numpy as np
    mt, pos, gauss = _words_of(state)
    out = np.empty(int(k), np.int64)
    check(lib.gcrl_pyrandom_sample_range(np_ptr(mt), C.byref(pos), int(n), int(k), np_ptr(out)))
    return out, _state_of(mt, pos, gauss)


def py_sample_range(n, k):
    """np.array(random.sample(range(n), k), int64), consuming the global stream identically."""
    import random

    import numpy as np
    ptrs = _direct_ptrs()
    if ptrs is not None:
        out = np.empty(int(k), np.int64)
        check(_pydll.gcrl_pyrandom_sample_range(ptrs[0], ptrs[1], int(n), int(k), np_ptr(out)))
        return out
    out, after = py_sample_range_from(random.getstate(), n, k)
    random.setstate(after)
    return out


def direct_stream_available():
    return _direct_ptrs() is not None
