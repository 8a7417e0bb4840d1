"""ctypes binding of libg2048.so (the C ABI declared in include/g2048.h).

The library is the product: there is no Python / PyTorch / CPU fallback anywhere in this
package.  If the shared object is missing the import of this module fails loudly; if no CUDA
device is present every compute call raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import os
import re
import threading
from pathlib import Path

import torch

PKG_ROOT = Path(__file__).resolve().parent.parent  # .../2048-ppo-agent_b200
REPO_ROOT = PKG_ROOT.parent
LIB_PATH = Path(os.environ.get("G2048_LIB", PKG_ROOT / "libg2048.so"))
HEADER_PATH = REPO_ROOT / "include" / "g2048.h"

RNG_ORIGINAL = 0
RNG_PARTITIONABLE = 1
POLICY_RANDOM = 0
POLICY_DRUL = 1
STATUS_MASK = 0x0F
STATUS_DONE = 0x10
STATUS_OVERFLOW = 0x20
OBS_BOOL, OBS_F32, OBS_BF16 = 0, 1, 2
PLAY_STATS_WORDS = 32

if not LIB_PATH.exists():
    raise ImportError(
        f"{LIB_PATH} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()' "
        "or make -C 2048-ppo-agent_b200/csrc).  There is no fallback implementation."
    )

lib = C.CDLL(str(LIB_PATH))

_P = C.c_void_p
_I64 = C.c_int64
_INT = C.c_int
_DBL = C.c_double
_U64 = C.c_uint64
_U32 = C.c_uint32
_FLT = C.c_float

_SIGNATURES = {
    "g2048_version": (_INT, []),
    "g2048_last_error": (C.c_char_p, []),
    "g2048_device_sm_count": (_INT, []),
    "g2048_threefry2x32": (_INT, [_P, _P, _I64, _P, _P]),
    "g2048_chain_advance": (_INT, [_P, _INT, _I64, _P, _P]),
    "g2048_split_keys": (_INT, [_P, _I64, _I64, _I64, _INT, _P, _P]),
    "g2048_env_init": (_INT, [_P, _I64, _I64, _I64, _INT, _P, _P, _P]),
    "g2048_env_step": (_INT, [_P, _P, _P, _P, _I64, _I64, _I64, _INT, _P, _P]),
    "g2048_env_step_draws": (_INT, [_P, _P, _P, _P, _P, _I64, _P, _P]),
    "g2048_act": (_INT, [_INT, _P, _P, _I64, _I64, _I64, _INT, _P, _P, _P]),
    "g2048_play_record_arena_slots": (_I64, [_I64, _I64, _I64]),
    "g2048_play_record": (_INT, [_INT, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "g2048_play_record_compact": (_INT, [_INT, _P, _P, _P, _P, _P, _I64, _I64, _I64, _P, _P, _P, _P, _P, _P, _P]),
    "g2048_pack_samples": (_INT, [_P, _P, _P, _P, _P, _P, _P, _I64, _P, _P, _P]),
    "g2048_gather_samples": (_INT, [_P, _I64, _P, _INT, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "g2048_policy_step_obs": (_INT, [_P, _P, _P, _P, _INT, _INT, _INT, _P, _P, _INT, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P,
                                     _P, _INT, _P, _P, _P]),
    "g2048_replay_envs": (_INT, [_INT, _P, _I64, _I64, _P, _P, _I64, _INT, _P, _P, _P]),
    "g2048_play": (_INT, [_INT, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P]),
    "g2048_play_tables": (_INT, [_INT, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P]),
    "g2048_play_swar": (_INT, [_INT, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P]),
    "g2048_row_table_lookup": (_INT, [_P, _I64, _P, _P, _P]),
    "g2048_playout_values": (_INT, [_INT, _P, _I64, _P, _I64, _I64, _I64, _P, _I64, _INT, _P, _P, _P, _P]),
    "g2048_expectimax_values": (_INT, [_P, _I64, _INT, _P, _FLT, _P, _P, _P]),
    "g2048_td_scratch_bytes": (_I64, []),
    "g2048_td_train": (_INT, [_P, _P, _P, _P, _I64, _P, _FLT, _P, _I64, _INT, _P, _P, _P]),
    "g2048_ntuple_td_scratch_bytes": (_I64, [_I64, _INT, _I64]),
    "g2048_ntuple_td_train": (_INT, [_P, _P, _P, _P, _I64, _P, _INT, _P, _I64, _FLT, _P, _I64, _INT, _P, _P, _P]),
    "g2048_ntuple_tc_scratch_bytes": (_I64, [_I64, _INT, _I64]),
    "g2048_ntuple_tc_train": (_INT, [_P, _P, _P, _P, _I64, _P, _INT, _P, _I64, _P, _P, _FLT, _P, _I64, _INT, _P, _P, _P]),
    "g2048_expectimax_values_ntuple": (_INT, [_P, _I64, _INT, _P, _INT, _P, _I64, _FLT, _P, _P, _P]),
    "g2048_ntuple_staged_td_train": (_INT, [_P, _P, _P, _P, _I64, _P, _INT, _P, _P, _I64, _FLT, _P, _I64, _INT, _P, _P, _P]),
    "g2048_ntuple_staged_tc_train": (_INT, [_P, _P, _P, _P, _I64, _P, _INT, _P, _P, _I64, _P, _P, _FLT, _P, _I64, _INT, _P,
                                            _P, _P]),
    "g2048_expectimax_values_ntuple_staged": (_INT, [_P, _I64, _INT, _P, _INT, _P, _P, _I64, _FLT, _P, _P, _P]),
    "g2048_ntuple_lambda_td_train": (_INT, [_P, _P, _P, _P, _I64, _P, _INT, _P, _P, _I64, _FLT, _FLT, _INT, _P, _P, _P,
                                            _I64, _INT, _P, _P, _P]),
    "g2048_ntuple_lambda_tc_train": (_INT, [_P, _P, _P, _P, _I64, _P, _INT, _P, _P, _I64, _P, _P, _FLT, _FLT, _INT, _P, _P,
                                            _P, _I64, _INT, _P, _P, _P]),
    "g2048_ntuple_carousel_scratch_bytes": (_I64, [_I64, _INT, _INT, _I64, _INT]),
    "g2048_ntuple_carousel_td_train": (_INT, [_P, _P, _P, _P, _I64, _P, _INT, _P, _P, _I64, _FLT, _FLT, _INT, _P, _P, _P,
                                              _P, _P, _I64, _INT, _P, _P, _P]),
    "g2048_ntuple_carousel_tc_train": (_INT, [_P, _P, _P, _P, _I64, _P, _INT, _P, _P, _I64, _P, _P, _FLT, _FLT, _INT, _P,
                                              _P, _P, _P, _P, _I64, _INT, _P, _P, _P]),
    "g2048_play_host":(_INT, [_INT, _U64, _P, _I64, _I64, _I64, _INT, _P, _P, _P, _P]),
    "g2048_play_host_packed": (_INT, [_INT, _U64, _P, _I64, _I64, _I64, _INT, _P, _P]),
    "g2048_play_packed": (_INT, [_INT, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P, _P]),
    "g2048_rollout_steps": (_INT, [_INT, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P]),
    "g2048_rollout_steps_live": (_INT, [_INT, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _INT, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "g2048_policy_step": (_INT, [_P, _P, _P, _P, _INT, _INT, _INT, _P, _P, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P, _P]),
    "g2048_policy_step_at": (_INT, [_P, _P, _P, _P, _INT, _INT, _INT, _P, _P, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P, _P]),
    "g2048_counter_add": (_INT, [_P, _INT, _P]),
    "g2048_policy_step_live": (_INT, [_P, _P, _P, _P, _INT, _INT, _INT, _P, _P, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P, _P]),
    "g2048_expand_obs_gather": (_INT, [_P, _P, _I64, _INT, _P, _P]),
    "g2048_sample_logits": (_INT, [_P, _P, _INT, _INT, _P, _I64, _I64, _I64, _INT, _P, _P, _P, _P]),
    "g2048_evaluate_logits": (_INT, [_P, _P, _INT, _P, _I64, _P, _P, _P]),
    "g2048_expand_obs": (_INT, [_P, _I64, _INT, _P, _I64, _I64, _P]),
    "g2048_pack_obs": (_INT, [_P, _INT, _I64, _P, _P]),
    "g2048_unpack_status": (_INT, [_P, _I64, _P, _P, _P]),
    "g2048_unpack_records": (_INT, [_P, _P, _P, _P, _I64, _I64, _P, _P, _P, _P, _P, _P, _P]),
    "g2048_episode_lengths": (_INT, [_P, _I64, _I64, _P, _P]),
    "g2048_exclusive_scan": (_INT, [_P, _I64, _P, _P]),
    "g2048_compact_records": (_INT, [_P, _P, _P, _P, _P, _I64, _I64, _P, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "g2048_first_done_rows": (_INT, [_P, _I64, _I64, _P, _P]),
    "g2048_compact_rows": (_INT, [_P, _I64, _I64, _I64, _P, _P, _I64, _P, _P]),
    "g2048_unpack_flat_meta": (_INT, [_P, _I64, _P, _P, _P, _P]),
    "g2048_gather_minibatch": (_INT, [_P, _I64, _P, _P, _P, _P, _P, _P, _INT, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "g2048_random_subset": (_INT, [_U32, _U32, _I64, _I64, _I64, _P, _P]),
    "g2048_embed_boards": (_INT, [_P, _I64, _P, _P, _INT, _INT, _P, _P]),
    "g2048_embed_boards_bulk": (_INT, [_P, _I64, _P, _P, _INT, _INT, _P, _P]),
    "g2048_embed_boards_plain": (_INT, [_P, _I64, _P, _P, _INT, _INT, _P, _P]),
    "g2048_embed_grad_scratch_bytes": (_I64, [_I64, _INT, _INT]),
    "g2048_embed_boards_grad": (_INT, [_P, _I64, _P, _P, _INT, _INT, _P, _P, _P]),
    "g2048_gae_flat_scratch_bytes": (_I64, [_I64]),
    "g2048_gae_flat": (_INT, [_P, _P, _P, _I64, _DBL, _DBL, _P, _P, _P, _P, _P]),
    "g2048_gae_flat_pipelined": (_INT, [_P, _P, _P, _I64, _DBL, _DBL, _P, _P, _P, _P, _P]),
    "g2048_gae_flat_tiled": (_INT, [_P, _P, _P, _I64, _DBL, _DBL, _P, _P, _P, _P, _P]),
    "g2048_gae_scan_scratch_bytes": (_I64, [_I64]),
    "g2048_gae_flat_scan": (_INT, [_P, _P, _P, _I64, _DBL, _DBL, _P, _P, _P, _P, _P]),
    "g2048_gae_time_major": (_INT, [_P, _P, _P, _I64, _I64, _P, _DBL, _DBL, _P, _P, _P, _P]),
    "g2048_normalize": (_INT, [_P, _I64, _P, _INT, _P]),
    "g2048_gae_host": (_INT, [_P, _P, _P, _I64, _DBL, _DBL, _INT, _P, _P]),
    "g2048_release_host_workspace": (_INT, []),
    "g2048_row_moments": (_INT, [_P, _I64, _I64, _P, _P]),
    "g2048_int_peak_probe": (_INT, [_INT, _INT, _INT, _P, _P]),
}

for _name, (_res, _args) in _SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = the .so is stale / incomplete
    _fn.restype = _res
    _fn.argtypes = _args


_extra_entry_points = {}  # name -> ctypes function of another library (tests register their legacy build here)


def register_entry_points(path, signatures: dict) -> None:
    """Make `call(name, ...)` reach entry points of ANOTHER shared library with this one's conventions -- test
    infrastructure: tests/legacy/libg2048_legacy.so carries the first-generation kernels the product library no longer
    exports."""
    other = C.CDLL(str(path))
    for name, (res, args) in signatures.items():
        fn = getattr(other, name)
        fn.restype = res
        fn.argtypes = args
        _extra_entry_points[name] = fn


LEGACY_SIGNATURES = {  # tests/legacy/g2048_legacy.h
    "g2048_play_v1": (_INT, [_INT, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P, _P, _P, _P]),
    "g2048_expand_obs_v1": (_INT, [_P, _I64, _INT, _P, _I64, _I64, _P]),
    "g2048_gae_flat_v1": (_INT, [_P, _P, _P, _I64, _DBL, _DBL, _P, _P, _P, _P, _P]),
}


def declared_symbols() -> list[str]:
    """Entry points declared in include/g2048.h (used by the CPU-side export test)."""
    text = HEADER_PATH.read_text()
    return sorted(set(re.findall(r"\b(g2048_[a-z0-9_]+)\s*\(", text)))


def last_error() -> str:
    return lib.g2048_last_error().decode()


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")


def require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("g2048 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


# The GPU a call runs on is the GPU its tensors live on, not whatever device happens to be current: ptr() notes the
# device of every CUDA tensor handed to the call being assembled, stream_ptr() returns THAT device's current stream,
# and call() makes the device current around the C entry point (which launches on the current device and keys its
# per-device caches -- SM count, function attributes, host workspaces -- off cudaGetDevice).  So
# BatchRunner(device="cuda:1") works in a process whose current device is 0.
_call_ctx = threading.local()


def ptr(t: torch.Tensor | None) -> int | None:
    """Device (or host) pointer of a contiguous tensor, None passes NULL."""
    if t is None:
        return None
    if not t.is_contiguous():
        raise ValueError("g2048 kernels need contiguous tensors")
    if t.is_cuda:
        seen = getattr(_call_ctx, "device", None)
        if seen is None:
            _call_ctx.device = t.device.index
        elif seen != t.device.index:
            _call_ctx.device = None
            raise ValueError(f"one g2048 call got tensors on cuda:{seen} and cuda:{t.device.index}")
    return t.data_ptr()


def stream_ptr() -> int:
    """Current stream of the device the call's tensors live on (of the current device for host-buffer calls)."""
    dev = getattr(_call_ctx, "device", None)
    return torch.cuda.current_stream(dev).cuda_stream


def call(name: str, *args) -> None:
    dev = getattr(_call_ctx, "device", None)
    _call_ctx.device = None
    fn = _extra_entry_points.get(name) or getattr(lib, name)
    if dev is not None and dev != torch.cuda.current_device():
        with torch.cuda.device(dev):
            rc = fn(*args)
    else:
        rc = fn(*args)
    check(rc, name)
