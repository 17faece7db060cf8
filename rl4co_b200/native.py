"""ctypes binding of libcorollout.so (C ABI in include/corollout.h).

This is the *only* compute backend of the package: there is no CPU or PyTorch fallback.
Every wrapper raises if the shared library is missing or a tensor is not a contiguous CUDA
tensor of the exact dtype the ABI declares.  torch is used for device memory and streams
only (``tensor.data_ptr()``, ``torch.cuda.current_stream().cuda_stream``).
"""

from __future__ import annotations

import ctypes
import os
import subprocess
import sys
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_uint64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")
LIB_PATH = os.path.join(_HERE, "libcorollout.so")
SOURCES = ["abi.cu", "env_kernels.cu", "decode_step.cu", "rollout.cu", "rollout_tsp.cu", "rollout_cvrp.cu", "rollout_ms_tsp.cu", "rollout_ms_cvrp.cu", "rollout_sdvrp.cu", "rollout_op.cu", "rollout_pctsp.cu", "gemm_tf32x3.cu",
           "encoder_mha.cu", "encoder_mha_tc.cu", "encoder_mha_tc2.cu", "encoder_mha_tc3.cu",
           "ffn_fused.cu", "data_kernels.cu", "attn_train.cu", "norm_kernels.cu", "op_kernels.cu",
           "two_opt.cu"]
HEADERS = ["co_common.cuh", "rollout_impl.cuh", "rollout_ms_impl.cuh"]

CO_OK = 0
ENV_TSP, ENV_CVRP = 0, 1
ENV_SDVRP = 2
ENV_OP, ENV_PCTSP = 3, 4
ENV_KIND = {"tsp": ENV_TSP, "cvrp": ENV_CVRP, "sdvrp": ENV_SDVRP, "op": ENV_OP, "pctsp": ENV_PCTSP}
#: environments the whole-episode kernel (co_rollout) is instantiated for; others take the stepping kernels
ROLLOUT_ENVS = ("tsp", "cvrp", "sdvrp", "op", "pctsp")
SELECT_GREEDY, SELECT_SAMPLE_NOISE, SELECT_EVALUATE, SELECT_SAMPLE_PHILOX = 0, 1, 2, 3
ROLLOUT_FORCED_START = 1
EMBED_DIM, NUM_HEADS = 128, 8
TWO_OPT_MAX_NODES = 1024  # CO_TWO_OPT_MAX_NODES

EXPORTS = [
    "co_version", "co_last_error_string", "co_device_sm_count", "co_tsp_step", "co_cvrp_action_mask",
    "co_cvrp_step", "co_tour_length", "co_check_tours", "co_pointer_logits", "co_select_action",
    "co_cache_width", "co_rollout_max_nodes", "co_rollout", "co_reward_stats", "co_split_tf32", "co_gemm_tf32x3", "co_encoder_mha",
    "co_ffn_fused", "co_ffn_tile_weights", "co_ffn_tiled_weight_floats", "co_generate_uniform", "co_generate_demand", "co_dihedral8",
    "co_sdvrp_step", "co_sdvrp_action_mask", "co_attn_fwd", "co_attn_bwd", "co_instance_norm", "co_op_step", "co_op_action_mask", "co_op_reward", "co_pctsp_step", "co_pctsp_action_mask",
    "co_tsp_two_opt",
]


class NativeLibraryError(RuntimeError):
    pass


class DecoderWeights(Structure):
    _fields_ = [("project_context_t", c_void_p), ("w_placeholder", c_void_p), ("project_out_t", c_void_p),
                ("dynamic_w", c_void_p), ("dynamic_feature", c_void_p)]


class RolloutArgs(Structure):
    _fields_ = [
        ("env_kind", c_int32), ("select_mode", c_int32), ("B_inst", c_int32), ("num_starts", c_int32),
        ("N", c_int32), ("T_max", c_int32), ("num_loc", c_int32), ("flags", c_int32),
        ("tanh_clipping", c_float), ("temperature", c_float),
        ("cache", c_void_p), ("graph_ctx", c_void_p), ("q_placeholder", c_void_p), ("w_capacity", c_void_p),
        ("locs", c_void_p), ("demand", c_void_p), ("vehicle_capacity", c_void_p),
        ("forced_actions", c_void_p), ("noise", c_void_p), ("seed", c_uint64), ("offset", c_uint64),
        ("actions_out", c_void_p), ("logp_out", c_void_p), ("reward_out", c_void_p), ("loglik_out", c_void_p),
        ("steps_out", c_void_p), ("max_steps_out", c_void_p), ("used_capacity_out", c_void_p),
        ("node_emb", c_void_p), ("w_first", c_void_p), ("cache_width", c_int32), ("reserved0", c_int32),
        ("dyn_w", c_void_p), ("node_limit", c_void_p),
    ]


class AttnArgs(Structure):
    _fields_ = ([(n, c_void_p) for n in ("q", "k", "v", "mask", "o", "lse", "dO", "dq", "dk", "dv")]
                + [(n, c_int32) for n in ("B", "M", "N", "reserved0")]
                + [(n, ctypes.c_int64) for n in ("q_bs", "k_bs", "v_bs", "o_bs", "dq_bs", "dk_bs", "dv_bs")]
                + [(n, c_int32) for n in ("q_rs", "k_rs", "v_rs", "o_rs", "dq_rs", "dk_rs", "dv_rs")]
                + [("scale", c_float)])


NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-I", INCLUDE]


def _nvcc() -> str:
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return nvcc if os.path.exists(nvcc) else "nvcc"


def build(force: bool = False, verbose: bool = False, extra_flags: list[str] | None = None) -> str:
    """Compile libcorollout.so in-tree for sm_100a (nvcc cross-compiles without a GPU).
    Translation units are compiled in parallel, then linked."""
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.join(INCLUDE, "corollout.h")]
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in deps):
        return LIB_PATH
    objdir = os.path.join(_HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + (extra_flags or []) + ["-c", os.path.join(CSRC, s), "-o", obj]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        procs.append((s, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs, log = [], []
    for s, obj, p in procs:
        out, _ = p.communicate()
        log.append(out)
        if p.returncode != 0:
            raise NativeLibraryError(f"nvcc failed on {s} ({p.returncode}):\n{out}")
        objs.append(obj)
    link = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs
    res = subprocess.run(link, capture_output=True, text=True)
    if res.returncode != 0:
        raise NativeLibraryError(f"link failed ({res.returncode}):\n{res.stdout}\n{res.stderr}")
    build.last_log = "\n".join(log)
    return LIB_PATH


_lib = None


def lib() -> ctypes.CDLL:
    """Load (once) and return the shared library; raise loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU/PyTorch fallback for the rollout path)")
    L = ctypes.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(L, name):
            raise NativeLibraryError(f"{LIB_PATH} does not export {name}")
    L.co_last_error_string.restype = c_char_p
    L.co_rollout.argtypes = [POINTER(RolloutArgs), c_void_p]
    L.co_pointer_logits.argtypes = [c_int, POINTER(DecoderWeights)] + [c_void_p] * 12 + [c_int, c_int, c_int, c_int, c_void_p]
    L.co_select_action.argtypes = [c_void_p] * 6 + [c_int, c_float, c_float, c_int, c_uint64, c_uint64, c_int, c_int, c_void_p]
    L.co_tsp_step.argtypes = [c_void_p] * 7 + [c_int, c_int, c_void_p]
    L.co_cvrp_action_mask.argtypes = [c_void_p] * 6 + [c_int, c_int, c_void_p]
    L.co_cvrp_step.argtypes = [c_void_p] * 10 + [c_int, c_int, c_void_p]
    L.co_tour_length.argtypes = [c_void_p] * 3 + [c_int] * 5 + [c_void_p]
    L.co_sdvrp_action_mask.argtypes = [c_void_p] * 5 + [c_int, c_int, c_void_p]
    L.co_sdvrp_step.argtypes = [c_void_p] * 9 + [c_int, c_int, c_void_p]
    L.co_check_tours.argtypes = [c_void_p] * 4 + [c_int] * 4 + [c_void_p]
    L.co_reward_stats.argtypes = [c_void_p, c_void_p, c_int, c_void_p]
    L.co_op_action_mask.argtypes = [c_void_p] * 6 + [c_int, c_int, c_void_p]
    L.co_op_step.argtypes = [c_void_p] * 12 + [c_int, c_int, c_void_p]
    L.co_pctsp_action_mask.argtypes = [c_void_p] * 3 + [c_int, c_int, c_void_p]
    L.co_pctsp_step.argtypes = [c_void_p] * 11 + [c_int, c_int, c_void_p]
    L.co_op_reward.argtypes = [c_void_p] * 3 + [c_int, c_int, c_int, c_void_p]
    L.co_tsp_two_opt.argtypes = [c_void_p] * 4 + [c_int, c_int, c_int, c_void_p]
    L.co_instance_norm.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_long, c_int, c_float, c_void_p]
    L.co_attn_fwd.argtypes = [POINTER(AttnArgs), c_void_p]
    L.co_attn_bwd.argtypes = [POINTER(AttnArgs), c_void_p]
    L.co_cache_width.argtypes = [c_int]
    L.co_split_tf32.argtypes = [c_void_p, c_void_p, c_void_p, ctypes.c_long, c_void_p]
    L.co_gemm_tf32x3.argtypes = [c_void_p] * 8 + [c_int] * 7 + [c_void_p]
    L.co_encoder_mha.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p]
    L.co_ffn_fused.argtypes = [c_void_p] * 7 + [c_int, c_int, c_int, c_void_p]
    L.co_ffn_tile_weights.argtypes = [c_void_p] * 5 + [c_void_p]
    L.co_ffn_tiled_weight_floats.restype = ctypes.c_long
    L.co_generate_uniform.argtypes = [c_void_p, ctypes.c_long, c_uint64, c_uint64, c_float, c_float, c_void_p]
    L.co_generate_demand.argtypes = [c_void_p, ctypes.c_long, c_uint64, c_uint64, c_int, c_int, c_float, c_void_p]
    L.co_dihedral8.argtypes = [c_void_p, c_void_p, ctypes.c_long, c_int, c_void_p]
    _lib = L
    return L


#: number of libcorollout kernel launches issued through this module (bench.py's gpu_launches)
LAUNCH_COUNT = 0


def _check(rc: int, what: str) -> None:
    global LAUNCH_COUNT
    LAUNCH_COUNT += 1
    if rc != CO_OK:
        msg = lib().co_last_error_string().decode("utf-8", "replace")
        raise NativeLibraryError(f"{what} failed with code {rc}: {msg}")


def _ptr(t: torch.Tensor | None, dtype: torch.dtype | None = None, name: str = "tensor", strided: bool = False):
    if t is None:
        return None
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise NativeLibraryError(f"{name}: libcorollout needs CUDA tensors (got device {t.device}); "
                                 "there is no CPU fallback")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not strided and not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _on_device_of_first_tensor(fn):
    """Run the wrapper with the CUDA device of its first tensor argument current, so the kernel is
    enqueued on that device's current stream (a process may hold tensors on several GPUs)."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        for a in list(args) + list(kwargs.values()):
            if isinstance(a, torch.Tensor) and a.is_cuda:
                if a.device.index != torch.cuda.current_device():
                    with torch.cuda.device(a.device):
                        return fn(*args, **kwargs)
                break
        return fn(*args, **kwargs)

    return wrapper


F32, I64, U8, I32 = torch.float32, torch.int64, torch.uint8, torch.int32


def _bool_ptr(t, name):
    """bool tensors are 1 byte; accept bool or uint8."""
    if t is None:
        return None
    if t.dtype not in (torch.bool, torch.uint8):
        raise TypeError(f"{name}: expected bool/uint8, got {t.dtype}")
    return _ptr(t, None, name)


# ----------------------------------------------------------------------------- wrappers


def version() -> int:
    return lib().co_version()


def cache_width(env_name: str) -> int:
    return lib().co_cache_width(ENV_KIND[env_name])


def rollout_max_nodes() -> int:
    return lib().co_rollout_max_nodes()


@_on_device_of_first_tensor
def tsp_step(action, mask_in, mask_out, first_node, current_node, i, done):
    B, N = mask_in.shape
    _check(lib().co_tsp_step(_ptr(action, I64, "action"), _bool_ptr(mask_in, "mask_in"), _bool_ptr(mask_out, "mask_out"),
                             _ptr(first_node, I64, "first_node"), _ptr(current_node, I64, "current_node"),
                             _ptr(i, I64, "i"), _bool_ptr(done, "done"), B, N, _stream()), "co_tsp_step")


@_on_device_of_first_tensor
def cvrp_action_mask(demand, used, cap, visited, current_node, mask_out):
    B, N = visited.shape
    _check(lib().co_cvrp_action_mask(_ptr(demand, F32, "demand"), _ptr(used, F32, "used"), _ptr(cap, F32, "cap"),
                                     _ptr(visited, U8, "visited"), _ptr(current_node, I64, "current_node"),
                                     _bool_ptr(mask_out, "mask_out"), B, N, _stream()), "co_cvrp_action_mask")


@_on_device_of_first_tensor
def cvrp_step(action, demand, cap, used_in, used_out, visited_in, visited_out, current_node, done, mask_out):
    B, N = visited_in.shape
    _check(lib().co_cvrp_step(_ptr(action, I64, "action"), _ptr(demand, F32, "demand"), _ptr(cap, F32, "cap"),
                              _ptr(used_in, F32, "used_in"), _ptr(used_out, F32, "used_out"),
                              _ptr(visited_in, U8, "visited_in"), _ptr(visited_out, U8, "visited_out"),
                              _ptr(current_node, I64, "current_node"), _bool_ptr(done, "done"),
                              _bool_ptr(mask_out, "mask_out"), B, N, _stream()), "co_cvrp_step")


@_on_device_of_first_tensor
def sdvrp_action_mask(demand_with_depot, used, cap, current_node, mask_out):
    B, N = demand_with_depot.shape
    _check(lib().co_sdvrp_action_mask(_ptr(demand_with_depot, F32, "demand_with_depot"), _ptr(used, F32, "used_capacity"),
                                      _ptr(cap, F32, "vehicle_capacity"), _ptr(current_node, I64, "current_node"),
                                      _bool_ptr(mask_out, "mask_out"), B, N, _stream()), "co_sdvrp_action_mask")
    return mask_out


@_on_device_of_first_tensor
def sdvrp_step(action, demand_in, demand_out, cap, used_in, used_out, current_node, done, mask_out):
    B, N = demand_in.shape
    _check(lib().co_sdvrp_step(_ptr(action, I64, "action"), _ptr(demand_in, F32, "demand_in"),
                               _ptr(demand_out, F32, "demand_out"), _ptr(cap, F32, "vehicle_capacity"),
                               _ptr(used_in, F32, "used_in"), _ptr(used_out, F32, "used_out"),
                               _ptr(current_node, I64, "current_node"), _bool_ptr(done, "done"),
                               _bool_ptr(mask_out, "mask_out"), B, N, _stream()), "co_sdvrp_step")


@_on_device_of_first_tensor
def op_action_mask(locs, max_length, visited, tour_length, current_node, mask_out):
    """co_op_action_mask (op/env.py:140-155)."""
    B, N = mask_out.shape
    _check(lib().co_op_action_mask(_ptr(locs, F32, "locs"), _ptr(max_length, F32, "max_length"), _bool_ptr(visited, "visited"),
                                   _ptr(tour_length, F32, "tour_length"), _ptr(current_node, I64, "current_node"),
                                   _bool_ptr(mask_out, "mask_out"), B, N, _stream()), "co_op_action_mask")
    return mask_out


@_on_device_of_first_tensor
def op_step(action, locs, prize, max_length, visited_in, visited_out, tour_length, current_total_prize, current_node, i,
            done, mask_out):
    """co_op_step (op/env.py:72-105 + get_action_mask): tour_length, current_total_prize, current_node, i in place."""
    B, N = mask_out.shape
    _check(lib().co_op_step(_ptr(action, I64, "action"), _ptr(locs, F32, "locs"), _ptr(prize, F32, "prize"),
                            _ptr(max_length, F32, "max_length"), _bool_ptr(visited_in, "visited_in"),
                            _bool_ptr(visited_out, "visited_out"), _ptr(tour_length, F32, "tour_length"),
                            _ptr(current_total_prize, F32, "current_total_prize"), _ptr(current_node, I64, "current_node"),
                            _ptr(i, I64, "i"), _bool_ptr(done, "done"), _bool_ptr(mask_out, "mask_out"), B, N, _stream()),
           "co_op_step")


@_on_device_of_first_tensor
def pctsp_action_mask(visited, cur_total_prize, mask_out):
    """co_pctsp_action_mask (pctsp/env.py:143-151)."""
    B, N = mask_out.shape
    _check(lib().co_pctsp_action_mask(_bool_ptr(visited, "visited"), _ptr(cur_total_prize, F32, "cur_total_prize"),
                                      _bool_ptr(mask_out, "mask_out"), B, N, _stream()), "co_pctsp_action_mask")
    return mask_out


@_on_device_of_first_tensor
def pctsp_step(action, real_prize, penalty, visited_in, visited_out, cur_total_prize, cur_total_penalty, current_node, i, done,
               mask_out):
    """co_pctsp_step (pctsp/env.py:62-93 + get_action_mask): prize / penalty sums, current_node, i in place."""
    B, N = mask_out.shape
    _check(lib().co_pctsp_step(_ptr(action, I64, "action"), _ptr(real_prize, F32, "real_prize"), _ptr(penalty, F32, "penalty"),
                               _bool_ptr(visited_in, "visited_in"), _bool_ptr(visited_out, "visited_out"),
                               _ptr(cur_total_prize, F32, "cur_total_prize"), _ptr(cur_total_penalty, F32, "cur_total_penalty"),
                               _ptr(current_node, I64, "current_node"), _ptr(i, I64, "i"), _bool_ptr(done, "done"),
                               _bool_ptr(mask_out, "mask_out"), B, N, _stream()), "co_pctsp_step")


@_on_device_of_first_tensor
def op_reward(prize, actions):
    """co_op_reward (op/env.py:157-165): prize [B_inst, N] (depot 0), actions [B, T] -> [B]; trajectory j uses instance
    j % B_inst."""
    B, T = actions.shape
    if prize.shape[0] != B:
        prize = prize.repeat(B // prize.shape[0], 1)
    out = torch.empty(B, dtype=F32, device=actions.device)
    _check(lib().co_op_reward(_ptr(prize.contiguous(), F32, "prize"), _ptr(actions, I64, "actions"), _ptr(out, F32, "reward"),
                              B, prize.shape[1], T, _stream()), "co_op_reward")
    return out


@_on_device_of_first_tensor
def tsp_two_opt(locs, tours, max_iterations, moves=None):
    """co_tsp_two_opt (tsp/local_search.py:16-81): 2-opt on tours [B, N] int64 over locs [B, N, 2] -> a new [B, N] int64
    tensor; the input is not modified.  `moves` ([B] int32), if given, receives the moves applied per row, or -1 for a
    row with a node index outside [0, N), which is returned unchanged.  max_iterations <= 0 changes nothing."""
    if tours.dim() != 2 or tuple(locs.shape) != (*tours.shape, 2):
        raise ValueError(f"tours must be [B, N] and locs [B, N, 2], got {tuple(tours.shape)} and {tuple(locs.shape)}")
    B, N = tours.shape
    if moves is not None and tuple(moves.shape) != (B,):
        raise ValueError(f"moves must be [{B}], got {tuple(moves.shape)}")
    out = torch.empty_like(tours)
    args = (_ptr(locs, F32, "locs"), _ptr(tours, I64, "tours"), _ptr(out, I64, "tours_out"), _ptr(moves, I32, "moves"))
    if B == 0:
        return out
    _check(lib().co_tsp_two_opt(*args, B, N, max(0, min(int(max_iterations), 2**31 - 1)), _stream()), "co_tsp_two_opt")
    return out


@_on_device_of_first_tensor
def tour_length(locs, actions, with_depot: bool):
    B, T = actions.shape
    B_locs, N = locs.shape[0], locs.shape[1]
    reward = torch.empty(B, dtype=F32, device=actions.device)
    _check(lib().co_tour_length(_ptr(locs, F32, "locs"), _ptr(actions, I64, "actions"), _ptr(reward, F32, "reward"),
                                B, B_locs, N, T, int(with_depot), _stream()), "co_tour_length")
    return reward


@_on_device_of_first_tensor
def check_tours(actions, N, demand=None, cap=None, B_inst=None) -> int:
    """Number of invalid tours (one host sync, like the reference's asserts)."""
    B, T = actions.shape
    bad = torch.zeros(1, dtype=I32, device=actions.device)
    _check(lib().co_check_tours(_ptr(actions, I64, "actions"), _ptr(demand, F32, "demand"), _ptr(cap, F32, "cap"),
                                _ptr(bad, I32, "bad"), B, B if B_inst is None else B_inst, N, T, _stream()),
           "co_check_tours")
    return int(bad.item())


@_on_device_of_first_tensor
def pointer_logits(env_name, weights: DecoderWeights, node_emb, graph_ctx, K, V, L, mask, first_node, current_node,
                   i, used, cap, B_traj, B_inst, N):
    """K / V / L: [B_inst, N, E] tensors, either contiguous or column-block views of one
    [B_inst, N, W] cache (same row stride, unit channel stride)."""
    ld = K.stride(1)
    for name, x in (("glimpse_key", K), ("glimpse_val", V), ("logit_key", L)):
        if x.stride(2) != 1 or x.stride(1) != ld or x.stride(0) != N * ld:
            raise ValueError(f"{name}: unsupported strides {x.stride()}")
    logits = torch.empty(B_traj, N, dtype=F32, device=node_emb.device)
    # "op" shares the cvrp decoder arithmetic (context = [h_cur ; budget - spent], context.py:201-213): max_length[:, 0]
    # and tour_length stand in for vehicle_capacity and used_capacity
    _check(lib().co_pointer_logits(ENV_KIND["cvrp" if env_name in ("op", "pctsp") else env_name], ctypes.byref(weights), _ptr(node_emb, F32, "node_emb"),
                                   _ptr(graph_ctx, F32, "graph_ctx"), _ptr(K, F32, "glimpse_key", True),
                                   _ptr(V, F32, "glimpse_val", True), _ptr(L, F32, "logit_key", True),
                                   _bool_ptr(mask, "action_mask"), _ptr(first_node, I64, "first_node"),
                                   _ptr(current_node, I64, "current_node"), _ptr(i, I64, "i"),
                                   _ptr(used, F32, "used_capacity"), _ptr(cap, F32, "vehicle_capacity"),
                                   _ptr(logits, F32, "logits"), B_traj, B_inst, N, ld, _stream()), "co_pointer_logits")
    return logits


@_on_device_of_first_tensor
def select_action(logits, mask, mode, noise=None, action=None, tanh_clipping=10.0, temperature=1.0,
                  mask_logits=True, store_all_logp=False, seed=0, offset=0):
    B, N = logits.shape
    if action is None:
        action = torch.empty(B, dtype=I64, device=logits.device)
    logp = torch.empty(B, dtype=F32, device=logits.device)
    all_lp = torch.empty(B, N, dtype=F32, device=logits.device) if store_all_logp else None
    _check(lib().co_select_action(_ptr(logits, F32, "logits"), _bool_ptr(mask, "mask"), _ptr(noise, F32, "noise"),
                                  _ptr(action, I64, "action"), _ptr(logp, F32, "logp"), _ptr(all_lp, F32, "logprobs"),
                                  mode, float(tanh_clipping), float(temperature), int(mask_logits), seed, offset,
                                  B, N, _stream()), "co_select_action")
    return action, logp, all_lp


@_on_device_of_first_tensor
def split_tf32(w: torch.Tensor):
    """(hi, lo) with hi = rna_tf32(w), lo = w - hi (both fp32) for co_gemm_tf32x3."""
    w = w.detach().contiguous()
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    _check(lib().co_split_tf32(_ptr(w, F32, "w"), _ptr(hi, F32, "hi"), _ptr(lo, F32, "lo"), w.numel(), _stream()),
           "co_split_tf32")
    return hi, lo


@_on_device_of_first_tensor
def gemm_tf32x3(a, w_hi, w_lo, out=None, bias=None, residual=None, scale=None, shift=None, relu=False):
    """out[M, Nout] = epilogue(a[M, K] @ W[Nout, K]^T) on tcgen05 tensor cores (3xTF32).
    `a`, `out`, `residual` may be row-strided 2-D views (unit column stride)."""
    M, K = a.shape
    Nout = w_hi.shape[0]
    if out is None:
        out = torch.empty(M, Nout, dtype=F32, device=a.device)
    for name, x in (("a", a), ("out", out), ("residual", residual)):
        if x is not None and (x.dim() != 2 or x.stride(1) != 1):
            raise ValueError(f"{name}: need a 2-D tensor with unit column stride")
    _check(lib().co_gemm_tf32x3(_ptr(a, F32, "a", True), _ptr(w_hi, F32, "w_hi"), _ptr(w_lo, F32, "w_lo"),
                                _ptr(out, F32, "out", True), _ptr(bias, F32, "bias"), _ptr(residual, F32, "residual", True),
                                _ptr(scale, F32, "scale"), _ptr(shift, F32, "shift"), M, Nout, K, a.stride(0),
                                out.stride(0), residual.stride(0) if residual is not None else 0, int(relu), _stream()),
           "co_gemm_tf32x3")
    return out


@_on_device_of_first_tensor
def encoder_mha(qkv, B, N):
    """Self-attention core on the packed [B*N, 384] projection -> [B*N, 128]."""
    out = torch.empty(B * N, EMBED_DIM, dtype=F32, device=qkv.device)
    _check(lib().co_encoder_mha(_ptr(qkv, F32, "qkv"), _ptr(out, F32, "out"), B, N, _stream()), "co_encoder_mha")
    return out


@_on_device_of_first_tensor
def ffn_tile_weights(w1_hi, w1_lo, w2_hi, w2_lo):
    """Pre-tile the split FFN weights (W1 [512,128], W2 [128,512]) into the image `ffn_fused` streams with TMA."""
    if tuple(w1_hi.shape) != (4 * EMBED_DIM, EMBED_DIM) or tuple(w2_hi.shape) != (EMBED_DIM, 4 * EMBED_DIM):
        raise ValueError("co_ffn_fused is instantiated for a 128 -> 512 -> 128 feed-forward block")
    out = torch.empty(lib().co_ffn_tiled_weight_floats(), dtype=F32, device=w1_hi.device)
    _check(lib().co_ffn_tile_weights(_ptr(w1_hi, F32, "w1_hi"), _ptr(w1_lo, F32, "w1_lo"), _ptr(w2_hi, F32, "w2_hi"),
                                     _ptr(w2_lo, F32, "w2_lo"), _ptr(out, F32, "wtiled"), _stream()), "co_ffn_tile_weights")
    return out


@_on_device_of_first_tensor
def ffn_fused(x, wtiled, b1, b2, scale=None, shift=None, out=None):
    """out = ((x + relu(x W1^T + b1) W2^T + b2)) * scale + shift in one kernel (co_ffn_fused); x [M, 128] with
    row stride % 4 == 0, `wtiled` from `ffn_tile_weights`."""
    M = x.shape[0]
    if x.dim() != 2 or x.shape[1] != EMBED_DIM or x.stride(1) != 1:
        raise ValueError(f"x must be [M, {EMBED_DIM}] with unit inner stride, got {tuple(x.shape)}")
    if out is None:
        out = torch.empty(M, EMBED_DIM, dtype=F32, device=x.device)
    _check(lib().co_ffn_fused(_ptr(x, F32, "x", True), _ptr(wtiled, F32, "wtiled"), _ptr(b1, F32, "b1"),
                              _ptr(b2, F32, "b2"), _ptr(scale, F32, "scale"), _ptr(shift, F32, "shift"),
                              _ptr(out, F32, "out", True), M, x.stride(0), out.stride(0), _stream()), "co_ffn_fused")
    return out


def generate_uniform(shape, device, seed: int, offset: int = 0, lo: float = 0.0, hi: float = 1.0):
    """U[lo, hi) floats generated on the device (Philox keyed by seed / offset)."""
    out = torch.empty(shape, dtype=F32, device=device)
    with torch.cuda.device(out.device):
        _check(lib().co_generate_uniform(_ptr(out, F32, "out"), out.numel(), int(seed), int(offset), float(lo), float(hi),
                                         _stream()), "co_generate_uniform")
    return out


def generate_demand(shape, device, seed: int, offset: int, min_demand: int, max_demand: int, capacity: float):
    """CVRP demands (int(U * (max-min) + (min-1)) + 1) / capacity generated on the device."""
    out = torch.empty(shape, dtype=F32, device=device)
    with torch.cuda.device(out.device):
        _check(lib().co_generate_demand(_ptr(out, F32, "out"), out.numel(), int(seed), int(offset), int(min_demand),
                                        int(max_demand), float(capacity), _stream()), "co_generate_demand")
    return out


@_on_device_of_first_tensor
def dihedral8(locs):
    """[B, N, 2] -> [8B, N, 2] (aug-major), one kernel."""
    B, N, _ = locs.shape
    out = torch.empty(8 * B, N, 2, dtype=F32, device=locs.device)
    _check(lib().co_dihedral8(_ptr(locs, F32, "locs"), _ptr(out, F32, "out"), B, N, _stream()), "co_dihedral8")
    return out


@_on_device_of_first_tensor
def instance_norm(x, gamma=None, beta=None, eps: float = 1e-5, out=None):
    """co_instance_norm: nn.InstanceNorm1d(E, affine) over the node dimension of x [B, N, 128] (contiguous)."""
    if x.dim() != 3 or x.shape[-1] != EMBED_DIM:
        raise ValueError(f"x: expected [B, N, {EMBED_DIM}], got {tuple(x.shape)}")
    if out is None:
        out = torch.empty_like(x)
    _check(lib().co_instance_norm(_ptr(x, F32, "x"), _ptr(gamma, F32, "gamma"), _ptr(beta, F32, "beta"),
                                  _ptr(out, F32, "out"), x.shape[0], x.shape[1], float(eps), _stream()), "co_instance_norm")
    return out


def _attn_view(t, name, rows=None):
    """[B, rows, 128] fp32 CUDA tensor whose last dimension is contiguous -> (ptr, batch stride, row stride)."""
    if t.dim() != 3 or t.shape[-1] != EMBED_DIM or t.stride(-1) != 1:
        raise ValueError(f"{name}: expected [B, rows, {EMBED_DIM}] with a contiguous last dimension, got {tuple(t.shape)} / {t.stride()}")
    if rows is not None and t.shape[1] != rows:
        raise ValueError(f"{name}: expected {rows} rows, got {t.shape[1]}")
    bs, rs = (t.stride(0) if t.shape[0] > 1 else t.shape[1] * t.stride(1)), t.stride(1)
    if bs % 4 or rs % 4 or t.data_ptr() % 16:
        raise ValueError(f"{name}: strides must be multiples of 4 floats and the base 16-byte aligned")
    return _ptr(t, F32, name, strided=True), bs, rs


def _attn_args(q, k, v, mask_words, o, lse):
    B, M, _ = q.shape
    N = k.shape[1]
    a = AttnArgs()
    a.q, a.q_bs, a.q_rs = _attn_view(q, "q")
    a.k, a.k_bs, a.k_rs = _attn_view(k, "k")
    a.v, a.v_bs, a.v_rs = _attn_view(v, "v", N)
    a.o, a.o_bs, a.o_rs = _attn_view(o, "o", M)
    if mask_words is not None:
        if tuple(mask_words.shape) != (B, M, 4) or mask_words.dtype != torch.int32:
            raise ValueError(f"mask_words: expected int32 [{B}, {M}, 4], got {mask_words.dtype} {tuple(mask_words.shape)}")
        a.mask = _ptr(mask_words, torch.int32, "mask_words")
    if tuple(lse.shape) != (B, NUM_HEADS, M):
        raise ValueError(f"lse: expected [{B}, {NUM_HEADS}, {M}], got {tuple(lse.shape)}")
    a.lse = _ptr(lse, F32, "lse")
    a.B, a.M, a.N = B, M, N
    a.scale = 0.25
    return a


@_on_device_of_first_tensor
def attn_fwd(q, k, v, mask_words, o, lse):
    """co_attn_fwd: o, lse <- attention(q, k, v[, mask]); q [B,M,E], k / v [B,N,E] (strided views allowed)."""
    a = _attn_args(q, k, v, mask_words, o, lse)
    _check(lib().co_attn_fwd(ctypes.byref(a), _stream()), "co_attn_fwd")
    return o


@_on_device_of_first_tensor
def attn_bwd(q, k, v, mask_words, o, lse, dO, dq, dk, dv):
    """co_attn_bwd: dq, dk, dv <- gradients of attention(q, k, v[, mask]) given dO (same strides as o)."""
    a = _attn_args(q, k, v, mask_words, o, lse)
    if dO.shape != o.shape or dO.stride() != o.stride():
        raise ValueError("dO must have the shape and strides of o")
    a.dO = _ptr(dO, F32, "dO", strided=True)
    a.dq, a.dq_bs, a.dq_rs = _attn_view(dq, "dq", q.shape[1])
    a.dk, a.dk_bs, a.dk_rs = _attn_view(dk, "dk", k.shape[1])
    a.dv, a.dv_bs, a.dv_rs = _attn_view(dv, "dv", k.shape[1])
    _check(lib().co_attn_bwd(ctypes.byref(a), _stream()), "co_attn_bwd")


@_on_device_of_first_tensor
def reward_stats(reward, out2):
    _check(lib().co_reward_stats(_ptr(reward, F32, "reward"), _ptr(out2, torch.float64, "out2"), reward.numel(),
                                 _stream()), "co_reward_stats")


@_on_device_of_first_tensor
def rollout(env_name, select_mode, cache, graph_ctx, q_placeholder, w_capacity, locs, demand, vehicle_capacity,
            B_inst, N, num_starts=1, forced_start=False, num_loc=0, T_max=None, forced_actions=None, noise=None,
            tanh_clipping=10.0, temperature=1.0, seed=0, offset=0, node_emb=None, w_first=None, dyn_w=None,
            node_limit=None):
    """Launch the persistent rollout kernel; returns dict of device tensors (no host sync).
    `cache` is [B_inst, N, W]: W = 4E ([K | V | L' | cur-table]; tsp then needs `node_emb` [B_inst, N, E] and
    `w_first` [E, E] for the per-episode first-node GEMV) or, tsp only, 5E (with the first-node table)."""
    dev = cache.device
    S = max(1, int(num_starts))
    B_traj = B_inst * S
    if T_max is None:
        T_max = {"tsp": N, "cvrp": 2 * (N - 1), "op": N + 1, "pctsp": N + 1}.get(env_name, 3 * (N - 1) + 2)
    actions = torch.empty(B_traj, T_max, dtype=I64, device=dev)
    logp = torch.empty(B_traj, T_max, dtype=F32, device=dev)
    reward = torch.empty(B_traj, dtype=F32, device=dev)
    loglik = torch.empty(B_traj, dtype=F32, device=dev)
    steps = torch.empty(B_traj, dtype=I32, device=dev)
    max_steps = torch.zeros(1, dtype=I32, device=dev)
    used_out = torch.empty(B_traj, dtype=F32, device=dev) if env_name in ("cvrp", "sdvrp") else None
    a = RolloutArgs()
    a.env_kind, a.select_mode, a.B_inst, a.num_starts = ENV_KIND[env_name], select_mode, B_inst, S
    a.N, a.T_max, a.num_loc, a.flags = N, T_max, int(num_loc), (ROLLOUT_FORCED_START if forced_start else 0)
    a.tanh_clipping, a.temperature = float(tanh_clipping), float(temperature)
    a.cache = _ptr(cache, F32, "cache")
    a.graph_ctx = _ptr(graph_ctx, F32, "graph_ctx")
    a.q_placeholder = _ptr(q_placeholder, F32, "q_placeholder")
    a.w_capacity = _ptr(w_capacity, F32, "w_capacity")
    a.locs = _ptr(locs, F32, "locs")
    a.demand = _ptr(demand, F32, "demand")
    a.vehicle_capacity = _ptr(vehicle_capacity, F32, "vehicle_capacity")
    a.forced_actions = _ptr(forced_actions, I64, "forced_actions")
    a.noise = _ptr(noise, F32, "noise")
    a.seed, a.offset = int(seed), int(offset)
    a.actions_out, a.logp_out = _ptr(actions, I64, "actions"), _ptr(logp, F32, "logp")
    a.reward_out, a.loglik_out = _ptr(reward, F32, "reward"), _ptr(loglik, F32, "loglik")
    a.steps_out, a.max_steps_out = _ptr(steps, I32, "steps"), _ptr(max_steps, I32, "max_steps")
    a.used_capacity_out = _ptr(used_out, F32, "used_out")
    W = cache.shape[-1]
    ok_w = (4 * EMBED_DIM, 5 * EMBED_DIM) if env_name == "tsp" else (4 * EMBED_DIM,)
    if cache.dim() != 3 or tuple(cache.shape[:2]) != (B_inst, N) or W not in ok_w:
        raise ValueError(f"cache shape {tuple(cache.shape)} != ({B_inst}, {N}, {' | '.join(map(str, ok_w))})")
    if env_name == "tsp" and W == 4 * EMBED_DIM:
        if node_emb is None or w_first is None:
            raise ValueError("tsp cache of width 4E needs node_emb and w_first")
        if tuple(node_emb.shape) != (B_inst, N, EMBED_DIM) or tuple(w_first.shape) != (EMBED_DIM, EMBED_DIM):
            raise ValueError("node_emb must be [B_inst, N, E] and w_first [E, E]")
        a.node_emb, a.w_first = _ptr(node_emb, F32, "node_emb"), _ptr(w_first, F32, "w_first")
    a.cache_width = W
    if env_name == "sdvrp":
        if dyn_w is None or tuple(dyn_w.shape) != (3 * EMBED_DIM,):
            raise ValueError("sdvrp needs dyn_w [3E] (dynamic-embedding weights, logit third folded)")
        a.dyn_w = _ptr(dyn_w, F32, "dyn_w")
    if env_name in ("op", "pctsp"):
        if node_limit is None or tuple(node_limit.shape) != (B_inst, N):
            raise ValueError(f"{env_name} needs node_limit [{B_inst}, {N}] (op: max_length, pctsp: penalty)")
        a.node_limit = _ptr(node_limit, F32, "node_limit")
    if forced_actions is not None and tuple(forced_actions.shape) != (B_traj, T_max):
        raise ValueError(f"forced_actions must be [{B_traj}, {T_max}], got {tuple(forced_actions.shape)}")
    if noise is not None and (noise.dim() != 3 or noise.shape[1] != B_traj or noise.shape[2] != N):
        raise ValueError(f"noise must be [T, {B_traj}, {N}], got {tuple(noise.shape)}")
    _check(lib().co_rollout(ctypes.byref(a), _stream()), "co_rollout")
    return {"actions": actions, "logprobs": logp, "reward": reward, "log_likelihood": loglik, "steps": steps,
            "max_steps": max_steps, "used_capacity": used_out}
