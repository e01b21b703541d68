"""ctypes binding of ``libgradjune_b200.so`` (C ABI in ``include/gradjune_b200.h``).

There is no CPU fallback: if the library is missing or an entry point fails, the call raises.
"""
import ctypes as C
import os
import subprocess
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC_DIR = PKG_DIR.parent / "csrc"
INCLUDE_DIR = PKG_DIR.parent.parent / "include"
LIB_PATH = Path(os.environ.get("GJ_LIB_PATH") or PKG_DIR / "libgradjune_b200.so")   # override: kernel experiments

GJ_MAX_TYPES = 8
GJ_MAX_NETS = 16
GJ_MAX_STAGES = 16
GJ_MAX_QUAR = 4
GJ_MAX_AGE_BINS = 8
GJ_MAX_CHANNELS = 8
GJ_ABI_VERSION = 12

KIND_PLAIN, KIND_HOUSEHOLD, KIND_LEISURE, KIND_CARE_VISIT = 0, 1, 2, 3
PHASE_NETWORKS, PHASE_SAMPLE, PHASE_INFECT, PHASE_SYMPTOMS, PHASE_ALL = 1, 2, 4, 8, 15
MODE_STEP, MODE_SEED = 0, 1
STAGE_ALL, STAGE_SUMS, STAGE_REST = 0, 1, 2

_u32p = C.c_void_p
_f32p = C.c_void_p


class WorldDesc(C.Structure):
    _fields_ = [
        ("n_agents", C.c_int64), ("n_groups", C.c_int64), ("n_edges", C.c_int64),
        ("n_types", C.c_int32), ("_pad0", C.c_int32),
        ("type_group_off", C.c_int64 * (GJ_MAX_TYPES + 1)),
        ("am_ptr", _u32p), ("am_ent", _u32p), ("gm_ptr", _u32p), ("gm_agent", _u32p),
        ("pc", _f32p), ("cls", C.c_void_p),
        ("small_groups", _u32p), ("n_small", C.c_int64),
        ("chunk_group", _u32p), ("chunk_begin", _u32p), ("chunk_end", _u32p), ("chunk_part", C.c_void_p),
        ("n_chunks", C.c_int64),
        ("big_groups", _u32p), ("big_part_ptr", _u32p), ("n_big", C.c_int64), ("n_parts", C.c_int64),
        ("type_tier", C.c_int32 * GJ_MAX_TYPES),
        ("range_slot", C.c_void_p * GJ_MAX_TYPES), ("range_pc", C.c_void_p * GJ_MAX_TYPES),
        ("range_pc_from_size", C.c_int32 * GJ_MAX_TYPES),
        ("n_tiles", C.c_int64), ("tile_begin", _u32p), ("tile_flags", _u32p),
        ("n_cells", C.c_int64 * GJ_MAX_TYPES), ("cell_off", C.c_int64 * GJ_MAX_TYPES), ("n_cells_total", C.c_int64),
        ("tile_cell", C.c_void_p * GJ_MAX_TYPES), ("cell_tile_ptr", C.c_void_p * GJ_MAX_TYPES),
        ("cell_grp_ptr", C.c_void_p * GJ_MAX_TYPES), ("cell_grp", C.c_void_p * GJ_MAX_TYPES),
        ("grp_cell_ptr", C.c_void_p * GJ_MAX_TYPES), ("grp_cell", C.c_void_p * GJ_MAX_TYPES),
        ("ent1", _u32p), ("n_giant_chunks", C.c_int64), ("n_giant_big", C.c_int64), ("dbeta_w", _f32p), ("orig_id", _u32p),
    ]


class WorldSrc(C.Structure):
    """gj_world_src: the reference's own arrays (device pointers for gj_world_build, host for gj_world_build_host)."""
    _fields_ = [
        ("n_agents", C.c_int64), ("n_types", C.c_int32), ("renumber", C.c_int32),
        ("type_name", C.c_char_p * GJ_MAX_TYPES),
        ("edge_agent", C.c_void_p * GJ_MAX_TYPES), ("edge_group", C.c_void_p * GJ_MAX_TYPES),
        ("n_edges", C.c_int64 * GJ_MAX_TYPES), ("n_groups", C.c_int64 * GJ_MAX_TYPES),
        ("people_i64", C.c_void_p * GJ_MAX_TYPES), ("people_f32", C.c_void_p * GJ_MAX_TYPES),
        ("age", C.c_void_p), ("sex", C.c_void_p), ("original_index", C.c_void_p), ("want_tier", C.c_void_p),
    ]


class Net(C.Structure):
    _fields_ = [("type", C.c_int32), ("kind", C.c_int32), ("prob_row", C.c_int32), ("s_off", C.c_int32)]


class Dist(C.Structure):
    _fields_ = [("kind", C.c_int32), ("loc", C.c_float), ("scale", C.c_float)]


class StepParams(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("phases", C.c_int32), ("now", C.c_float), ("dt", C.c_float),
        ("day_type", C.c_int32), ("n_nets", C.c_int32), ("nets", Net * GJ_MAX_NETS),
        ("n_quar", C.c_int32), ("quar_thr", C.c_float * GJ_MAX_QUAR),
        ("n_stages", C.c_int32), ("trans_time", Dist * GJ_MAX_STAGES), ("rec_time", Dist * GJ_MAX_STAGES),
        ("n_age_bins", C.c_int32), ("age_bins", C.c_int32 * (GJ_MAX_AGE_BINS + 1)),
        ("tau", C.c_float), ("seed", C.c_uint64), ("call_index", C.c_uint32), ("exact_order", C.c_uint32),
        ("stage", C.c_uint32), ("t_ready", C.c_uint32), ("reset_scatter", C.c_uint32), ("_pad1", C.c_uint32),
        ("agent_offset", C.c_uint64),
    ]


_FWD_FIELDS = [
    "beta", "leisure_prob", "stage_prob", "seed_fraction", "inj_E", "inj_u", "inj_z",
    "s", "inf", "tinf", "cur", "nxt", "ttn", "maxinf", "shape", "rate", "shift", "k0", "prof4",
    "T_in", "q_in", "n_in",
    "s_o", "inf_o", "tinf_o", "cur_o", "nxt_o", "ttn_o", "T", "Tq", "q", "lam", "n",
    "tape_v", "tape_y0", "S_scaled", "S_unscaled", "red", "scratch", "T_next", "Tq_next",
]
_BWD_FIELDS = [
    "beta", "leisure_prob", "stage_prob", "seed_fraction", "inj_E", "inj_u", "inj_z",
    "s", "inf", "tinf", "cur", "nxt", "ttn", "maxinf", "shape", "rate", "shift", "k0", "prof4",
    "inf_o", "n_in", "T_in", "q_in", "tape_v", "tape_y0", "S_unscaled",
    "g_s_o", "g_inf_o", "g_tinf_o", "g_cur_o", "g_nxt_o", "g_ttn_o", "g_red", "g_q", "g_lam", "g_n",
    "g_s", "g_inf", "g_tinf", "g_cur", "g_nxt", "g_ttn", "g_T", "g_q_out", "g_n_out", "g_beta",
    "g_seed_fraction", "w", "wq", "R", "cR", "scratch",
]


class FwdIO(C.Structure):
    # results by label: codes, column count, fp32 table and its integer accumulator
    _fields_ = [(name, C.c_void_p) for name in _FWD_FIELDS] + [
        ("label", C.c_void_p), ("n_labels", C.c_int32), ("_pad_label", C.c_int32), ("red_label", C.c_void_p),
        ("label_acc", C.c_void_p),
        # seeding by label: region codes and their count
        ("seed_label", C.c_void_p), ("n_seed_labels", C.c_int32), ("_pad_seed", C.c_int32)]


class BwdIO(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in _BWD_FIELDS] + [("label", C.c_void_p), ("g_red_label", C.c_void_p)] + [
        ("seed_label", C.c_void_p), ("n_seed_labels", C.c_int32), ("_pad_seed", C.c_int32), ("seed_order", C.c_void_p),
        ("seed_offsets", C.c_void_p), ("seed_work", C.c_void_p)]


class Batch(C.Structure):
    """gj_batch: strides of a batched ensemble call (gj_step_forward_batch / gj_step_backward_batch)."""
    _fields_ = [("n_samples", C.c_int32), ("_pad0", C.c_int32), ("agent_stride", C.c_int64),
                ("group_stride", C.c_int64), ("beta_stride", C.c_int64), ("red_stride", C.c_int64),
                ("scratch_stride", C.c_int64), ("noise", C.c_void_p), ("label_stride", C.c_int64)]


class GradJuneLibraryError(RuntimeError):
    pass


_lib = None
_config = None

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "--fmad=false",
    "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "--extended-lambda",
]


def build(force=False, verbose=False):
    """Compile csrc/*.cu into libgradjune_b200.so for sm_100a (nvcc cross-compiles without a GPU): one object per
    source file, compiled in parallel, then linked."""
    srcs = sorted(CSRC_DIR.glob("*.cu"))
    deps = srcs + sorted(CSRC_DIR.glob("*.cuh")) + sorted(INCLUDE_DIR.glob("*.h"))
    if not force and LIB_PATH.exists() and all(LIB_PATH.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    objdir = PKG_DIR.parent / "build"
    objdir.mkdir(exist_ok=True)
    procs = []
    for src in srcs:
        obj = objdir / (src.stem + ".o")
        cmd = [nvcc] + flags + ["-I", str(INCLUDE_DIR), "-I", str(CSRC_DIR), "-c", "-o", str(obj), str(src)]
        if verbose:
            print(" ".join(cmd))
        procs.append((cmd, obj, subprocess.Popen(cmd)))
    for cmd, obj, proc in procs:
        if proc.wait() != 0:
            raise subprocess.CalledProcessError(proc.returncode, cmd)
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-o", str(LIB_PATH)] \
        + [str(obj) for _, obj, _ in procs]
    if verbose:
        print(" ".join(link))
    subprocess.run(link, check=True)
    return LIB_PATH


def lib():
    """The loaded library; raises GradJuneLibraryError (loudly) if it cannot be loaded."""
    global _lib, _config
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        try:
            build()
        except Exception as e:  # noqa: BLE001
            raise GradJuneLibraryError(
                f"{LIB_PATH} is missing and could not be built ({e}); run `python __graft_entry__.py build`. "
                "There is no CPU fallback for the infection step."
            ) from e
    try:
        L = C.CDLL(str(LIB_PATH))
    except OSError as e:
        raise GradJuneLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    if L.gj_abi_version() != GJ_ABI_VERSION:
        raise GradJuneLibraryError(f"{LIB_PATH} has ABI version {L.gj_abi_version()}, this binding needs "
                                   f"{GJ_ABI_VERSION}: rebuild with `python __graft_entry__.py build`")
    L.gj_last_error.restype = C.c_char_p
    L.gj_scratch_bytes.restype = C.c_int64
    L.gj_scratch_bytes.argtypes = [C.POINTER(WorldDesc)]
    L.gj_config.argtypes = [C.POINTER(C.c_int64), C.c_int]
    L.gj_profile_prepare.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gj_profile_pack.argtypes = [C.c_int64] + [C.c_void_p] * 7
    L.gj_transmission_forward.argtypes = [C.c_int64, C.c_float] + [C.c_void_p] * 9
    L.gj_transmission_backward.argtypes = [C.c_int64, C.c_float] + [C.c_void_p] * 11
    L.gj_step_forward.argtypes = [C.POINTER(WorldDesc), C.POINTER(StepParams), C.POINTER(FwdIO), C.c_void_p]
    L.gj_step_forward_next.argtypes = [C.POINTER(WorldDesc), C.POINTER(StepParams), C.POINTER(StepParams),
                                       C.POINTER(FwdIO), C.c_void_p]
    L.gj_step_backward.argtypes = [C.POINTER(WorldDesc), C.POINTER(StepParams), C.POINTER(BwdIO), C.c_void_p]
    L.gj_step_forward_batch.argtypes = [C.POINTER(WorldDesc), C.POINTER(StepParams), C.POINTER(FwdIO), C.POINTER(Batch),
                                        C.c_void_p]
    L.gj_step_backward_batch.argtypes = [C.POINTER(WorldDesc), C.POINTER(StepParams), C.POINTER(BwdIO),
                                         C.POINTER(Batch), C.c_void_p]
    L.gj_philox_fill_at.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p]
    L.gj_step_plan.argtypes = [C.POINTER(WorldDesc), C.POINTER(StepParams), C.POINTER(C.c_int64), C.c_int]
    L.gj_philox_fill.argtypes = [C.c_uint64, C.c_uint32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.gj_philox4x32_10.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.gj_philox4x32_10.restype = None
    L.gj_philox2x32_10.argtypes = [C.POINTER(C.c_uint32), C.c_uint32, C.POINTER(C.c_uint32)]
    L.gj_philox2x32_10.restype = None
    L.gj_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int]
    L.gj_profile_kernel_name.restype = C.c_char_p
    L.gj_boundary_pack.argtypes = [C.c_int64] + [C.c_void_p] * 5
    L.gj_boundary_unpack.argtypes = [C.c_int64] + [C.c_void_p] * 5
    L.gj_peer_create.argtypes = [C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_void_p)]
    L.gj_peer_handle.argtypes = [C.c_void_p, C.c_void_p]
    L.gj_peer_connect.argtypes = [C.c_void_p, C.c_void_p]
    L.gj_peer_exchange.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 4 + [C.c_int64, C.c_void_p, C.c_void_p]
    L.gj_peer_status.argtypes = [C.c_void_p]
    L.gj_peer_destroy.argtypes = [C.c_void_p]
    L.gj_world_build.argtypes = [C.POINTER(WorldSrc), C.POINTER(C.c_void_p)]
    L.gj_world_build_host.argtypes = [C.POINTER(WorldSrc), C.POINTER(C.c_void_p)]
    L.gj_world_descriptor.argtypes = [C.c_void_p]
    L.gj_world_descriptor.restype = C.POINTER(WorldDesc)
    L.gj_world_permutation.argtypes = [C.c_void_p]
    L.gj_world_permutation.restype = C.c_void_p
    L.gj_world_last_error.restype = C.c_char_p
    L.gj_world_destroy.argtypes = [C.c_void_p]
    L.gj_memcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    cfg = (C.c_int64 * 10)()
    L.gj_config(cfg, 10)
    _config = {
        "small_group": cfg[0], "chunk": cfg[1], "red_blocks": cfg[6], "tile_agents": cfg[7], "scatter_max": cfg[8],
    }
    sizes = {"gj_world_desc": (cfg[2], C.sizeof(WorldDesc)), "gj_step_params": (cfg[3], C.sizeof(StepParams)),
             "gj_fwd_io": (cfg[4], C.sizeof(FwdIO)), "gj_bwd_io": (cfg[5], C.sizeof(BwdIO)),
             "gj_batch": (cfg[9], C.sizeof(Batch))}
    for name, (c_size, py_size) in sizes.items():
        if c_size != py_size:
            raise GradJuneLibraryError(f"ABI mismatch for {name}: library {c_size} bytes, binding {py_size} bytes")
    _lib = L
    return L


def config():
    lib()
    return dict(_config)


def check(rc, what):
    if rc != 0:
        raise GradJuneLibraryError(f"{what} failed ({rc}): {lib().gj_last_error().decode()}")


EXPORTED_SYMBOLS = [
    "gj_abi_version", "gj_last_error", "gj_config", "gj_scratch_bytes", "gj_profile_prepare", "gj_profile_pack",
    "gj_transmission_forward", "gj_transmission_backward", "gj_step_forward", "gj_step_forward_next", "gj_step_backward",
    "gj_step_forward_batch", "gj_step_backward_batch",
    "gj_philox_fill", "gj_philox_fill_at", "gj_step_plan", "gj_philox4x32_10", "gj_philox2x32_10", "gj_profile_enable", "gj_profile_read",
    "gj_profile_kernel_name", "gj_pipeline_enable", "gj_boundary_pack", "gj_boundary_unpack",
    "gj_peer_create", "gj_peer_handle", "gj_peer_connect", "gj_peer_exchange", "gj_peer_status", "gj_peer_destroy",
    "gj_world_build", "gj_world_build_host", "gj_world_descriptor", "gj_world_permutation", "gj_world_last_error",
    "gj_world_destroy", "gj_memcpy",
]


def pipeline_enable(on=True, lookahead=False, uncompacted=False):
    """Bulk-copy pipelined agent kernels on/off (bit-identical results) and, with them, the fused transmission pass
    of the following step (``lookahead``); ``uncompacted`` selects the transmission pass without the per-warp
    compaction of the infectious agents.  Returns the previous setting as (on, lookahead, uncompacted).
    ``on=None`` queries."""
    prev = lib().gj_pipeline_enable(-1 if on is None else ((1 if on else 0) | (2 if (on and lookahead) else 0)
                                                           | (4 if uncompacted else 0)))
    return bool(prev & 1), bool(prev & 2), bool(prev & 4)


def profile_enable(on=True):
    check(lib().gj_profile_enable(1 if on else 0), "gj_profile_enable")


def profile_read():
    """{kernel name: (summed ms, timed launches, launches)} since profile_enable()."""
    n = 24
    ms, timed, launches = (C.c_double * n)(), (C.c_int64 * n)(), (C.c_int64 * n)()
    k = lib().gj_profile_read(ms, timed, launches, n)
    if k < 0:
        check(k, "gj_profile_read")
    return {lib().gj_profile_kernel_name(i).decode(): (ms[i], timed[i], launches[i]) for i in range(k)}
