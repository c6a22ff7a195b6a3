"""The C-ABI library loads on a machine without a GPU, exports every symbol include/stomp_b200.h
declares, and fails loudly (no CPU fallback) when asked to compute without a device."""
import ctypes
import os
import re

import numpy as np
import pytest

from motion_planners_b200 import binding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "stomp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(stomp_b200_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    assert _declared() == sorted(binding.SYMBOLS)


def test_library_exports_every_declared_symbol():
    L = binding.lib()
    for name in _declared():
        assert hasattr(L, name), name
    assert L.stomp_b200_abi_version() == 1


def test_config_struct_layout_matches_the_header():
    cfg = binding.default_config()
    assert cfg.abi_version == 1 and cfg.num_queries == 1 and cfg.world_size == 1
    assert cfg.cost_scaling_h == 10.0 and cfg.use_cumulative_costs == 1 and cfg.use_projection == 0
    assert list(cfg.derivative_weights) == [0.0, 0.0, 1.0, 0.0]
    assert cfg.noise_decay[31] == 1.0 and cfg.seed == 2024


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_has_gpu(), reason="this test is about machines without a GPU")
def test_no_device_means_an_error_not_a_fallback():
    with pytest.raises(binding.StompB200Error) as err:
        binding.Engine(num_time_steps=20, num_dimensions=7, min_rollouts=4, max_rollouts=4, num_rollouts_per_iteration=4)
    assert err.value.code == binding.ERR_NO_DEVICE


def test_invalid_configurations_are_rejected_before_touching_the_device():
    L = binding.lib()
    cfg = binding.default_config()
    h = ctypes.c_void_p()
    cfg.num_time_steps, cfg.num_dimensions = 20, 40      # too many joints
    cfg.min_rollouts = cfg.max_rollouts = cfg.num_rollouts_per_iteration = 4
    assert L.stomp_b200_create(ctypes.byref(cfg), ctypes.byref(h)) == -1
    cfg.num_dimensions, cfg.use_cumulative_costs = 7, 0   # per-time-step costs ...
    cfg.min_rollouts, cfg.max_rollouts = 2, 8             # ... with rollout reuse: a combination that is not built
    assert L.stomp_b200_create(ctypes.byref(cfg), ctypes.byref(h)) == binding.ERR_UNSUPPORTED
    cfg.use_cumulative_costs, cfg.shard_mode = 1, 7       # no such sharding mode
    assert L.stomp_b200_create(ctypes.byref(cfg), ctypes.byref(h)) == -1
    cfg.shard_mode, cfg.world_size, cfg.rank = 0, 2, 0    # rollout sharding ...
    cfg.min_rollouts, cfg.max_rollouts, cfg.num_rollouts_per_iteration = 4, 8, 4   # ... with rollout reuse
    assert L.stomp_b200_create(ctypes.byref(cfg), ctypes.byref(h)) == binding.ERR_UNSUPPORTED
    cfg.min_rollouts, cfg.max_rollouts, cfg.num_rollouts_per_iteration = 5, 5, 5   # ... with shards of unequal size
    assert L.stomp_b200_create(ctypes.byref(cfg), ctypes.byref(h)) == binding.ERR_UNSUPPORTED
    assert L.stomp_b200_status_string(-2).decode().startswith("no CUDA device")


def test_generated_state_kernel_compiles_for_sm_100a_without_a_device():
    """csrc/state_codegen.hpp: the state kernel is generated per robot structure and compiled with NVRTC at run time.
    The self-test generates it for a structure that uses every template branch (all axis kinds, fixed rotation,
    prismatic joint, chain restart, every zero mask, narrow and wide voxel index) and compiles both to sm_100a cubins."""
    rc, log = binding.codegen_selftest()
    assert rc == 0, log
    assert log.count("byte cubin") == 3 and "pair rule" in log      # narrow and wide SDF index, and the walk with the sphere-pair rule inside
    # the first sphere of each of the two chains sits at its joint's origin: no joint value moves it, so it leaves the walk for
    # stomp_b200_static_spheres (state_codegen.hpp: FoldingEmitter::centre_is_static); the second chain starts with an x axis
    import re
    counts = [int(n) for n in re.findall(r"(\d+) static spheres", log)]
    assert len(counts) == 2 and all(c >= 1 for c in counts), log


def test_header_is_plain_c():
    """The drop-in boundary is a C ABI: include/stomp_b200.h must compile as C99 on its own (no C++, no torch types)."""
    import subprocess
    hdr = os.path.join(ROOT, "include", "stomp_b200.h")
    out = subprocess.run(["gcc", "-x", "c", "-std=c99", "-fsyntax-only", "-Wall", "-Wextra", "-Werror", hdr], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
