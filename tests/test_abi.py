"""CPU checks of the drop-in boundary: the library loads, exports every symbol the header
declares, and fails loudly (no fallback) without a GPU."""
import ctypes
import os
import re

import pytest

from tests.conftest import ROOT


def _header_functions():
    src = open(os.path.join(ROOT, 'include', 'mpe_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    names = re.findall(r'^\s*(?:const\s+char\s*\*|int64_t|int)\s*\*?\s*((?:mpe|actor|critic|replay)_\w+)\s*\(', src, flags=re.M)
    return sorted(set(names))


def test_library_is_built_in_tree():
    from multiagent_rl_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), 'run python -m multiagent_rl_b200.build'


def test_every_declared_symbol_is_exported_and_bound():
    from multiagent_rl_b200 import _lib
    declared = _header_functions()
    assert len(declared) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), 'libmpe_b200.so does not export %s' % name
    assert sorted(_lib.SIGNATURES) == declared, 'python binding and header disagree'
    assert _lib.load().mpe_abi_version() == _lib.ABI_VERSION


def test_struct_layouts_match_header():
    from multiagent_rl_b200 import _lib
    assert ctypes.sizeof(_lib.MpeConfig) == 64
    assert ctypes.sizeof(_lib.MpeDims) == 48
    assert ctypes.sizeof(_lib.ActorConfig) == 24
    assert ctypes.sizeof(_lib.ActorWeights) == 16 * 8
    assert ctypes.sizeof(_lib.CriticConfig) == 24 and ctypes.sizeof(_lib.CriticWeights) == 10 * 8
    assert ctypes.sizeof(_lib.MpeHostBlockLayout) == 48


def test_bad_arguments_are_rejected_before_cuda():
    from multiagent_rl_b200 import _lib
    lib = _lib.load()
    assert lib.mpe_create(None, None) == _lib.MPE_EINVAL
    assert b'null' in lib.mpe_last_error()
    h = ctypes.c_void_p()
    cfg = _lib.MpeConfig(scenario=7, num_envs=4)
    assert lib.mpe_create(ctypes.byref(cfg), ctypes.byref(h)) == _lib.MPE_EUNSUPPORTED
    cfg = _lib.MpeConfig(scenario=0, num_agents=13, num_envs=4)  # simple_spread teams of 1..12 have kernels
    assert lib.mpe_create(ctypes.byref(cfg), ctypes.byref(h)) == _lib.MPE_EUNSUPPORTED
    assert b'13 agents' in lib.mpe_last_error()
    cfg = _lib.MpeConfig(scenario=0, num_envs=0)
    assert lib.mpe_create(ctypes.byref(cfg), ctypes.byref(h)) == _lib.MPE_EINVAL
    assert lib.mpe_step(None, None, None, None, None, None, None, None, None, None) == _lib.MPE_EINVAL
    assert lib.mpe_destroy(None) == _lib.MPE_OK
    # the round-2 entry points reject bad arguments before touching CUDA as well
    assert lib.mpe_act_step_host_async(None, None, None, 0, None, None) == _lib.MPE_EINVAL
    assert lib.mpe_host_block_layout(None, None) == _lib.MPE_EINVAL
    assert lib.mpe_host_alloc(None, 0) == _lib.MPE_EINVAL and lib.mpe_host_free(None) == _lib.MPE_OK
    assert lib.mpe_step_host(None, None, None, None, None, None, None) == _lib.MPE_EINVAL
    assert lib.mpe_reset_host_async(None, None, None) == _lib.MPE_EINVAL
    assert lib.actor_forward_host(None, None, 1, 3, 0, 0, 0, None, None, None, None) == _lib.MPE_EINVAL
    assert lib.critic_create(None, None) == _lib.MPE_EINVAL and lib.critic_destroy(None) == _lib.MPE_OK
    cc = _lib.CriticConfig(obs_dim=60, act_dim=10, out_dim=1)
    assert lib.critic_create(ctypes.byref(cc), ctypes.byref(h)) == _lib.MPE_EUNSUPPORTED
    assert lib.critic_forward(None, None, None, 1, 3, None, None, None) == _lib.MPE_EINVAL
    # a ring whose records replay_add cannot stage (over 48 KB) is refused when it is created, not on every add:
    # record_bytes(32, 191) = 48,976 is the largest accepted, record_bytes(32, 192) = 49,232
    rc = _lib.ReplayConfig(capacity=16, num_agents=32, obs_dim=192, act0=5)
    assert lib.replay_create(ctypes.byref(rc), ctypes.byref(h)) == _lib.MPE_EUNSUPPORTED
    assert b'49232 bytes' in lib.mpe_last_error()
    rc = _lib.ReplayConfig(capacity=16, num_agents=1, obs_dim=1 << 20, act0=5)
    assert lib.replay_create(ctypes.byref(rc), ctypes.byref(h)) == _lib.MPE_EUNSUPPORTED
    assert lib.replay_create(None, None) == _lib.MPE_EINVAL


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    import multiagent_rl_b200 as m
    with pytest.raises(RuntimeError, match='CUDA'):
        m.make_env('simple_spread')
    with pytest.raises(RuntimeError, match='CUDA'):
        m.FusedActor({})


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, 'multiagent_rl_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', txt, flags=re.M), f


def test_only_the_cpu_arms_of_the_bench_touch_the_oracle():
    """tools/ and the B200 arm of bench.py take their synthetic weights from the package; bench.py imports the
    oracle in exactly one place, the CPU loop that serves cpu_baseline and --impl reference."""
    import glob
    for f in glob.glob(os.path.join(ROOT, 'tools', '*.py')):
        assert not re.search(r'^\s*(from|import)\s+oracle\b', open(f).read(), flags=re.M), f
    txt = open(os.path.join(ROOT, 'bench.py')).read()
    hits = [m_.start() for m_ in re.finditer(r'^\s*(from|import)\s+oracle\b', txt, flags=re.M)]
    assert len(hits) == 1
    assert txt.rfind('def cpu_loop', 0, hits[0]) > txt.rfind('def run_b200', 0, hits[0])
