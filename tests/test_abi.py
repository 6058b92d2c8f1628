"""The C-ABI library loads on a CPU-only box, exports every symbol include/*.h declares, agrees
with the ctypes mirror on struct layout, and FAILS LOUDLY (no CPU fallback) without a GPU."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "cleanrl_cuda.h")


def header_symbols():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"CRL_API\s+(?:int|const char\*)\s+(crl_\w+)\s*\(", src)))


def test_header_declares_the_expected_surface_with_the_dqn_raw_kernels():
    """the 50 entry points before the raw DQN kernels plus crl_dqn_forward_raw and crl_dqn_loss_raw"""
    syms = header_symbols()
    assert len(syms) == 52
    for s in ("crl_create", "crl_rollout", "crl_gae", "crl_update_minibatch", "crl_train_update", "crl_gae_raw",
              "crl_env_step_raw", "crl_policy_forward_raw", "crl_ppo_loss_raw", "crl_clip_adam_raw", "crl_comm_init", "crl_dqn_run",
              "crl_dqn_comm_init", "crl_dqn_forward_raw", "crl_dqn_loss_raw"):
        assert s in syms


def test_library_exports_every_header_symbol(crl):
    lib = crl.load()
    for s in header_symbols():
        assert hasattr(lib, s), "libcleanrl_cuda.so does not export %s" % s
    assert set(crl.SIGNATURES) == set(header_symbols())
    assert lib.crl_version() == 100


def test_library_does_not_link_the_oracle_or_nccl_at_load_time():
    out = subprocess.check_output(["ldd", os.path.join(ROOT, "cleanrl.jl_b200", "libcleanrl_cuda.so")], text=True)
    assert "oracle" not in out and "nccl" not in out
    syms = subprocess.check_output(["nm", "-D", os.path.join(ROOT, "cleanrl.jl_b200", "libcleanrl_cuda.so")], text=True)
    assert "orc_" not in syms


def test_struct_layout_matches_the_c_header(tmp_path, abi):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cleanrl_cuda.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(crl_config),offsetof(crl_config,seed),offsetof(crl_config,gamma),sizeof(crl_loss_stats),'
                   'sizeof(crl_episode),sizeof(crl_episode_agg),sizeof(crl_kernel_times),sizeof(crl_dqn_config),sizeof(crl_dqn_stats));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert got == [C.sizeof(abi.crl_config), abi.crl_config.seed.offset, abi.crl_config.gamma.offset,
                   C.sizeof(abi.crl_loss_stats), C.sizeof(abi.crl_episode), C.sizeof(abi.crl_episode_agg),
                   C.sizeof(abi.crl_kernel_times), C.sizeof(abi.crl_dqn_config), C.sizeof(abi.crl_dqn_stats)]


@pytest.mark.skipif("torch" in sys.modules and sys.modules["torch"].cuda.is_available(), reason="CPU-box behaviour")
def test_no_cpu_fallback_without_a_gpu(crl, abi):
    """on a box with no GPU every compute entry point returns CRL_ERR_CUDA with a message"""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is visible")
    except ImportError:
        pass
    lib = crl.load()
    h = C.c_void_p()
    cfg = abi.make_config()
    assert lib.crl_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_CUDA
    assert not h.value
    assert len(lib.crl_last_error()) > 0
    n = C.c_int32()
    assert lib.crl_device_count(C.byref(n)) == abi.CRL_ERR_CUDA
    from cleanrl_jl_b200.handle import PPOHandle
    with pytest.raises(crl.CleanRLCudaError):
        PPOHandle(cfg)
    # argument validation happens before any device work
    bad = abi.make_config(num_envs=3, num_steps=5, num_minibatches=2)
    assert lib.crl_create(C.byref(bad), C.byref(h)) == abi.CRL_ERR_INVALID
    assert b"divisible" in lib.crl_last_error()


ENV_SWITCHES = {"CRL_NO_TC", "CRL_EXACT", "CRL_MULTI_EXACT", "CRL_NO_GRAPH", "CRL_NO_P2P", "CRL_P2P_TIMEOUT_MS",
                "CRL_NCCL_LIB"}


def test_library_reads_exactly_the_documented_environment_switches():
    """every environment variable the native library reads is one of the switches README.md documents, and each is there"""
    csrc = os.path.join(ROOT, "cleanrl.jl_b200", "csrc")
    read = set()
    for f in os.listdir(csrc):
        read |= set(re.findall(r'getenv\(\s*"(\w+)"\s*\)', open(os.path.join(csrc, f)).read()))
    assert read == ENV_SWITCHES
    readme = open(os.path.join(ROOT, "README.md")).read()
    for name in sorted(ENV_SWITCHES):
        assert "`%s" % name in readme, name


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "cleanrl.jl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".jl")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("the oracle", "").replace("oracle's", "").replace("ppo_oracle.c", "").lower() \
                    or f in ("device_math.cuh", "gae.cu", "update.cu"), (dirpath, f)
                assert "import oracle" not in text and "from oracle" not in text and "libppo_oracle" not in text, f


def _build_c_smoke(tmp_path):
    exe = tmp_path / "c_abi_smoke"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c_abi_smoke.c"), "-o", str(exe), "-ldl", "-lm"])
    return str(exe)


def test_pure_c_consumer_compiles_against_the_header_and_fails_loudly_without_a_gpu(tmp_path):
    """tests/c_abi_smoke.c uses nothing but include/cleanrl_cuda.h + dlopen; on a CPU-only box crl_create must fail with
    CRL_ERR_CUDA and a message (no CPU fallback), after the bad configuration has been rejected with CRL_ERR_INVALID"""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is visible")
    except ImportError:
        pass
    exe = _build_c_smoke(tmp_path)
    p = subprocess.run([exe, os.path.join(ROOT, "cleanrl.jl_b200", "libcleanrl_cuda.so")], capture_output=True, text=True)
    assert p.returncode == 1 and "-> -2" in p.stderr and "bad config was not rejected" not in p.stderr, p.stderr


@pytest.mark.gpu
def test_pure_c_consumer_trains_through_the_header_alone(tmp_path, torch_cuda):
    """create -> set_params -> env_reset -> train_update x 3 with lag-1 fetches -> get_params -> destroy, from plain C"""
    exe = _build_c_smoke(tmp_path)
    p = subprocess.run([exe, os.path.join(ROOT, "cleanrl.jl_b200", "libcleanrl_cuda.so")], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "c_abi_smoke ok" in p.stdout
