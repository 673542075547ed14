"""The C++ host adapter that mirrors the reference's NN facade (alphazero_risk_b200/host/az_nn_service.hpp).
CPU part: it compiles standalone against include/az_b200.h and fails loudly without a GPU.
GPU part (marked gpu): concurrent predictFuture batching equals direct evaluation."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_exe(name="test_nn_service"):
    from alphazero_risk_b200 import build
    build.build()
    src = os.path.join(ROOT, "tests", "host", name + ".cpp")
    exe = os.path.join(ROOT, "tests", "host", name)
    hdrs = [os.path.join(ROOT, "alphazero_risk_b200", "host", h) for h in ("az_nn_service.hpp", "az_play.hpp", "az_cluster.hpp")]
    if not os.path.exists(exe) or os.path.getmtime(exe) < max([os.path.getmtime(src), os.path.getmtime(build.LIB)] + [os.path.getmtime(h) for h in hdrs]):
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-pthread", "-I" + os.path.join(ROOT, "include"),
                               "-I" + os.path.join(ROOT, "alphazero_risk_b200", "host"), src, "-o", exe,
                               "-L" + os.path.join(ROOT, "alphazero_risk_b200"), "-laz_b200",
                               "-Wl,-rpath," + os.path.join(ROOT, "alphazero_risk_b200"), "-Wl,-rpath,$ORIGIN/../../alphazero_risk_b200"])
    return exe


def test_adapter_compiles_and_has_no_cpu_fallback():
    exe = build_exe()
    from alphazero_risk_b200 import api
    if api.lib().az_device_count() > 0:
        pytest.skip("a GPU is present")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and "NO_DEVICE_OK" in out.stdout, out.stdout + out.stderr


@pytest.mark.gpu
def test_adapter_batches_concurrent_requests(tmp_path):
    out = subprocess.run([build_exe(), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "SERVICE_OK" in out.stdout, out.stdout + out.stderr


def test_play_adapter_compiles_and_has_no_cpu_fallback():
    exe = build_exe("test_play")
    from alphazero_risk_b200 import api
    if api.lib().az_device_count() > 0:
        pytest.skip("a GPU is present")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and "NO_DEVICE_OK" in out.stdout, out.stdout + out.stderr


@pytest.mark.gpu
def test_play_adapter_runs_a_match(tmp_path):
    """GameGroup::playGames(az group, script group, 41) through azb200::DevicePlay: 40 games, reproducible tallies"""
    out = subprocess.run([build_exe("test_play"), str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "PLAY_OK" in out.stdout, out.stdout + out.stderr


def test_dist_adapter_compiles_and_has_no_cpu_fallback():
    exe = build_exe("test_dist")
    from alphazero_risk_b200 import api
    if api.lib().az_device_count() > 0:
        pytest.skip("a GPU is present")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and "NO_DEVICE_OK" in out.stdout, out.stdout + out.stderr


@pytest.mark.gpu
def test_dist_weight_broadcast_and_stats_gather_from_cpp():
    """az_dist_* and azb200::DeviceCluster driven from C++ in ONE process (the reference's multi-GPU model): every visible GPU up to
    two; with one GPU the world has a single rank and the same calls must work"""
    out = subprocess.run([build_exe("test_dist")], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "DIST_OK" in out.stdout, out.stdout + out.stderr
