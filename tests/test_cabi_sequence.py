"""tests/cabi/cgo_sequence.c: the call sequence of the (uncompilable here) Go shim go/kgpuscheduler/kgpu_cgo.go as
a plain C99 program against include/kgpu.h + libkgpu.so.
 - not gpu: the header compiles as strict C99 (what cgo's C compiler sees), the program links, and without a
   CUDA device it fails loudly with exit code 3 (no CPU path in the product);
 - gpu: every output of the sequence is checked against the oracle."""
import os
import subprocess

import numpy as np
import pytest

from kubegpu_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cabi", "cgo_sequence.c")
LIBDIR = os.path.join(ROOT, "kubegpu_b200", "lib")


def _build(tmp_path):
    exe = str(tmp_path / "cgo_sequence")
    subprocess.check_call(["gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-O1", "-I", os.path.join(ROOT, "include"),
                           SRC, "-o", exe, "-L", LIBDIR, "-lkgpu", "-Wl,-rpath," + LIBDIR])
    return exe


def _inputs(tmp_path, N=1500, P=96):
    topo, free, pods = synth.gen_c4(N=N, P=P, seed=0xC60)
    free[:12] |= 0x0F                       # the nodes the sequence takes GPUs from have some
    topo.astype(np.int32).tofile(tmp_path / "topo.bin")
    free.astype(np.int32).tofile(tmp_path / "free.bin")
    pods.astype(np.int32).tofile(tmp_path / "pods.bin")
    return topo, free, pods


def test_c99_program_builds_and_fails_loudly_without_gpu(tmp_path):
    if not os.path.exists(os.path.join(LIBDIR, "libkgpu.so")):
        pytest.skip("libkgpu.so not built")
    exe = _build(tmp_path)
    topo, free, pods = _inputs(tmp_path, N=64, P=8)
    r = subprocess.run([exe, str(tmp_path / "topo.bin"), str(tmp_path / "free.bin"), str(tmp_path / "pods.bin"), "64", "8",
                        str(tmp_path / "out.bin")], capture_output=True, text=True, timeout=120,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))      # no device, also on a machine that has one
    assert r.returncode == 3, (r.returncode, r.stderr)
    assert "no usable CUDA device" in r.stderr and not os.path.exists(tmp_path / "out.bin")


@pytest.mark.gpu
def test_cgo_call_sequence_against_oracle(tmp_path, oracle_b):
    exe = _build(tmp_path)
    N, P = 1500, 96
    topo, free, pods = _inputs(tmp_path, N, P)
    r = subprocess.run([exe, str(tmp_path / "topo.bin"), str(tmp_path / "free.bin"), str(tmp_path / "pods.bin"), str(N), str(P),
                        str(tmp_path / "out.bin")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "libkgpu 0.2" in r.stdout and "error path: kgpu_set_free_mask: index 1500 out of range" in r.stdout
    raw = np.fromfile(tmp_path / "out.bin", dtype=np.uint8)
    o = 0

    def take(dtype, n):
        nonlocal o
        a = raw[o:o + n * np.dtype(dtype).itemsize].view(dtype)
        o += n * np.dtype(dtype).itemsize
        return a
    keys1, nk, keys2, keys3, fit, keys4, masks = (take(np.uint64, P), take(np.uint32, 8), take(np.uint64, P), take(np.uint64, P),
                                                   take(np.uint32, 8), take(np.uint64, P), take(np.int32, N))
    assert o == raw.size
    f = free.copy()
    want1 = oracle_b.score_batch(topo, f, pods)
    assert (keys1 == want1).all()
    pair_node = [int(want1[i] >> np.uint64(8)) & 0xFFFFFFFF if want1[i] != np.uint64(0xFFFFFFFFFFFFFFFF) else i for i in range(8)]
    for i in range(8):                      # scorePair == PodFitsDevice(node the batch chose, pod i): same cost and mask
        assert int(nk[i]) == oracle_b.node_key(topo[pair_node[i]], int(f[pair_node[i]]), int(pods[i, 0]))
    if want1[0] != np.uint64(0xFFFFFFFFFFFFFFFF):
        f[pair_node[0]] &= ~int(want1[0] & np.uint64(0xFF))
    assert (keys2 == oracle_b.score_batch(topo, f, pods)).all()
    for i in range(5):                      # the batched Take
        n = 1 + 2 * i
        m = int(f[n]); m &= m - 1; m &= m - 1
        f[n] = m
    assert (keys3 == oracle_b.score_batch(topo, f, pods)).all()
    for i in range(8):                      # fit table after the state changes
        assert int(fit[i]) == oracle_b.node_key(topo[pair_node[i]], int(f[pair_node[i]]), int(pods[i, 0]))
    want4, wf = oracle_b.place_batch(topo, f, pods)
    assert (keys4 == want4).all() and (masks == wf).all()
