"""CPU tests of the host side: the overlap-save plan arithmetic against the oracle (through a
numpy model of the kernels' dataflow), the C-ABI library's exported symbols and struct layout,
and the env sharding over a world_size-2 gloo group."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from kernel_model import render_model
from oracle import audio_oracle as ao
from synth import make_rir, make_source

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def close(a, b, tol=1e-9):
    peak = max(np.abs(b).max(), 1e-30)
    assert np.abs(a - b).max() <= tol * peak


@pytest.mark.parametrize("P", [2048, 4096, 8192])
@pytest.mark.parametrize("L", [1, 100, 4096, 4097, 16000, 20000, 47999])
def test_plan_head_mode(P, L):
    sr = 16000
    src, rir = make_source(1, sr).astype(np.float64), make_rir(L, L).astype(np.float64)
    close(render_model(src, rir, sr, P, -(-48000 // P)), ao.compute_audiogoal(src, rir, sr))


@pytest.mark.parametrize("P", [2048, 4096])
@pytest.mark.parametrize("index", [0, 1, 2, 3])
@pytest.mark.parametrize("L", [7001, 20000, 40000])
def test_plan_multisecond(P, index, L):
    sr = 16000
    src, rir = make_source(2, 4 * sr).astype(np.float64), make_rir(L, L).astype(np.float64)
    got = render_model(src, rir, sr, P, -(-48000 // P), offset=index * sr)
    close(got, ao.compute_audiogoal(src, rir, sr, audio_index=index))


@pytest.mark.parametrize("idx", [0, 4000, 12000, 44000, 46000])
def test_plan_continuous(idx):
    sr, P = 16000, 4096
    src, rir = make_source(3, 3 * sr).astype(np.float64), make_rir(9, 9000).astype(np.float64)
    got = render_model(src, rir, sr, P, 12, offset=idx, out_samples=4000, wrap=True)
    close(got, ao.continuous_convolve_with_rir(src, rir, sr, 0.25, idx))


def test_empty_and_fallback():
    sr = 16000
    src = make_source(4, sr).astype(np.float64)
    assert not render_model(src, None, sr, 4096, 4).any()
    assert not ao.compute_audiogoal(src, None, sr).any()


# ---------------------------------------------------------------------------------- C ABI
def header_functions():
    text = open(os.path.join(ROOT, "include", "ssb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ssb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from soundspaces_b200 import _lib
    path = _lib.build_library()
    lib = ctypes.CDLL(path)
    names = header_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/ssb200.h but not exported"
    assert sorted(_lib.EXPORTS) == names, "ctypes prototypes out of sync with the header"
    assert _lib.load_library().ssb_version() >= 100
    assert _lib.load_library().ssb_spec_cols(16000) == 26 and _lib.load_library().ssb_spec_cols(44100) == 69


def test_request_struct_layout_matches_c(tmp_path):
    from soundspaces_b200 import _lib
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ssb200.h"\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(ssb_conv_term), sizeof(ssb_req),'
                   'offsetof(ssb_conv_term, x_offset), offsetof(ssb_conv_term, rir_taps), offsetof(ssb_conv_term, x_wofs),'
                   'offsetof(ssb_req, out_samples), offsetof(ssb_req, flags), sizeof(ssb_plan));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    vals = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    t, r = _lib.TERM_DTYPE, _lib.REQ_DTYPE
    assert vals == [t.itemsize, r.itemsize, t.fields["x_offset"][1], t.fields["rir_taps"][1], t.fields["x_wofs"][1],
                    r.fields["out_samples"][1], r.fields["flags"][1], ctypes.sizeof(_lib.Plan)]


def test_product_has_no_oracle_import_and_no_cpu_fallback():
    pkg = os.path.join(ROOT, "soundspaces_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            text = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in text.replace("no CPU fallback", ""), f"{fn} mentions the oracle"
            assert "fftconvolve" not in text or fn == "simulator.py" or "reference" in text
    import torch
    if not torch.cuda.is_available():
        from soundspaces_b200 import BatchedAudioRenderer
        with pytest.raises(RuntimeError):
            BatchedAudioRenderer(16000, 4096, device="cuda:0")
        with pytest.raises(RuntimeError):
            BatchedAudioRenderer(16000, 4096, device="cpu")


# ---------------------------------------------------------------------------------- sharding
def _gloo_worker(rank, world, port, tmp):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from soundspaces_b200.distributed import gather_observations, shard_envs
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    n_envs = 7
    mine = shard_envs(n_envs, rank, world)
    # fake "rendered" rows: row value = env index
    local = torch.stack([torch.full((65, 3, 2), float(i)) for i in mine]) if mine else torch.zeros((0, 65, 3, 2))
    full = gather_observations(local, n_envs, rank, world)
    assert full.shape == (n_envs, 65, 3, 2)
    assert all(float(full[i, 0, 0, 0]) == float(i) for i in range(n_envs))
    # the same through the pre-allocated gather buffer the kernels write into (in-place all-gather)
    from soundspaces_b200.distributed import GatheredObservations
    g = GatheredObservations(n_envs, (65, 3, 2), rank, world, "cpu")
    assert g.local.is_contiguous() and g.local.shape[0] == len(mine)
    g.local.copy_(local)                                    # stands for execute(out=g.local)
    flat = g.gather()
    assert flat.data_ptr() == g.buffer.data_ptr()           # no staging copy
    for row, env in enumerate(g.env_ids.reshape(-1).tolist()):
        if env < n_envs:
            assert float(flat[row, 0, 0, 0]) == float(env)
    assert torch.equal(g.in_env_order(), full)
    dist.barrier()
    dist.destroy_process_group()
    open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")


def test_shard_and_gather_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    port = 29600 + os.getpid() % 300
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


def test_shard_envs_partition():
    from soundspaces_b200.planning import shard_envs
    for world in (1, 2, 4, 8):
        parts = [shard_envs(13, r, world) for r in range(world)]
        assert sorted(sum(parts, [])) == list(range(13))


# ---------------------------------------------------------------------------------- request preparation
def _host_only_renderer(n_terms=2):
    """A BatchedAudioRenderer with the device parts stubbed out: exercises the host-side request arithmetic
    of prepare() (bank offsets, effective taps, window-set lookups) without CUDA."""
    import torch
    from soundspaces_b200._lib import Plan
    from soundspaces_b200.renderer import BatchedAudioRenderer
    from soundspaces_b200.planning import window_layout
    r = object.__new__(BatchedAudioRenderer)
    r.sr, r.P, r.N, r.max_taps = 16000, 2048, 4096, 20000
    plan = Plan()
    plan.log2n, plan.block, plan.sr, plan.n_blocks, plan.max_parts, plan.n_terms = 12, 2048, 16000, 8, 10, n_terms
    plan.h_elems_per_env = n_terms * 10 * 4096
    r.plan = plan
    r.plan64, r.block64_taps, r.force_block64 = None, 65536 - 16000 + 1, False     # partitioned plan only
    r.device = torch.device("cpu")
    r._bank_index = None
    r._rir_len = [100, 4097, 0, 20000, 9000, 16000]
    r._rir_off = [0, 100, 0, 4197, 24197, 33197]
    calls = []

    def windows(source, offset, wrap, out_samples, block64=False):   # deterministic stand-in for the cached spectra
        assert not block64
        calls.append((source, offset, wrap, out_samples))
        nblk, wofs, nw = window_layout(r.P, plan.max_parts, offset, out_samples)
        return (1000 * source + offset + 7 * int(wrap) + out_samples, nw, wofs)
    r._windows = windows
    return r, calls


def _prepare_reference(r, requests):
    """The per-request loop the vectorised _prepare replaced (same field semantics)."""
    from soundspaces_b200._lib import REQ_DTYPE, SSB_FLAG_SILENT
    from soundspaces_b200.planning import effective_taps
    reqs = np.zeros(len(requests), dtype=REQ_DTYPE)

    def fill(term, rir_id, source, offset, wrap, out_samples):
        if rir_id is None or rir_id < 0 or r._rir_len[rir_id] == 0:
            return
        x_off, nw, wofs = r._windows(source, offset, wrap, out_samples)
        term["rir_offset"], term["x_offset"] = r._rir_off[rir_id], x_off
        term["rir_taps"] = effective_taps(r._rir_len[rir_id], offset, out_samples)
        term["x_nw"], term["x_wofs"] = nw, wofs
    for i, q in enumerate(requests):
        outs = r.sr if q.out_samples is None else int(q.out_samples)
        reqs[i]["out_samples"] = outs
        if q.silent:
            reqs[i]["flags"] = SSB_FLAG_SILENT
            continue
        fill(reqs[i]["term"][0], q.rir, q.source, int(q.offset), q.wrap, outs)
        if q.distractor_source is not None:
            fill(reqs[i]["term"][1], q.distractor_rir, q.distractor_source, 0, False, outs)
    return reqs


def test_prepare_vectorised_matches_per_request_loop():
    from soundspaces_b200 import AudioRequest
    rng = np.random.default_rng(3)
    r, calls = _host_only_renderer()
    reqs = []
    for i in range(200):
        reqs.append(AudioRequest(
            rir=[0, 1, 2, 3, 4, 5, -1, None][rng.integers(8)], source=int(rng.integers(3)),
            offset=int(rng.choice([0, 0, 0, 16000, 32000, 8000, 12345])),
            out_samples=[None, None, 4000, 16000, 1][rng.integers(5)], wrap=bool(rng.integers(2)),
            silent=bool(rng.random() < 0.1),
            distractor_rir=[None, 1, 2, 4][rng.integers(4)], distractor_source=[None, None, 0, 2][rng.integers(4)]))
    got = r._prepare(reqs)
    n_vec = len(calls)
    del calls[:]
    ref = _prepare_reference(r, reqs)
    assert got.n == 200 and got.reqs_host.dtype == ref.dtype
    assert got.reqs_host.tobytes() == ref.tobytes()                       # identical, byte for byte
    assert bytes(got.reqs_dev.numpy()) == ref.tobytes()
    assert n_vec <= 2 * len(set(calls)) and n_vec < len(calls)            # one lookup per distinct window set and term
    # empty batch, all-silent batch
    assert r._prepare([]).n == 0
    z = r._prepare([AudioRequest(rir=0, source=0, silent=True)] * 3).reqs_host
    assert (z["flags"] == 1).all() and not z["term"]["rir_taps"].any()


def test_prepare_errors_like_before():
    from soundspaces_b200 import AudioRequest
    r, _ = _host_only_renderer(n_terms=1)
    with pytest.raises(ValueError, match="unknown RIR id"):
        r._prepare([AudioRequest(rir=0, source=0), AudioRequest(rir=6, source=0)])
    with pytest.raises(ValueError, match="out_samples"):
        r._prepare([AudioRequest(rir=0, source=0, out_samples=0)])
    with pytest.raises(ValueError, match="out_samples"):
        r._prepare([AudioRequest(rir=0, source=0, out_samples=16001)])
    with pytest.raises(ValueError, match="n_terms=1"):
        r._prepare([AudioRequest(rir=0, source=0, distractor_rir=1, distractor_source=0)])
    r.plan.max_parts = 4                                                  # 8192 taps: RIR 3 (20000, cut to 16000) no longer fits
    with pytest.raises(ValueError, match="RIR 3 needs 16000 taps"):
        r._prepare([AudioRequest(rir=1, source=0), AudioRequest(rir=3, source=0)])
    # the bank index follows the bank
    r.plan.max_parts = 10
    a = r._prepare([AudioRequest(rir=4, source=0)]).reqs_host["term"][0, 0]
    assert a["rir_offset"] == 24197 and a["rir_taps"] == 9000
    r._rir_off[4], r._rir_len[4] = 5, 50
    r._bank_index = None                                                  # what every bank mutation does
    a = r._prepare([AudioRequest(rir=4, source=0)]).reqs_host["term"][0, 0]
    assert a["rir_offset"] == 5 and a["rir_taps"] == 50


def test_prepare_arrays_equals_prepare():
    from soundspaces_b200 import AudioRequest
    r, _ = _host_only_renderer()
    rir = np.array([0, 1, -1, 3, 4, 5, 2, 1])
    off = np.array([0, 16000, 0, 0, 8000, 0, 0, 32000])
    sil = np.array([0, 0, 0, 1, 0, 0, 0, 0], dtype=bool)
    drir = np.array([-1, 4, -1, -1, -1, 1, -1, -1])
    dsrc = np.array([-1, 2, -1, -1, -1, 0, -1, -1])
    a = r.prepare_arrays(rir, 1, offset=off, silent=sil, distractor_rir=drir, distractor_source=dsrc)
    b = r.prepare([AudioRequest(rir=int(rir[i]), source=1, offset=int(off[i]), silent=bool(sil[i]),
                                distractor_rir=None if drir[i] < 0 else int(drir[i]),
                                distractor_source=None if dsrc[i] < 0 else int(dsrc[i])) for i in range(8)])
    assert a.n == 8 and a.reqs_host.tobytes() == b.reqs_host.tobytes()
    assert r.prepare_arrays(np.arange(3), 0, out_samples=4000).reqs_host["out_samples"].tolist() == [4000] * 3


# ---------------------------------------------------------------------------------- bench.py timed_region across ranks
def _timed_region_worker(rank, world, port, tmp):
    """Two gloo ranks of different speed: each times exactly the K steps it was asked for, once, between barriers
    (any extra region on one rank alone would leave the other waiting in a barrier)."""
    import time
    import types
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    import bench

    class FakeEvent:
        def __init__(self, enable_timing=True):
            self.t = None

        def record(self):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3
    fake_torch = types.SimpleNamespace(cuda=types.SimpleNamespace(Event=FakeEvent))
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    calls = []

    def step(i):
        calls.append(i)
        time.sleep(0.0015 if rank == 0 else 0.0004)          # rank 0: 15 ms per region, rank 1: 4 ms
    ms = bench.timed_region(step, 10, dist.barrier, fake_torch)
    open(os.path.join(tmp, f"region{rank}"), "w").write(json.dumps({"calls": calls, "ms": ms}))
    dist.barrier()
    dist.destroy_process_group()


def test_bench_timed_region_times_exactly_k_steps_on_every_rank(tmp_path):
    import torch.multiprocessing as mp
    port = 29300 + os.getpid() % 300
    mp.spawn(_timed_region_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = (json.loads(open(tmp_path / f"region{k}").read()) for k in (0, 1))
    assert r0["calls"] == r1["calls"] == list(range(10))
    assert r0["ms"] >= 15.0 and r1["ms"] >= 4.0
