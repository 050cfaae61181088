"""CPU tests of the host logic behind the per-env plugin surface (no CUDA: a stand-in renderer records the
launches): the deferred-handle batcher and its ring, the ``batch_obs`` replacement, the scene-safe memo of
``VectorAudioObservations``, the RIR service (prefetch, misses, LRU compaction), the continuous simulator's
wrap rule, and ``patch_simulator`` applied to classes with the REAL reference classes' members."""
import gc
import json
import os
import time

import numpy as np
import pytest
import torch

from oracle.ref_harness import AttrDict, write_rir
from stubs import StubRenderer
from synth import make_rir, make_source

from soundspaces_b200.batching import AudioObservationBatcher, DeferredObservation
from soundspaces_b200.renderer import AudioRequest
from soundspaces_b200.simulator import (AudioRenderService, B200AudioMixin, B200ContinuousAudioMixin, CONTINUOUS_READS,
                                        DISCRETE_READS, patch_simulator)


def make_service(sr=16000, **kw):
    return AudioRenderService(sr, renderer=StubRenderer(sr), **kw)


class FakeSim(B200AudioMixin):
    scene = "apartment_0"

    @property
    def binaural_rir_dir(self):
        return os.path.join(self.config.AUDIO.BINAURAL_RIR_DIR, self.config.SCENE_DATASET, self.scene)

    @property
    def current_source_sound(self):
        return self._source_sound_dict[self._current_sound]

    @property
    def azimuth_angle(self):
        return -(self._rotation_angle + 0) % 360


def make_sim(svc, rir_root, sr, src, receiver=0, source=1, scene="apartment_0", deferred=True):
    sim = FakeSim()
    sim.scene = scene
    sim.b200_deferred = deferred
    sim._b200_svc = svc
    sim.config = AttrDict(USE_RENDERED_OBSERVATIONS=True, SCENE_DATASET="replica",
                          AUDIO=AttrDict(RIR_SAMPLING_RATE=sr, HAS_DISTRACTOR_SOUND=False, BINAURAL_RIR_DIR=rir_root))
    sim._episode_step_count, sim._duration, sim._rotation_angle = 0, 500, 0
    sim._receiver_position_index, sim._source_position_index = receiver, source
    sim._current_sound, sim._source_sound_dict = "telephone.wav", {"telephone.wav": src}
    sim._audio_index, sim._audio_length = 0, src.shape[0] // sr
    sim._audiogoal_cache, sim._spectrogram_cache = {}, {}
    return sim


# ---------------------------------------------------------------------------------- batcher
def test_batcher_one_render_per_step_and_zero_copy_view():
    svc = make_service()
    b = AudioObservationBatcher(svc, capacity=16)
    svc.renderer.add_rirs([np.zeros((10, 2), np.float32)] * 8)
    hs = [b.enqueue(AudioRequest(rir=i, source=0)) for i in range(5)]
    assert all(h.pending for h in hs) and not svc.renderer.renders
    t = b.gather(hs)
    assert len(svc.renderer.renders) == 1 and len(svc.renderer.renders[0]) == 5          # ONE render for the step
    assert t.shape == (5, 65, 26, 2) and t.data_ptr() == b.ring.data_ptr()              # a view of the ring
    assert [float(t[i, 0, 0, 0]) for i in range(5)] == [0.0, 1000.0, 2000.0, 3000.0, 4000.0]
    assert not any(h.pending for h in hs)
    # host compat: np.asarray(handle) is the array the reference's sensor would have returned
    a = np.asarray(hs[3])
    assert isinstance(a, np.ndarray) and a.shape == (65, 26, 2) and a.dtype == np.float32 and a[0, 0, 0] == 3000.0
    # next step: rows follow on in the ring, again one render
    hs2 = [b.enqueue(AudioRequest(rir=i, source=0)) for i in (7, 6)]
    t2 = b.gather(hs2)
    assert len(svc.renderer.renders) == 2 and float(t2[0, 0, 0, 0]) == 7000.0 and hs2[0].slot == 5
    # out-of-order / mixed generations: a gathered copy with the right rows
    mix = b.gather([hs2[1], hs[0], hs[4]])
    assert [float(mix[i, 0, 0, 0]) for i in range(3)] == [6000.0, 0.0, 4000.0]


def test_batcher_render_into_rollout_slot():
    svc = make_service()
    b = AudioObservationBatcher(svc, capacity=16)
    svc.renderer.add_rirs([np.zeros((10, 2), np.float32)] * 4)
    hs = [b.enqueue(AudioRequest(rir=i, source=0)) for i in range(4)]
    slot = torch.full((4, 65, 26, 2), -1.0)
    got = b.gather(hs, out=slot)
    assert got is slot and [float(slot[i, 0, 0, 0]) for i in range(4)] == [0.0, 1000.0, 2000.0, 3000.0]
    assert torch.equal(b.gather(hs), slot)                       # the handles still resolve (ring rows were filled too)


def test_ring_reuse_detaches_live_handles_only():
    svc = make_service()
    b = AudioObservationBatcher(svc, capacity=4)
    svc.renderer.add_rirs([np.zeros((10, 2), np.float32)] * 20)
    kept = b.enqueue(AudioRequest(rir=1, source=0))              # e.g. memoised in a simulator's _spectrogram_cache
    dropped = b.enqueue(AudioRequest(rir=2, source=0))
    b.flush()
    dropped_slot = dropped.slot
    del dropped
    gc.collect()
    for step in range(3):                                         # wraps around the 4-row ring
        hs = [b.enqueue(AudioRequest(rir=10 + 2 * step + j, source=0)) for j in range(2)]
        b.gather(hs)
    assert kept._row is not None                                  # detached: private copy taken before slot reuse
    assert float(kept.resolve()[0, 0, 0]) == 1000.0               # ... and still its own observation
    assert float(b.ring[kept.slot][0, 0, 0]) != 1000.0            # the ring row itself has been reused
    assert b._owners[dropped_slot]() is not kept


# ---------------------------------------------------------------------------------- batch_obs
def test_batch_obs_replacement_matches_reference_semantics():
    from soundspaces_b200.sensors import batch_obs
    svc = make_service()
    b = svc.batcher
    svc.renderer.add_rirs([np.zeros((10, 2), np.float32)] * 3)
    obs = [{"spectrogram": b.enqueue(AudioRequest(rir=i, source=0)), "pointgoal": np.array([i, -i], np.float64),
            "depth": np.full((2, 2, 1), i, np.float32), "skip_me": np.zeros(3)} for i in range(3)]
    batch = batch_obs(obs, device=torch.device("cpu"), skip_list=["skip_me"])
    assert set(batch) == {"spectrogram", "pointgoal", "depth"}
    assert batch["spectrogram"].shape == (3, 65, 26, 2) and batch["spectrogram"].dtype == torch.float32
    assert batch["pointgoal"].dtype == torch.float32 and batch["pointgoal"].tolist() == [[0, 0], [1, -1], [2, -2]]
    assert batch["depth"].shape == (3, 2, 2, 1)
    assert len(svc.renderer.renders) == 1
    # reference-style host arrays still work, and `out` receives the batch in place
    dst = {"spectrogram": torch.empty((3, 65, 26, 2))}
    host = [{"spectrogram": np.full((65, 26, 2), i, np.float64)} for i in range(3)]
    got = batch_obs(host, out=dst)
    assert got["spectrogram"].data_ptr() == dst["spectrogram"].data_ptr() and float(got["spectrogram"][2, 0, 0, 0]) == 2.0


# ---------------------------------------------------------------------------------- scene-safe memo
def test_vector_collect_memo_is_per_scene(tmp_path):
    """ADVICE r1 (high): equal (source, receiver, azimuth) indices in ANOTHER scene must not hit the memo."""
    from soundspaces_b200.sensors import VectorAudioObservations
    sr = 16000
    src = make_source(0, sr)
    d = str(tmp_path)
    for scene, seed in (("apartment_0", 1), ("office_3", 2)):
        for recv in range(2):
            write_rir(d, "replica", scene, 0, recv, 1, sr, make_rir(seed * 10 + recv, 200 + 100 * seed))
    svc = make_service(sr)
    vec = VectorAudioObservations.__new__(VectorAudioObservations)
    vec.service, vec.renderer, vec.batcher = svc, svc.renderer, svc.batcher
    sims = [make_sim(svc, d, sr, src, receiver=i) for i in range(2)]
    a = vec.collect(sims).clone()
    assert len(svc.renderer.renders) == 1
    again = vec.collect(sims)
    assert len(svc.renderer.renders) == 1 and torch.equal(a, again)          # memo hits: nothing rendered
    # new episode in another scene, SAME node indices: the reference replaces both memo dicts (simulator.py:395-397)
    for s in sims:
        s.scene = "office_3"
        s._audiogoal_cache, s._spectrogram_cache = dict(), dict()
    b = vec.collect(sims)
    assert len(svc.renderer.renders) == 2, "scene change must re-render"
    ids_a = [q.rir for q in svc.renderer.renders[0]]
    ids_b = [q.rir for q in svc.renderer.renders[1]]
    assert set(ids_a).isdisjoint(ids_b)
    assert svc.renderer._rir_len[ids_a[0]] == 300 and svc.renderer._rir_len[ids_b[0]] == 400
    assert not torch.equal(a, b)


def test_multisecond_memo_hit_does_not_advance_audio_index(tmp_path):
    sr = 16000
    src = make_source(0, 3 * sr)
    write_rir(str(tmp_path), "replica", "apartment_0", 0, 0, 1, sr, make_rir(1, 300))
    svc = make_service(sr)
    sim = make_sim(svc, str(tmp_path), sr, src)
    h1 = sim._b200_deferred_spectrogram()
    assert sim._audio_index == 1
    assert sim._b200_deferred_spectrogram() is h1 and sim._audio_index == 1    # simulator.py:683-686 quirk
    sim._receiver_position_index = 5                                          # (file missing -> zero RIR, still a request)
    write_rir(str(tmp_path), "replica", "apartment_0", 0, 5, 1, sr, make_rir(2, 300))
    h2 = sim._b200_deferred_spectrogram()
    assert h2 is not h1 and sim._audio_index == 2
    svc.batcher.flush()
    assert [q.offset for q in svc.renderer.renders[0]] == [0, sr]


# ---------------------------------------------------------------------------------- RIR service (N1)
def test_service_prefetch_hits_misses_and_lru_compaction(tmp_path):
    sr = 16000
    d = os.path.join(str(tmp_path), "replica", "apartment_0")
    for recv in range(6):
        write_rir(str(tmp_path), "replica", "apartment_0", 0, recv, 1, sr, make_rir(recv, 1000))
    svc = make_service(sr, max_bank_bytes=4 * 1000 * 8)
    k = [(d, 0, recv, 1) for recv in range(6)]
    rid0 = svc.rir(k[0])
    assert svc.stats["misses"] == 1 and svc.renderer._rir_len[rid0] == 1000
    assert svc.rir(k[0]) == rid0 and svc.stats["hits"] == 1
    svc.prefetch([k[1], k[2], k[0]])                       # k[0] is resident: not re-read
    assert set(svc._inflight) == {k[1], k[2]}
    t0 = time.time()
    while not all(f.done() for f in svc._inflight.values()) and time.time() - t0 < 10:
        time.sleep(0.01)
    svc.maybe_trim()                                       # between steps: lands the prefetches in one batched upload
    assert not svc._inflight and svc.stats["prefetched"] == 2
    svc.rir(k[1]); svc.rir(k[2])
    assert svc.stats["misses"] == 1 and svc.stats["hits"] == 3
    svc.prefetch([k[3]])
    svc.rir(k[3])                                          # asked for while (possibly) still in flight: waits, no second read
    assert svc.stats["misses"] + svc.stats["waited"] + svc.stats["hits"] == 5 and k[3] in svc._rir_ids
    # unreadable / missing files are the zero-RIR fallback (simulator.py:617-624), not an exception
    assert svc.renderer._rir_len[svc.rir((d, 0, 99, 1))] == 0
    # budget: 4 RIRs; touching 5 + 6 pushes the bank over -> the least recently used are dropped, the rest compacted
    svc.rir(k[4]); svc.rir(k[5])
    assert svc.renderer.bank_bytes > svc.max_bank_bytes
    svc.maybe_trim()
    assert svc.stats["compactions"] == 1 and svc.renderer.bank_bytes <= svc.max_bank_bytes // 2 + 8000
    assert k[5] in svc._rir_ids and k[0] not in svc._rir_ids
    assert svc.renderer._rir_len[svc._rir_ids[k[5]]] == 1000
    assert 0.0 < svc.miss_rate < 1.0


def test_prefetch_targets_follow_the_action_space(tmp_path):
    """simulator.py:496-516: the next observation is at a graph neighbour (same heading) or at the same node turned
    by +-90 degrees -- exactly those files are read ahead."""
    import networkx as nx
    sr = 16000
    src = make_source(0, sr)
    write_rir(str(tmp_path), "replica", "apartment_0", 90, 3, 1, sr, make_rir(1, 100))
    svc = make_service(sr, prefetch_workers=1)
    sim = make_sim(svc, str(tmp_path), sr, src, receiver=3)
    sim._rotation_angle = 270                              # azimuth 90
    sim.graph = nx.Graph([(3, 4), (3, 7), (4, 8)])
    asked = []
    svc.prefetch = lambda keys: asked.extend(keys)
    sim._b200_request()
    d = sim.binaural_rir_dir
    assert sorted(asked) == sorted([(d, 180, 3, 1), (d, 0, 3, 1), (d, 90, 4, 1), (d, 90, 7, 1)])


# ---------------------------------------------------------------------------------- continuous simulator
def test_continuous_wrap_only_in_steady_state_branch():
    """continuous_simulator.py:433-445 (ADVICE r1): the early branch (index < len(rir)) sees zeros past the clip."""
    class Sim(B200ContinuousAudioMixin):
        @property
        def current_source_sound(self):
            return self._source_sound_dict[self._current_sound]
    sr = 16000
    sim = Sim()
    sim._b200_svc = make_service(sr)
    sim.config = AttrDict(STEP_TIME=0.25, AUDIO=AttrDict(RIR_SAMPLING_RATE=sr, CROSSFADE=True))
    sim._current_sound, sim._source_sound_dict = "s", {"s": make_source(0, sr)}
    sim._prev_sim_obs = {"audio_sensor": np.zeros((2, 9000)).tolist()}
    sim._last_rir = np.zeros((20000, 2))
    sim._current_sample_index = 14000
    cur, prev = sim._b200_requests()
    assert cur.wrap is True and prev.wrap is False          # 14000 >= 9000 taps, but 14000 < 20000 taps
    assert cur.offset == prev.offset == 14000 and cur.out_samples == 4000


# ---------------------------------------------------------------------------------- the real reference classes
def reference_stand_in(name):
    """A class with every member name of the reference's simulator class ``name`` (recorded from the unmodified
    reference by tests/golden/make_golden.py), each a placeholder of its kind, and the recorded facts."""
    with open(os.path.join(os.path.dirname(__file__), "golden", "reference_classes.json")) as f:
        facts = json.load(f)[name]

    def placeholder(self, *a, **k):
        raise AssertionError("reference member called")
    ns = {n: property(placeholder) if kind == "property" else placeholder if kind == "function" else object()
          for n, kind in facts["members"].items()}
    return type("Patched" + name, (), ns), facts


def test_patch_simulator_on_reference_classes():
    """INTEGRATION.md advertises ``patch_simulator(SoundSpacesSim)``: apply it to classes with the REAL classes' members
    with the renderer stubbed; exactly the three audio methods are replaced, everything the replacements read exists on
    the reference object, and the patched object renders through the service."""
    Sim, facts = reference_stand_in("SoundSpacesSim")
    CSim, cfacts = reference_stand_in("ContinuousSoundSpacesSim")
    before = {n: getattr(Sim, n) for n in facts["members"]}
    patch_simulator(Sim, deferred=True)
    patch_simulator(CSim, continuous=True)
    changed = sorted(n for n, v in before.items() if getattr(Sim, n) is not v)
    assert changed == ["_compute_audiogoal", "get_current_audiogoal_observation", "get_current_spectrogram_observation"]
    added = sorted(n for n in dir(Sim) if n not in before and not n.startswith("__"))
    assert all(n.startswith(("_b200", "b200_")) or n == "get_current_audiogoal_device" for n in added), added
    # every attribute the patched methods read is provided by the reference class or set by its __init__/reconfigure
    for name in DISCRETE_READS:
        assert name in facts["members"] or name in facts["self_attributes"], name
    for name in CONTINUOUS_READS:
        assert name in cfacts["members"] or name in cfacts["self_attributes"], name

    # drive a patched object (bare instance, App. D attributes) through the service with the renderer stubbed; the
    # properties the replacements read return what the reference's own properties returned on the same bare object
    bare = facts["bare_object"]
    Sim.binaural_rir_dir = property(lambda s: os.path.join(s.config.AUDIO.BINAURAL_RIR_DIR, bare["binaural_rir_dir_under_root"]))
    Sim.azimuth_angle = property(lambda s: bare["azimuth_angle_by_rotation"][str(s._rotation_angle)])
    Sim.current_source_sound = property(lambda s: s._source_sound_dict[s._current_sound])
    import tempfile
    import types
    from oracle import ref_harness
    sr = 16000
    with tempfile.TemporaryDirectory() as d:
        write_rir(d, "replica", "apartment_0", 0, 0, 1, sr, make_rir(3, 500))
        ref = {"simulator": types.SimpleNamespace(SoundSpacesSim=Sim)}
        sim = ref_harness.make_discrete_sim(ref, d, sr, source_sounds={"telephone.wav": make_source(1, sr)})
        svc = make_service(sr)
        sim._b200_svc = svc
        sim.graph = None
        h = sim.get_current_spectrogram_observation(_native())
        assert isinstance(h, DeferredObservation) and h.pending
        assert sim.get_current_spectrogram_observation(_native()) is h         # memo in the reference's own dict
        assert sim._spectrogram_cache[(1, 0, 0)] is h
        np.asarray(h)
        assert len(svc.renderer.renders) == 1 and svc.renderer._rir_len[svc.renderer.renders[0][0].rir] == 500


def _native():
    from soundspaces_b200.sensors import SpectrogramSensor
    return SpectrogramSensor.compute_spectrogram
