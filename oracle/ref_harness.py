"""Stub-import harness: load the UNMODIFIED reference modules
``soundspaces/simulator.py``, ``soundspaces/continuous_simulator.py`` and
``soundspaces/tasks/nav.py`` from a sound-spaces checkout (``SOUNDSPACES_REFERENCE``)
and drive their audio methods on synthetic wav trees.

TEST INFRASTRUCTURE ONLY (see ``oracle/audio_oracle.py``).  Works only where
a reference checkout exists, so only ``tests/golden/make_golden.py`` (fixture
generation) calls :func:`load_reference`; the tests use the recorded fixtures
and the plain helpers (``AttrDict``, ``write_rir``, ``make_discrete_sim``).

habitat / habitat_sim / gym / librosa / skimage are absent and un-installable
here, so they are replaced by inert stubs; ``librosa.stft`` and
``skimage.measure.block_reduce`` are bound to the restatements in
``oracle/audio_oracle.py``.  ``scipy.signal.fftconvolve`` and
``scipy.io.wavfile`` are the genuine dependencies.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("SOUNDSPACES_REFERENCE", "/root/reference")


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "soundspaces", "simulator.py"))


class _Anything:
    """Inert stand-in: attribute access, calls and subclassing all succeed."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Anything()

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Anything()


class _Registry:
    def _reg(self, *args, **kwargs):
        if len(args) == 1 and callable(args[0]) and not kwargs:
            return args[0]
        return lambda cls: cls

    register_simulator = register_sensor = register_measure = _reg
    register_task = register_action_space_configuration = register_dataset = _reg
    register_task_action = _reg


class AttrDict(dict):
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


_LOADED = {}


def load_reference(pad_mode="reflect"):
    """Return dict(simulator=<module>, continuous=<module>, nav=<module>)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if pad_mode in _LOADED:
        return _LOADED[pad_mode]
    from oracle import audio_oracle as ao
    import torch  # noqa: F401  (reference utils.py imports it; load before stubbing)
    import networkx  # noqa: F401

    saved = dict(sys.modules)

    class Base:
        def __init__(self, *a, **k):
            pass

    class Actions:
        STOP, MOVE_FORWARD, TURN_LEFT, TURN_RIGHT = 0, 1, 2, 3

        @staticmethod
        def extend_action_space(name):
            return 4

    _mod("habitat", Config=dict)
    _mod("habitat.core")
    _mod("habitat.core.registry", registry=_Registry())
    _mod("habitat.core.simulator", Simulator=Base, Sensor=Base, SensorSuite=Base,
         AgentState=Base, ShortestPathPoint=Base, Config=dict, Observations=dict,
         SensorTypes=_Anything(), RGBSensor=Base, DepthSensor=Base)
    _mod("habitat.core.dataset", Episode=Base, Dataset=Base)
    _mod("habitat.config", Config=dict)
    _mod("habitat.sims")
    _mod("habitat.sims.habitat_simulator")
    _mod("habitat.sims.habitat_simulator.actions", HabitatSimActions=Actions)
    _mod("habitat.sims.habitat_simulator.habitat_simulator",
         HabitatSimSensor=Base, overwrite_config=lambda *a, **k: None)
    _mod("habitat.tasks")
    _mod("habitat.tasks.nav")
    _mod("habitat.tasks.nav.nav", DistanceToGoal=Base, Measure=Base, EmbodiedTask=Base,
         Success=Base, NavigationEpisode=Base, NavigationTask=Base)
    _mod("habitat.tasks.utils", cartesian_to_polar=lambda *a: (0.0, 0.0))
    _mod("habitat.utils")
    _mod("habitat.utils.geometry_utils", quaternion_from_coeff=_Anything(),
         quaternion_rotate_vector=_Anything())
    hs = _mod("habitat_sim", Configuration=Base, AgentState=Base, Simulator=Base,
              AudioSensorSpec=Base, SensorSpec=Base, SimulatorConfiguration=Base,
              AgentConfiguration=Base)

    def _hs_getattr(name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Anything()

    hs.__getattr__ = _hs_getattr
    _mod("habitat_sim.utils")
    _mod("habitat_sim.utils.common", quat_from_angle_axis=_Anything(),
         quat_from_coeffs=_Anything(), quat_to_angle_axis=_Anything(),
         d3_40_colors_rgb=np.zeros((40, 3), dtype=np.uint8))
    spaces = _mod("gym.spaces", Box=_Anything, Dict=_Anything, Discrete=_Anything)
    _mod("gym", spaces=spaces)
    _mod("librosa", stft=lambda y, **kw: ao.librosa_stft(y, pad_mode=pad_mode, **kw),
         load=_Anything())
    _mod("skimage")
    _mod("skimage.measure",
         block_reduce=lambda a, block_size, func=np.mean: ao.block_reduce_mean(a, block_size))
    if "attr" not in sys.modules:
        try:
            import attr  # noqa: F401
        except Exception:
            _mod("attr", s=lambda *a, **k: (lambda c: c), ib=lambda *a, **k: None)
    if "cv2" not in sys.modules:
        try:
            import cv2  # noqa: F401
        except Exception:
            _mod("cv2")
    if "PIL" not in sys.modules:
        try:
            import PIL.Image  # noqa: F401
        except Exception:
            _mod("PIL", Image=_Anything())
            _mod("PIL.Image")

    pkg = types.ModuleType("soundspaces")
    pkg.__path__ = [os.path.join(REFERENCE_ROOT, "soundspaces")]
    sys.modules["soundspaces"] = pkg
    tpkg = types.ModuleType("soundspaces.tasks")
    tpkg.__path__ = [os.path.join(REFERENCE_ROOT, "soundspaces", "tasks")]
    sys.modules["soundspaces.tasks"] = tpkg

    def load(modname, rel):
        spec = importlib.util.spec_from_file_location(modname, os.path.join(REFERENCE_ROOT, rel))
        m = importlib.util.module_from_spec(spec)
        sys.modules[modname] = m
        spec.loader.exec_module(m)
        return m

    try:
        load("soundspaces.utils", "soundspaces/utils.py")
        load("soundspaces.mp3d_utils", "soundspaces/mp3d_utils.py")
        out = dict(
            simulator=load("soundspaces.simulator", "soundspaces/simulator.py"),
            continuous=load("soundspaces.continuous_simulator", "soundspaces/continuous_simulator.py"),
            nav=load("soundspaces.tasks.nav", "soundspaces/tasks/nav.py"),
        )
    finally:
        # do not leak stubs into the rest of the test session
        for k in list(sys.modules):
            if k not in saved:
                del sys.modules[k]
    _LOADED[pad_mode] = out
    return out


def make_discrete_sim(ref, rir_root, sr, *, dataset="replica", scene="apartment_0",
                      source_sounds=None, current_sound="telephone.wav", receiver=0,
                      source=1, rotation_angle=0, step_count=0, duration=500,
                      distractor=None, distractor_sound=None, audio_index=0):
    """A bare ``SoundSpacesSim`` (no habitat) with just the attributes the audio
    slice reads (SURVEY.md App. D)."""
    Sim = ref["simulator"].SoundSpacesSim
    sim = object.__new__(Sim)
    sim.config = AttrDict(
        USE_RENDERED_OBSERVATIONS=True, SCENE_DATASET=dataset,
        AUDIO=AttrDict(RIR_SAMPLING_RATE=sr, HAS_DISTRACTOR_SOUND=distractor is not None,
                       BINAURAL_RIR_DIR=rir_root, EVERLASTING=True))
    sim._current_scene = f"data/scene_datasets/{dataset}/{scene}/x.glb"
    sim._episode_step_count = step_count
    sim._duration = duration
    sim._rotation_angle = rotation_angle
    sim._receiver_position_index = receiver
    sim._source_position_index = source
    sim._current_sound = current_sound
    sim._source_sound_dict = dict(source_sounds or {})
    sim._audio_index = audio_index
    cur = sim._source_sound_dict[current_sound]
    sim._audio_length = cur.shape[0] // sr
    sim._audiogoal_cache = {}
    sim._spectrogram_cache = {}
    if distractor is not None:
        sim._distractor_position_index = distractor
        sim._current_distractor_sound = distractor_sound
    return sim


def make_continuous_sim(ref, sr, source, rir, *, step_time=0.25, sample_index=0, last_rir=None,
                        crossfade=False, step_count=0, duration=500):
    Sim = ref["continuous"].ContinuousSoundSpacesSim
    sim = object.__new__(Sim)
    sim.config = AttrDict(STEP_TIME=step_time,
                          AUDIO=AttrDict(RIR_SAMPLING_RATE=sr, CROSSFADE=crossfade))
    sim._episode_step_count = step_count
    sim._duration = duration
    sim._current_sound = "s"
    sim._source_sound_dict = {"s": source}
    sim._current_sample_index = sample_index
    sim._prev_sim_obs = {"audio_sensor": np.asarray(rir).T.tolist()}
    sim._last_rir = last_rir
    return sim


def write_rir(rir_root, dataset, scene, azimuth, receiver, source, sr, rir):
    from scipy.io import wavfile
    d = os.path.join(rir_root, dataset, scene, str(azimuth))
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, f"{receiver}_{source}.wav")
    if rir is None:
        with open(path, "wb") as f:      # unreadable -> ValueError in wavfile.read
            f.write(b"not a wav file at all")
    else:
        wavfile.write(path, sr, np.asarray(rir, dtype=np.float32))
    return path
