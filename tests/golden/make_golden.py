"""Generate the reference fixtures under tests/golden/ by running the UNMODIFIED
reference (``soundspaces/{simulator,continuous_simulator,tasks/nav}.py`` of a
sound-spaces checkout, located by ``SOUNDSPACES_REFERENCE``) through
``oracle/ref_harness.py`` on seeded synthetic wav trees:

    SOUNDSPACES_REFERENCE=<sound-spaces checkout> python tests/golden/make_golden.py

The fixtures hold the reference's own outputs (``reference_golden.npz``:
spectrograms and metadata, ``reference_golden_waves.npz``: waveforms,
``reference_classes.json``: the member names of its simulator classes);
``tests/test_oracle_golden.py`` pins ``oracle/audio_oracle.py`` to them and the
GPU parity tests compare the CUDA path against the same arrays.  The tests need
only these files, never the reference itself.
"""
import inspect
import json
import os
import re
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ref_harness as rh  # noqa: E402
from synth import make_rir, make_source  # noqa: E402

# name -> dict(kind, params).  Inputs are regenerated from the seeds by the tests.
DISCRETE_CASES = {
    # A2: 1-s clip, full conv, keep [:sr]
    "a2_16k": dict(sr=16000, S=16000, L=5000, seed=1),
    "a2_16k_longrir": dict(sr=16000, S=16000, L=48000, seed=2),      # L > sr: only first sr taps matter
    "a2_44k": dict(sr=44100, S=44100, L=16384, seed=3),
    "a2_44k_odd": dict(sr=44100, S=44100, L=22050, seed=4),
    # A3 / A4: multi-second clip
    "a3_early": dict(sr=16000, S=64000, L=20000, seed=5, audio_index=1),   # 1*sr - L < 0
    "a3_first": dict(sr=16000, S=64000, L=20000, seed=5, audio_index=0),
    "a4_valid": dict(sr=16000, S=64000, L=20000, seed=5, audio_index=2),   # 2*sr - L >= 0
    "a4_valid_last": dict(sr=16000, S=64000, L=7001, seed=6, audio_index=3),
    # A5
    "a5_distractor": dict(sr=16000, S=16000, L=6000, seed=7, distractor=dict(S=24000, L=9000, seed=70)),
    "a5_unreadable": dict(sr=16000, S=16000, L=0, seed=8, rir_mode="unreadable"),
    "a5_empty": dict(sr=16000, S=16000, L=0, seed=9, rir_mode="empty"),
    "a5_silent": dict(sr=16000, S=16000, L=5000, seed=10, step_count=501),
    # azimuth addressing: rotation 90 -> azimuth 270
    "a6_azimuth": dict(sr=16000, S=16000, L=3000, seed=11, rotation_angle=90),
}

CONTINUOUS_CASES = {
    "a7_early": dict(sr=16000, S=48000, L=9000, seed=20, sample_index=4000),
    "a7_steady": dict(sr=16000, S=48000, L=9000, seed=21, sample_index=12000),
    "a7_wrap": dict(sr=16000, S=48000, L=9000, seed=22, sample_index=46000),
    "a7_crossfade": dict(sr=16000, S=48000, L=9000, seed=23, sample_index=20000, last_seed=230, last_L=7000),
    "a7_crossfade_early": dict(sr=16000, S=48000, L=9000, seed=24, sample_index=0, last_seed=240, last_L=9000),
    "a7_silent": dict(sr=16000, S=48000, L=9000, seed=25, sample_index=8000, step_count=501),
}


# round 2: the continuous simulator's EARLY branch with a window that runs past the end of the clip
# (continuous_simulator.py:433-437: the clip is NOT wrapped there -- zeros past its end); kept in a second file so that the
# round-1 fixture stays byte-identical
CONTINUOUS_EDGE_CASES = {
    "a7_early_past_clip_end": dict(sr=16000, S=15000, L=14000, seed=26, sample_index=12000),
    "a7_early_past_clip_end_crossfade": dict(sr=16000, S=15000, L=14000, seed=27, sample_index=12000, last_seed=270, last_L=5000),
}


# one 3-s clip x 21000-tap RIR at azimuth 180, mp3d layout, rendered at each audio index: the oracle must reproduce the
# reference bit for bit (tests/test_oracle_golden.py::test_oracle_vs_reference_outputs)
AUDIO_INDEX_CASE = dict(sr=16000, S=48000, L=21000, seed=77, dataset="mp3d", scene="sc", rotation_angle=180,
                        receiver=4, source=9, audio_indices=(0, 1, 2))

# the waveforms a test feeds back in as input are stored whole; every other discrete waveform as every 5th sample
# (the spectrogram of every case is stored whole)
FULL_WAVES = ("a2_16k/wave",)


def discrete_inputs(c):
    src = make_source(c["seed"], c["S"])
    rir = make_rir(c["seed"], c["L"]) if c["L"] > 0 else None
    d = c.get("distractor")
    dsrc = make_source(d["seed"], d["S"]) if d else None
    drir = make_rir(d["seed"], d["L"]) if d else None
    return src, rir, dsrc, drir


def continuous_inputs(c):
    src = make_source(c["seed"], c["S"])
    rir = make_rir(c["seed"], c["L"]).astype(np.float64)       # habitat-sim lists -> float64 (:419)
    last = make_rir(c["last_seed"], c["last_L"]).astype(np.float64) if "last_seed" in c else None
    return src, rir, last


def reference_class_facts(ref):
    """What ``patch_simulator`` meets in the reference's two simulator classes: every member name (with its kind), every
    ``self.<name>`` their module mentions (attributes set by ``__init__`` / ``reconfigure``), and for the discrete class
    the values its own properties return on the bare object ``ref_harness.make_discrete_sim`` builds."""
    facts = {}
    for key, mod in (("SoundSpacesSim", ref["simulator"]), ("ContinuousSoundSpacesSim", ref["continuous"])):
        cls = getattr(mod, key)
        members = {}
        for n in dir(cls):
            if not n.startswith("__"):
                v = inspect.getattr_static(cls, n)
                members[n] = "property" if isinstance(v, property) else "function" if inspect.isfunction(v) else "other"
        with open(mod.__file__) as f:
            self_attrs = sorted(set(re.findall(r"self\.(\w+)", f.read())))
        facts[key] = {"members": members, "self_attributes": self_attrs}
    root = os.path.join("rir", "root")
    clip = np.zeros(16000, np.float32)
    sims = {rot: rh.make_discrete_sim(ref, root, 16000, source_sounds={"telephone.wav": clip}, rotation_angle=rot)
            for rot in (0, 90, 180, 270)}
    assert all(s.current_source_sound is clip for s in sims.values())
    facts["SoundSpacesSim"]["bare_object"] = {
        "binaural_rir_dir_under_root": os.path.relpath(sims[0].binaural_rir_dir, root),
        "azimuth_angle_by_rotation": {str(rot): int(s.azimuth_angle) for rot, s in sims.items()}}
    return facts


def main():
    out = {}
    for pad_mode in ("reflect", "constant"):
        ref = rh.load_reference(pad_mode)
        spec_fn = ref["nav"].SpectrogramSensor.compute_spectrogram
        for name, c in DISCRETE_CASES.items():
            src, rir, dsrc, drir = discrete_inputs(c)
            sr = c["sr"]
            rot = c.get("rotation_angle", 0)
            with tempfile.TemporaryDirectory() as d:
                sounds = {"telephone.wav": src}
                kw = {}
                azimuth = -(rot) % 360
                if c.get("rir_mode") == "unreadable":
                    rh.write_rir(d, "replica", "apartment_0", azimuth, 0, 1, sr, None)
                elif c.get("rir_mode") == "empty":
                    rh.write_rir(d, "replica", "apartment_0", azimuth, 0, 1, sr, np.zeros((0, 2), np.float32))
                else:
                    rh.write_rir(d, "replica", "apartment_0", azimuth, 0, 1, sr, rir)
                if dsrc is not None:
                    sounds["distractor.wav"] = dsrc
                    rh.write_rir(d, "replica", "apartment_0", azimuth, 0, 2, sr, drir)
                    kw = dict(distractor=2, distractor_sound="distractor.wav")
                sim = rh.make_discrete_sim(ref, d, sr, source_sounds=sounds, rotation_angle=rot,
                                           step_count=c.get("step_count", 0),
                                           audio_index=c.get("audio_index", 0), **kw)
                assert sim.azimuth_angle == azimuth
                wave = sim.get_current_audiogoal_observation()
                if dsrc is None:
                    spec = sim.get_current_spectrogram_observation(spec_fn)
                else:  # distractor path recomputes (no cache); call the sensor fn on the same wave
                    spec = spec_fn(wave)
                if pad_mode == "reflect":
                    out[f"{name}/wave"] = wave
                    out[f"{name}/wave_dtype"] = np.array(str(wave.dtype))
                    out[f"{name}/audio_index_after"] = np.array(sim._audio_index)
                out[f"{name}/spec_{pad_mode}"] = spec
                out[f"{name}/spec_dtype"] = np.array(str(spec.dtype))
        for name, c in CONTINUOUS_CASES.items():
            src, rir, last = continuous_inputs(c)
            sim = rh.make_continuous_sim(ref, c["sr"], src, rir, sample_index=c["sample_index"],
                                         last_rir=last, crossfade=last is not None,
                                         step_count=c.get("step_count", 0))
            wave = sim.get_current_audiogoal_observation()
            spec = sim.get_current_spectrogram_observation(spec_fn)
            if pad_mode == "reflect":
                out[f"{name}/wave"] = wave
                out[f"{name}/wave_dtype"] = np.array(str(wave.dtype))
            out[f"{name}/spec_{pad_mode}"] = spec
        # observation-space probe (nav.py:77) and shapes
        for sr in (16000, 44100, 48000):
            out[f"ones_{sr}/spec_{pad_mode}"] = spec_fn(np.ones((2, sr)))

    # res/singing.wav (the only audio fixture in the reference repo): 1-s int16 excerpt
    from scipy.io import wavfile
    fs, sing = wavfile.read(os.path.join(rh.REFERENCE_ROOT, "res", "singing.wav"))
    assert fs == 48000 and sing.dtype == np.int16 and sing.shape == (233873,)
    excerpt = sing[48000:96000].copy()
    out["singing/pcm16"] = excerpt
    out["singing/meta"] = np.array([fs, sing.shape[0], int(sing.min()), int(sing.max())])
    ref = rh.load_reference("reflect")
    x = excerpt.astype(np.float32) / np.float32(32768.0)
    rir = make_rir(99, 12000)
    with tempfile.TemporaryDirectory() as d:
        rh.write_rir(d, "replica", "apartment_0", 0, 0, 1, 48000, rir)
        sim = rh.make_discrete_sim(ref, d, 48000, source_sounds={"telephone.wav": x})
        out["singing/wave"] = sim.get_current_audiogoal_observation()
        out["singing/spec_reflect"] = sim.get_current_spectrogram_observation(
            ref["nav"].SpectrogramSensor.compute_spectrogram)

    c = AUDIO_INDEX_CASE
    src, rir = make_source(c["seed"], c["S"]), make_rir(c["seed"], c["L"])
    azimuth = -c["rotation_angle"] % 360
    with tempfile.TemporaryDirectory() as d:
        rh.write_rir(d, c["dataset"], c["scene"], azimuth, c["receiver"], c["source"], c["sr"], rir)
        for idx in c["audio_indices"]:
            sim = rh.make_discrete_sim(ref, d, c["sr"], dataset=c["dataset"], scene=c["scene"], receiver=c["receiver"],
                                       source=c["source"], rotation_angle=c["rotation_angle"],
                                       source_sounds={"telephone.wav": src}, audio_index=idx)
            out[f"audio_index_{idx}/wave"] = sim.get_current_audiogoal_observation()
            out[f"audio_index_{idx}/spec_reflect"] = sim.get_current_spectrogram_observation(
                ref["nav"].SpectrogramSensor.compute_spectrogram)

    # keep each file under 1 MB: waveforms go to a file of their own, most of them as every 5th sample
    packed, waves = {}, {}
    for k, v in out.items():
        if not k.endswith("/wave"):
            packed[k] = v
        elif k.startswith(tuple(CONTINUOUS_CASES)) or k in FULL_WAVES:
            waves[k] = v
        else:
            waves[k + "_stride5"] = np.ascontiguousarray(v[:, ::5])
    for name, arrays in (("reference_golden.npz", packed), ("reference_golden_waves.npz", waves)):
        path = os.path.join(ROOT, "tests", "golden", name)
        np.savez_compressed(path, **arrays)
        print("wrote", path, os.path.getsize(path), "bytes,", len(arrays), "arrays")

    path = os.path.join(ROOT, "tests", "golden", "reference_classes.json")
    with open(path, "w") as f:
        json.dump(reference_class_facts(ref), f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", path)

    edge = {}
    ref = rh.load_reference("reflect")
    spec_fn = ref["nav"].SpectrogramSensor.compute_spectrogram
    for name, c in CONTINUOUS_EDGE_CASES.items():
        src, rir, last = continuous_inputs(c)
        sim = rh.make_continuous_sim(ref, c["sr"], src, rir, sample_index=c["sample_index"], last_rir=last,
                                     crossfade=last is not None)
        edge[f"{name}/wave"] = sim.get_current_audiogoal_observation()
        edge[f"{name}/spec_reflect"] = sim.get_current_spectrogram_observation(spec_fn)
    path2 = os.path.join(ROOT, "tests", "golden", "reference_golden_r2.npz")
    np.savez_compressed(path2, **edge)
    print("wrote", path2, os.path.getsize(path2), "bytes,", len(edge), "arrays")


if __name__ == "__main__":
    main()
