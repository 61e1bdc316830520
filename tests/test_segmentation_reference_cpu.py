"""CPU: this library's segmentation (through the C ABI, `skip_transcription`) against the REFERENCE's own
VoiceActivityDetector compiled from core/voice-activity-detector.cpp (oracle/_ref), with the Silero network
replaced on both sides by a constant speech probability of 1.0.  Covers the documented bypass
(`vad_threshold=0`), the smoothing window + max-segment fade at positive thresholds, look-behind across cuts,
resampling, and audio fed in uneven pieces."""
import numpy as np
import pytest

from moonshine_b200 import api
from tests.util import digest, reference_golden


@pytest.fixture(scope="module")
def ref():
    return reference_golden("ref_segmentation.json")


def check_lines(lines, want):
    """`want`: the reference detector's segments, [start_time, end_time, is_complete, sample count, SHA-256 of the
    float32 samples] each."""
    assert len(lines) == len(want)
    for line, (st, en, complete, n, audio_sha) in zip(lines, want):
        assert bool(line.is_complete) == complete
        assert abs(line.start_time - st) < 1e-6 and abs(line.start_time + line.duration - en) < 1e-5
        assert line.audio_data.size == n and digest(np.ascontiguousarray(line.audio_data, np.float32)) == audio_sha


CASES = [
    ({"vad_threshold": "0"}, 16000 * 23 + 777, 16000),
    ({}, 16000 * 40, 16000),                                             # defaults: threshold 0.5, window 16 hops
    ({"vad_threshold": "0.9", "vad_window_duration": "0.25"}, 16000 * 33 + 5, 16000),
    ({"vad_threshold": "0.3", "vad_max_segment_duration": "4.0", "vad_look_behind_sample_count": "2048"}, 16000 * 21, 16000),
    # (a look-behind shorter than one hop is undefined behaviour in the reference itself -- not compared)
    ({"vad_threshold": "0.5", "vad_hop_size": "256", "vad_look_behind_sample_count": "512"}, 16000 * 18 + 1, 16000),
    ({"vad_threshold": "0"}, 44100 * 9 + 13, 44100),                      # resampled inside the VAD
    ({"vad_threshold": "0.5"}, 8000 * 30, 8000),
]
CASE_IDS = [f"case{i}" for i in range(len(CASES))]


def one_shot_audio(n):
    rng = np.random.default_rng(n)
    return (rng.standard_normal(n) * 0.05).astype(np.float32)


@pytest.mark.parametrize("opts,n,rate,case", [c + (i,) for c, i in zip(CASES, CASE_IDS)], ids=CASE_IDS)
def test_one_shot_segmentation_matches_reference_vad(ref, opts, n, rate, case):
    audio = one_shot_audio(n)
    want = ref["one_shot"][case]
    assert len(want) >= 1 and all(complete for _, _, complete, _, _ in want)
    o = {"skip_transcription": "true"}
    o.update(opts)
    t = api.Transcriber(None, api.ModelArch.TINY, o)
    tr = t.transcribe_without_streaming(audio, sample_rate=rate)
    check_lines(tr.lines, want)
    t.close()


STREAM_OPTS = {"bypass": {"vad_threshold": "0"}, "default": {},
               "short_segments": {"vad_threshold": "0.7", "vad_max_segment_duration": "5"}}


def streamed_pieces():
    rng = np.random.default_rng(5)
    audio = (rng.standard_normal(16000 * 26) * 0.05).astype(np.float32)
    cuts = np.sort(rng.choice(np.arange(1, len(audio)), 17, replace=False))
    return [np.ascontiguousarray(p) for p in np.split(audio, cuts)]


@pytest.mark.parametrize("name", ["bypass", "default", "short_segments"])
def test_streamed_segmentation_matches_reference_vad(ref, name):
    """Same audio fed in uneven pieces (hops straddle calls): after every update the lines equal the reference
    detector's segments, including the still-open one."""
    pieces = streamed_pieces()
    want = ref["streamed"][name]
    assert len(want) == len(pieces)
    o = {"skip_transcription": "true"}
    o.update(STREAM_OPTS[name])
    t = api.Transcriber(None, api.ModelArch.TINY, o)
    s = t.create_stream()
    s.start()
    for p, w in zip(pieces, want):
        s.add_audio(p)
        check_lines(s.update_transcription(api.MOONSHINE_FLAG_FORCE_UPDATE).lines, w)
    s.close()
    t.close()


def restart_sessions():
    rng = np.random.default_rng(11)
    first = (rng.standard_normal(16000 * 7 + 123) * 0.05).astype(np.float32)
    second = (rng.standard_normal(16000 * 12 + 7) * 0.05).astype(np.float32)
    return first, second


@pytest.mark.parametrize("name", ["default", "short_segments", "bypass"])
def test_restarted_stream_matches_reference_vad(ref, name):
    """stop() + start() on the same stream: the reference's start() leaves the probability smoothing window as
    it was (resize on an already-sized vector), so the second session's first segments open earlier than on a
    fresh stream.  Compared segment by segment after the restart."""
    want = ref["restarted"][name]
    o = {"skip_transcription": "true"}
    o.update(STREAM_OPTS[name])
    t = api.Transcriber(None, api.ModelArch.TINY, o)
    s = t.create_stream()
    for audio, w in zip(restart_sessions(), want):
        s.start()
        s.add_audio(audio)
        assert len(w) >= 1
        check_lines(s.update_transcription(api.MOONSHINE_FLAG_FORCE_UPDATE).lines, w)
        s.stop()
    s.close()
    t.close()
