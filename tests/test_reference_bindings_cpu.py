"""CPU: this repo's libmoonshine.so against the C ABI the REFERENCE's own Python binding
(language-bindings/python/src/moonshine_voice, pure ctypes) declares, and the calls its `Transcriber` / stream
classes make, on the segmentation-only path (`skip_transcription`, no GPU needed).

What the binding declares is stored in golden/ref_python_binding.json (recorded by golden/make_golden_reference.py
from the binding itself): the field layout of every struct it passes through the ABI (its struct-size guard,
moonshine_api.py:137-146, asks for 24 / 40 / 88 / 16 bytes), every symbol `_setup_function_signatures` binds, and
its header version.  The binding dlopens "libmoonshine.so" by name; this library carries that SONAME."""
import ctypes

import numpy as np
import pytest

from moonshine_b200 import api
from tests.util import reference_golden


@pytest.fixture(scope="module")
def binding():
    lib = api.load_library()
    # the library under test is this repo's, not some other libmoonshine
    assert hasattr(lib, "moonshine_b200_transcribe_device")
    return reference_golden("ref_python_binding.json"), lib


def layout(cls):
    return [[name, getattr(cls, name).offset, getattr(cls, name).size] for name, _ in cls._fields_]


def test_struct_sizes_and_symbols(binding):
    want, lib = binding
    for name, fields in want["structs"].items():
        cls = getattr(api, name)
        assert layout(cls) == fields, name
        assert ctypes.sizeof(cls) == want["sizes"][name], name
    assert ctypes.sizeof(api.TranscriptWordC) == 24
    assert ctypes.sizeof(api.SpeakerSpanC) == 40
    assert ctypes.sizeof(api.TranscriptLineC) == 88
    assert ctypes.sizeof(api.TranscriptC) == 16
    missing = [s for s in want["symbols"] if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.moonshine_get_version() == want["header_version"] == api.MOONSHINE_HEADER_VERSION
    assert api.MOONSHINE_FLAG_FORCE_UPDATE == want["flag_force_update"]
    assert lib.moonshine_error_to_string(-2) == b"Invalid handle"


def test_reference_transcriber_class_segments_audio(binding):
    t = api.Transcriber("/nonexistent-model-dir", api.ModelArch.TINY,
                        options={"skip_transcription": "true", "vad_threshold": "0"})
    rng = np.random.default_rng(3)
    audio = (rng.standard_normal(16000 * 21) * 0.05).astype(np.float32)
    tr = t.transcribe_without_streaming(audio, 16000)
    # vad_threshold=0 is the documented bypass: everything is voice (core/voice-activity-detector.cpp:152-157);
    # whole hops only, so the line holds the input up to one hop (512 samples)
    assert len(tr.lines) == 1
    assert all(ln.is_complete and ln.is_new and ln.is_updated for ln in tr.lines)
    assert tr.lines[0].start_time < 1e-3
    assert 0 <= len(audio) - len(tr.lines[0].audio_data) < 512
    np.testing.assert_array_equal(np.asarray(tr.lines[0].audio_data, np.float32), audio[:len(tr.lines[0].audio_data)])
    # default threshold: the max-segment fade cuts the clip (two lines, distinct ids)
    t2 = api.Transcriber("/nonexistent-model-dir", api.ModelArch.TINY, options={"skip_transcription": "true"})
    tr2 = t2.transcribe_without_streaming(audio, 16000)
    assert len(tr2.lines) >= 2 and len({ln.line_id for ln in tr2.lines}) == len(tr2.lines)
    t2.close()
    t.close()


def test_reference_stream_class(binding):
    t = api.Transcriber("/nonexistent-model-dir", api.ModelArch.TINY,
                        options={"skip_transcription": "true", "vad_threshold": "0"})
    s = t.create_stream()
    s.start()
    rng = np.random.default_rng(4)
    for _ in range(5):
        chunk = (rng.standard_normal(16000) * 0.05).astype(np.float32)
        s.add_audio(chunk, 16000)
        tr = s.update_transcription(api.MOONSHINE_FLAG_FORCE_UPDATE)
        assert len(tr.lines) == 1 and not tr.lines[0].is_complete
    s.stop()
    tr = s.update_transcription(api.MOONSHINE_FLAG_FORCE_UPDATE)
    assert len(tr.lines) == 1 and tr.lines[0].is_complete
    s.close()
    t.close()


def test_reference_binding_error_paths(binding):
    _, lib = binding
    with pytest.raises(api.MoonshineError):   # unknown option key must fail the load (moonshine-c-api.cpp:193-196)
        api.Transcriber("/nonexistent-model-dir", api.ModelArch.TINY,
                        options={"skip_transcription": "true", "no_such_option": "1"})
    out = ctypes.POINTER(api.TranscriptC)()
    buf = (ctypes.c_float * 16)()
    assert lib.moonshine_transcribe_without_streaming(12345, buf, 16, 16000, 0, ctypes.byref(out)) == -2
