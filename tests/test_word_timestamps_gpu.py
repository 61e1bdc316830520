"""GPU: word timestamps through the reference ABI (`word_timestamps=true` -> transcript_line_t.words).
Expected values: the oracle's decoder cross-attention fed to the REFERENCE's own align_words (core/word-alignment.cpp),
stored in golden/ref_word_timestamps.json by golden/make_golden_reference.py.  The GPU attention differs from the
oracle's by ~1e-5, which can move a DTW boundary by a frame on a near-tie, so times are compared within two frames
and required to be identical for most words."""
import numpy as np
import pytest

from moonshine_b200 import api
from moonshine_b200.weights import synth_audio
from tests.util import memory_files, reference_golden

pytestmark = pytest.mark.gpu

CLASSIC_CASES = [("test", 0, 48333), ("base", 0, 40000), ("tiny", 0, 80000)]
STREAMING_AUDIO = (9, 16000 * 3 + 100)


@pytest.fixture(scope="module")
def ref():
    return reference_golden("ref_word_timestamps.json")


def compare(line, words, st, en, tpf):
    got = line.words or []
    assert [w.word for w in got] == words
    gs = np.array([w.start for w in got], np.float32) - np.float32(line.start_time)
    ge = np.array([w.end for w in got], np.float32) - np.float32(line.start_time)
    assert np.abs(gs - st).max() <= 2.01 * tpf and np.abs(ge - en).max() <= 2.01 * tpf
    same = (np.abs(gs - st) < 1e-4) & (np.abs(ge - en) < 1e-4)
    assert same.mean() >= 0.8, same.mean()


@pytest.mark.parametrize("arch,seed,n", CLASSIC_CASES)
def test_word_timestamps_classic(ref, arch, seed, n):
    audio = synth_audio(7, n)
    t = api.Transcriber(model_arch={"test": api.ModelArch.TEST, "base": api.ModelArch.BASE,
                                    "tiny": api.ModelArch.TINY}[arch],
                        options={"vad_threshold": "0", "word_timestamps": "true"},
                        memory_files=memory_files(arch, seed))
    tr = t.transcribe_without_streaming(audio)
    assert len(tr.lines) == 1
    w = ref["classic"][f"{arch}_s{seed}_{n}"]
    assert len(w["words"]) > 0
    compare(tr.lines[0], w["words"], np.array(w["start"], np.float32), np.array(w["end"], np.float32), w["time_per_frame"])
    t.close()


def test_word_timestamps_streaming_arch(ref):
    arch = "test_streaming"
    audio = synth_audio(*STREAMING_AUDIO)
    t = api.Transcriber(model_arch=api.ModelArch.TEST_STREAMING,
                        options={"vad_threshold": "0", "word_timestamps": "true"}, memory_files=memory_files(arch, 0))
    tr = t.transcribe_without_streaming(audio)
    w = ref["streaming"]
    assert len(w["words"]) > 0
    compare(tr.lines[0], w["words"], np.array(w["start"], np.float32), np.array(w["end"], np.float32), w["time_per_frame"])
    t.close()
