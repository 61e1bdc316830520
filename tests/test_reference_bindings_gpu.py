"""GPU: the reference's own C++ client -- core/benchmark.cpp through the header-only core/moonshine-cpp.h --
compiled from the reference source tree (recipe: oracle/build_ref.py::build_benchmark, output
oracle/_ref/ref_benchmark) and linked against this repo's libmoonshine.so, transcribes beckett.wav from a model
directory.  It drives the streaming half of the ABI the way the reference's tool does (21.4 ms chunks, an update
every 0.481 s).  The final text must equal what this library returns for the same clip in one shot.  The client is
the reference's own program, so this test runs only where build() could compile it and skips elsewhere."""
import os
import re
import subprocess
import wave

import numpy as np
import pytest

from moonshine_b200 import api
from moonshine_b200.arch import ARCHS
from moonshine_b200.weights import pack_msw, synth_tokenizer_bin
from oracle import build_ref
from tests.util import GOLD, weights_for

pytestmark = pytest.mark.gpu


def test_reference_benchmark_cpp_runs_against_this_library(tmp_path):
    exe = build_ref.build_benchmark()
    if exe is None or not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_benchmark not built (needs the reference source tree)")
    arch = "tiny"
    d = ARCHS[arch]
    model_dir = tmp_path / "tiny-en"
    model_dir.mkdir()
    (model_dir / "model.msw").write_bytes(pack_msw(arch, weights_for(arch, 0, "scaled")))
    (model_dir / "tokenizer.bin").write_bytes(synth_tokenizer_bin(d.vocab))
    pcm16 = np.load(os.path.join(GOLD, "beckett_pcm16.npy")).astype(np.int16)
    wav = tmp_path / "beckett.wav"
    with wave.open(str(wav), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000)
        w.writeframes(pcm16.tobytes())
    r = subprocess.run([exe, "-m", str(model_dir), "-a", "0", "-w", str(wav)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "Transcription took" in r.stderr
    # the same clip through this library's own binding, fed the way the tool feeds it (default options on both sides)
    pcm = pcm16.astype(np.float32) / np.float32(32768.0)
    t = api.Transcriber(str(model_dir), api.ModelArch.TINY)
    s = t.create_stream()
    s.start()
    chunk, every, since = int(0.0214 * 16000), int(0.481 * 16000), 0
    for i in range(0, len(pcm), chunk):
        piece = pcm[i:i + chunk]
        s.add_audio(piece)
        since += len(piece)
        if since >= every:
            since = 0
            s.update_transcription()
    s.stop()
    tr = s.update_transcription()
    s.close()
    t.close()
    assert len(tr.lines) >= 1
    printed = re.findall(r"\] '(.*)' \(", r.stderr)
    assert printed == [line.text for line in tr.lines], (printed, [line.text for line in tr.lines])
    m = re.search(r"Average Latency: (\d+)ms", r.stderr)
    assert m is not None
