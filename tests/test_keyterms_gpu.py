"""GPU: key-term biasing on a streaming architecture through the reference ABI (`keyterms` / `keyterm_boost`
options and moonshine_transcriber_set_keyterms).  Expected text: the streaming oracle's logits with the
REFERENCE's own ContextBiaser (core/context-biaser.cpp) applied before each argmax, key terms spelled by the
reference's own tokenizer; the resulting ids are stored in golden/ref_keyterms.json by
golden/make_golden_reference.py."""
import pytest

from moonshine_b200 import api
from moonshine_b200.arch import ARCHS
from moonshine_b200.weights import synth_audio, synth_tokenizer_bin
from oracle import moonshine_oracle as orc
from tests.util import memory_files, reference_golden

pytestmark = pytest.mark.gpu

KEYTERM_AUDIO = (21, 16000 * 3)


@pytest.fixture(scope="module")
def ref():
    return reference_golden("ref_keyterms.json")


def test_keyterm_bias_changes_the_transcript_like_the_reference_biaser(ref):
    """`plain`: the oracle's unbiased greedy ids; `terms`: spelled from vocabulary pieces that decode does not produce,
    each starting with the word-boundary marker so it has exactly one spelling (ContextBiaser::variants_for_term);
    `biased`: the oracle's greedy ids with the reference biaser at its fixed default boost of 2."""
    arch = "test_streaming"
    d = ARCHS[arch]
    vocab = orc.load_tokenizer_bin(synth_tokenizer_bin(d.vocab))
    audio = synth_audio(*KEYTERM_AUDIO)
    plain, terms, want_default = ref["plain"], ref["terms"], ref["biased"]
    boost = 60.0
    t = api.Transcriber(model_arch=api.ModelArch.TEST_STREAMING,
                        options={"vad_threshold": "0", "keyterms": ",".join(terms)},
                        memory_files=memory_files(arch, 0))
    got = t.transcribe_without_streaming(audio).lines[0].text
    assert got == orc.sanitize_utf8(orc.tokens_to_text(vocab, want_default)).decode()
    # runtime call: clearing the list restores the unbiased transcript
    t.set_keyterms([])
    assert t.transcribe_without_streaming(audio).lines[0].text == orc.sanitize_utf8(orc.tokens_to_text(vocab, plain)).decode()
    t.close()
    # a large boost forces the key terms into the transcript (the reference biaser's boost is fixed, so this half is
    # checked on the product alone)
    t2 = api.Transcriber(model_arch=api.ModelArch.TEST_STREAMING,
                         options={"vad_threshold": "0", "keyterms": ",".join(terms), "keyterm_boost": str(boost)},
                         memory_files=memory_files(arch, 0))
    forced = t2.transcribe_without_streaming(audio).lines[0].text
    assert forced != orc.sanitize_utf8(orc.tokens_to_text(vocab, plain)).decode()
    assert any(term.replace("▁", "") in forced.replace(" ", "") for term in terms)
    t2.close()


def test_keyterms_are_rejected_on_classic_architectures():
    t = api.Transcriber(model_arch=api.ModelArch.TEST, options={"vad_threshold": "0"}, memory_files=memory_files("test", 0))
    with pytest.raises(Exception):
        t.set_keyterms(["anything"])
    with pytest.raises(Exception):
        t.set_context("a passage with Kubernetes in it")
    t.close()


def byte_fallback_tokenizer(vocab_size):
    """A vocabulary with the 256-entry byte block BPE needs (ids 3..258), the word-boundary marker and filler
    pieces up to the model's vocabulary size."""
    recs = [b"<unk>", b"<s>", b"</s>"] + [bytes([i]) for i in range(256)] + ["▁".encode()]
    i = 0
    while len(recs) < vocab_size:
        recs.append(("▁" if i % 3 == 0 else "").encode() + bytes([97 + i % 26, 97 + (i // 26) % 26]))
        i += 1
    out = bytearray()
    for r in recs:
        out.append(len(r))
        out += r
    return bytes(out)


def test_set_context_extracts_terms_and_biases():
    """moonshine_transcriber_set_context on a streaming architecture: terms come from the passage
    (ContextExtractor rules), the decode then runs biased; an empty passage clears the bias."""
    arch = "test_streaming"
    d = ARCHS[arch]
    audio = synth_audio(21, 16000 * 3)
    t = api.Transcriber(model_arch=api.ModelArch.TEST_STREAMING, options={"vad_threshold": "0", "keyterm_boost": "60"},
                        memory_files=memory_files(arch, 0, tokenizer=byte_fallback_tokenizer(d.vocab)))
    plain = t.transcribe_without_streaming(audio).lines[0].text
    word = "Zqxj"   # no piece of the vocabulary spells it: several byte-fallback subwords
    assert word not in plain
    t.set_context(f"The {word} meeting: {word}, again {word}.")
    biased = t.transcribe_without_streaming(audio).lines[0].text
    # every word of the passage needs several byte-fallback subwords here, so each became a key term; with this
    # boost the transcript is made of them
    assert biased != plain and any(w in biased for w in (word, "meeting", "again"))
    t.set_context("")
    assert t.transcribe_without_streaming(audio).lines[0].text == plain
    t.close()
