"""CPU: this repo's host-side helpers against the REFERENCE's own code: detokeniser, tokenizer encoder, resampler,
align_words, key-term biaser and passage-to-terms extraction, bit-exact.  What the reference's code returns for these
inputs is stored in golden/ref_helpers.json (recorded by golden/make_golden_reference.py from the reference's sources
compiled into oracle/_ref): short results as values, long byte strings and float arrays as length + SHA-256."""
import ctypes

import numpy as np
import pytest

from moonshine_b200 import api
from moonshine_b200.weights import synth_tokenizer_bin
from oracle import moonshine_oracle as orc
from tests.util import digest, reference_golden


@pytest.fixture(scope="module")
def ref():
    return reference_golden("ref_helpers.json")


@pytest.fixture(scope="module")
def product():
    return api.load_library()


def _i32(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))


def _f32(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def detok_inputs():
    vocab_n = 2000
    tok = synth_tokenizer_bin(vocab_n)
    # add pieces the synthetic table lacks: multi-byte UTF-8, embedded markers, angle-bracket lookalikes
    extra = ["▁héllo", "wörld▁", "<x>", "<>", "a<b>", "▁", "▁▁two", " lead", "trail ", "日本語"]
    blob = bytearray(tok)
    for e in extra:
        b = e.encode("utf-8")
        blob.append(len(b))
        blob += b
    blob = bytes(blob)
    n_vocab = vocab_n + len(extra)
    rng = np.random.default_rng(0)
    trials = []
    for trial in range(200):
        n = int(rng.integers(0, 40))
        ids = rng.integers(0, n_vocab, n).astype(np.int32)
        if trial % 3 == 0 and n:
            ids[rng.integers(0, n, max(1, n // 4))] = rng.integers(vocab_n, n_vocab, max(1, n // 4))
        if trial % 5 == 0 and n:
            ids[0] = 1
            ids[-1] = 2
        trials.append(ids)
    return blob, n_vocab, trials


def test_detokeniser_matches_reference_code(ref, product):
    blob, n_vocab, trials = detok_inputs()
    vocab = orc.load_tokenizer_bin(blob)
    assert len(vocab) == n_vocab
    want = ref["detokeniser"]
    assert len(want) == len(trials)
    for ids, (nr, text_sha) in zip(trials, want):
        buf_p = ctypes.create_string_buffer(4096)
        npd = product.moonshine_b200_debug_tokens_to_text(blob, len(blob), _i32(ids), len(ids), buf_p, 4096)
        got = buf_p.raw[:npd]
        assert nr >= 0 and npd == nr and digest(got) == text_sha
        assert orc.tokens_to_text(vocab, ids.tolist()) == got


RESAMPLE_RATES = [8000, 11025, 22050, 32000, 44100, 48000, 16000]


def resample_inputs(rate):
    rng = np.random.default_rng(rate)
    return [(rng.standard_normal(n) * 0.3).astype(np.float32) for n in (1, 2, 17, 1000, 44100 // 3 + 5)]


@pytest.mark.parametrize("rate", RESAMPLE_RATES)
def test_resampler_matches_reference_code(ref, product, rate):
    inputs = resample_inputs(rate)
    want = ref["resample"][str(rate)]
    assert len(want) == len(inputs)
    for x, (nr, out_sha) in zip(inputs, want):
        n = len(x)
        cap = n * 3 + 16
        out_p = np.zeros(cap, np.float32)
        npd = product.moonshine_b200_debug_resample(_f32(x), n, float(rate), 16000.0, _f32(out_p), cap)
        assert nr == npd
        assert digest(out_p[:npd]) == out_sha
        np.testing.assert_array_equal(orc.resample_audio(x, rate), out_p[:npd])


def align_inputs():
    vocab_n = 600
    blob = synth_tokenizer_bin(vocab_n)
    rng = np.random.default_rng(3)
    cases = []
    for trial in range(40):
        layers, heads = int(rng.integers(1, 4)), int(rng.integers(1, 5))
        steps = int(rng.integers(1, 24))
        frames = int(rng.integers(1, 90)) if trial % 4 else int(rng.integers(1, 6))
        x = rng.random((layers * heads, steps, frames)).astype(np.float32)
        if trial % 2:  # monotonic ridge + noise, softmax-normalised like real cross-attention
            centre = np.linspace(0, frames - 1, steps)[None, :, None]
            x = np.exp(-0.5 * ((np.arange(frames)[None, None, :] - centre) / 2.0) ** 2) * 4 + x
            x = (np.exp(x) / np.exp(x).sum(-1, keepdims=True)).astype(np.float32)
        n_tok = steps + 1 if trial % 3 else steps  # with / without a final EOS row
        toks = np.concatenate([[1], rng.integers(3, vocab_n, n_tok - 1)]).astype(np.int32)
        if trial % 3:
            toks[-1] = 2
        tpf = np.float32(10.0 / frames)
        cases.append((layers, heads, steps, frames, x, toks, tpf))
    return blob, cases


def test_word_alignment_matches_reference_code(ref, product):
    """align_words (core/word-alignment.cpp): z-score, width-7 median, head mean, DTW, word grouping, overlap
    fix -- this library's implementation against the reference's compiled one, on random and on peaked
    (speech-like, monotonic) attention maps."""
    blob, cases = align_inputs()
    want = ref["align_words"]
    assert len(want) == len(cases)
    for (layers, heads, steps, frames, x, toks, tpf), w in zip(cases, want):
        st, en = np.zeros(64, np.float32), np.zeros(64, np.float32)
        txt = ctypes.create_string_buffer(8192)
        n = product.moonshine_b200_debug_align_words(blob, len(blob), _f32(x), layers * heads, steps, frames, _i32(toks),
                                                     len(toks), tpf, _f32(st), _f32(en), txt, 8192, 64)
        words = txt.raw.split(b"\0")[:max(n, 0)]
        assert n == w["n"] and words == [bytes.fromhex(h) for h in w["words"]]
        np.testing.assert_array_equal(st[:max(n, 0)], np.array(w["start"], np.float32))
        np.testing.assert_array_equal(en[:max(n, 0)], np.array(w["end"], np.float32))


def bpe_vocab():
    """A small byte-fallback vocabulary: control tokens, the 256-byte block, then merged pieces."""
    recs = [b"<unk>", b"<s>", b"</s>"] + [bytes([i]) for i in range(256)]
    merged = ["▁", "th", "the", "▁the", "er", "in", "▁k", "ub", "▁kub", "ern", "etes", "▁kubern", "▁kubernetes",
              "ku", "kub", "ber", "net", "es", "▁a", "an", "▁an", "é", "▁é", "lu", "min", "ous", "umin", "▁l", "日本"]
    recs += [m.encode("utf-8") for m in merged]
    out = bytearray()
    for r in recs:
        out.append(len(r))
        out += r
    return bytes(out), len(recs)


TEXTS = ["the", " the", "kubernetes", " kubernetes", "Kubernetes", "luminous", " an éclair", "日本語", "a  b",
         "thethe", "", " ", "x", "\xff\xfe".encode("latin1").decode("latin1")]


def text_bytes(t):
    return t.encode("utf-8", errors="surrogateescape") if isinstance(t, str) else t


def test_text_to_tokens_matches_reference_code(ref, product):
    blob, _ = bpe_vocab()
    for bpe in (1, 0):
        want = ref["text_to_tokens"]["bpe" if bpe else "longest_match"]
        assert len(want) == len(TEXTS)
        for t, w in zip(TEXTS, want):
            b = np.zeros(128, np.int32)
            npd = product.moonshine_b200_debug_text_to_tokens(blob, len(blob), text_bytes(t), bpe, _i32(b), 128)
            assert w["n"] == npd, (t, bpe, w["n"], npd)
            if npd > 0:
                np.testing.assert_array_equal(b[:npd], np.array(w["ids"], np.int32))


BIASER_VOCAB = 300


def biaser_inputs():
    rng = np.random.default_rng(11)
    vocab = BIASER_VOCAB
    cases = []
    for trial in range(30):
        seqs = [rng.integers(0, 40, int(rng.integers(1, 6))).astype(np.int32) for _ in range(int(rng.integers(1, 12)))]
        if trial % 4 == 0:
            seqs.append(np.array([5, 6, 7, vocab + 3], np.int32))   # an id outside the vocabulary is skipped
        # walk along a path that follows one sequence part of the way, with detours
        base = seqs[int(rng.integers(0, len(seqs)))]
        path = np.concatenate([rng.integers(0, 40, 2), base[: max(1, len(base) - 1)]]).astype(np.int32)
        logits = rng.standard_normal(vocab).astype(np.float32)
        cases.append((seqs, path, logits))
    return cases


def test_keyterm_biaser_matches_reference_code(ref, product):
    vocab = BIASER_VOCAB
    cases = biaser_inputs()
    want = ref["biaser"]
    assert len(want) == len(cases)
    for (seqs, path, lr0), w in zip(cases, want):
        flat = np.concatenate(seqs).astype(np.int32)
        lens = np.array([len(s) for s in seqs], np.int32)
        # the reference's biased logits: the unbiased ones with the stored entries it changed
        lr = lr0.copy()
        lr[np.array(w["index"], np.int64)] = np.array(w["value"], np.float32)
        lp = lr0.copy()
        rc = product.moonshine_b200_debug_biaser_apply(_i32(flat), _i32(lens), len(seqs), 2.0, _i32(path), len(path),
                                                       _f32(lp), vocab)
        assert rc == 0
        np.testing.assert_array_equal(lp, lr)
        # the sparse form the GPU path uploads (shared root bonuses + this step's per-token extras) adds up to the same
        ls = lr0.copy()
        rc = product.moonshine_b200_debug_biaser_apply_sparse(_i32(flat), _i32(lens), len(seqs), 2.0, _i32(path), len(path),
                                                              _f32(ls), vocab)
        assert rc == 0
        np.testing.assert_allclose(ls, lr, rtol=0, atol=1e-6)
        assert np.array_equal(ls != lr0, lr != lr0)   # exactly the same tokens are touched


PASSAGE = """It was the best of times at Tellson’s Bank — Tellson's, by Temple Bar, was an old-fashioned place.
Madame Defarge knitted; madame Defarge saw nothing. The Kubernetes cluster (kubernetes v1.29, IPv6 only) restarted twice.
Dr. Manette’s luminous notes mention luminous paint, “luminous” dials and the éclair au café …
A well-known, so-called state-of-the-art re-entry; the Joneses' dog. an it of to. 日本語 の テキスト.
Madame Madame Madame the the the kubernetes Kubernetes KUBERNETES --dash-- 'quoted' x-ray."""
MAX_TERMS = (0, 3, 1, 50)
SHORT_PASSAGE = b"abc abcd bcd efgh ab cdefgh"


def test_key_term_extraction_matches_reference_code(ref, product):
    """ContextExtractor::extract with the tokenizer-as-rarity-oracle, on a passage with typographic punctuation,
    possessives, case variants, digits, hyphens and non-ASCII words; both the BPE and the longest-match vocabularies."""
    want = ref["extract_terms"]
    blob, _ = bpe_vocab()
    text = PASSAGE.encode("utf-8")
    for max_terms in MAX_TERMS:
        w = want["passage"][str(max_terms)]
        bp = ctypes.create_string_buffer(1 << 14)
        npd = product.moonshine_b200_debug_extract_terms(blob, len(blob), text, max_terms, bp, 1 << 14)
        assert w["n"] == npd and npd > 0
        assert bp.raw.split(b"\0")[:npd] == [bytes.fromhex(h) for h in w["terms"]]
    # a vocabulary without the byte block (longest match, unspellable words count as 0 subwords)
    blob2 = synth_tokenizer_bin(400)
    w = want["short"]
    bp = ctypes.create_string_buffer(1 << 14)
    npd = product.moonshine_b200_debug_extract_terms(blob2, len(blob2), SHORT_PASSAGE, 0, bp, 1 << 14)
    assert w["n"] == npd and bp.raw.split(b"\0")[:max(npd, 0)] == [bytes.fromhex(h) for h in w["terms"]]
