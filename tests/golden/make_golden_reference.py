#!/usr/bin/env python
"""Record what the REFERENCE's own code returns on the inputs of the tests that compare this library with it, so
that those tests run from this repository alone.

    python tests/golden/make_golden_reference.py

Needs the reference source tree (located as in oracle/build_ref.py, MOONSHINE_REFERENCE) and a built
libmoonshine.so; no GPU.  The reference's host-side helpers are compiled from that tree into oracle/_ref by
oracle/build_ref.py; its Python binding is imported from the tree unmodified.  The inputs come from the test
modules themselves, so a test and its fixture cannot drift apart.

Writes (all small; byte strings and float arrays too long to store as values are kept as length + SHA-256):
  tests/golden/ref_helpers.json          detokeniser, resampler, align_words, tokenizer encoder, key-term biaser,
                                         passage-to-terms extraction (tests/test_reference_helpers_cpu.py)
  tests/golden/ref_segmentation.json     VoiceActivityDetector segments with the constant-probability Silero
                                         stand-in (tests/test_segmentation_reference_cpu.py)
  tests/golden/ref_word_timestamps.json  align_words on the oracle's cross-attention (tests/test_word_timestamps_gpu.py)
  tests/golden/ref_keyterms.json         ContextBiaser over the streaming oracle's logits (tests/test_keyterms_gpu.py)
  tests/golden/ref_python_binding.json   struct layouts, bound symbols and header version of the Python binding
                                         (tests/test_reference_bindings_cpu.py)
"""
import ctypes
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from moonshine_b200 import api  # noqa: E402
from moonshine_b200.arch import ARCHS  # noqa: E402
from moonshine_b200.weights import synth_audio, synth_tokenizer_bin, synth_weights  # noqa: E402
from oracle import build_ref  # noqa: E402
from oracle import moonshine_oracle as orc  # noqa: E402
from oracle.moonshine_streaming_oracle import SDims, StreamingOracle  # noqa: E402
from tests import test_keyterms_gpu as tk  # noqa: E402
from tests import test_reference_bindings_cpu as tb  # noqa: E402
from tests import test_reference_helpers_cpu as th  # noqa: E402
from tests import test_segmentation_reference_cpu as ts  # noqa: E402
from tests import test_word_timestamps_gpu as tw  # noqa: E402
from tests.util import GOLD, digest, oracle_for  # noqa: E402

c = ctypes
F32P, I32P = c.POINTER(c.c_float), c.POINTER(c.c_int32)


def f32(a):
    return a.ctypes.data_as(F32P)


def i32(a):
    return a.ctypes.data_as(I32P)


def load_ref():
    path = build_ref.build()
    if path is None:
        sys.exit(f"the reference tree is not at {build_ref.REF} (set MOONSHINE_REFERENCE)")
    lib = c.CDLL(path)
    for f in ("ref_tokenizer_new", "ref_tokenizer_new_bpe", "ref_vad_new", "ref_biaser_new"):
        getattr(lib, f).restype = c.c_void_p
    for f in ("ref_tokenizer_new", "ref_tokenizer_new_bpe"):
        getattr(lib, f).argtypes = [c.c_char_p, c.c_uint64]
    for f in ("ref_tokenizer_free", "ref_vad_free", "ref_vad_start", "ref_vad_stop", "ref_biaser_free", "ref_biaser_reset"):
        getattr(lib, f).argtypes = [c.c_void_p]
    lib.ref_tokens_to_text.restype = c.c_int64
    lib.ref_tokens_to_text.argtypes = [c.c_void_p, I32P, c.c_int32, c.c_char_p, c.c_int64]
    lib.ref_resample.restype = c.c_int64
    lib.ref_resample.argtypes = [F32P, c.c_int64, c.c_float, c.c_float, F32P, c.c_int64]
    lib.ref_align_words.restype = c.c_int32
    lib.ref_align_words.argtypes = [c.c_void_p, F32P, c.c_int32, c.c_int32, c.c_int32, c.c_int32, I32P, c.c_int32,
                                    c.c_float, F32P, F32P, c.c_char_p, c.c_int64, c.c_int32]
    lib.ref_text_to_tokens.restype = c.c_int32
    lib.ref_text_to_tokens.argtypes = [c.c_void_p, c.c_char_p, I32P, c.c_int32]
    lib.ref_extract_terms.restype = c.c_int32
    lib.ref_extract_terms.argtypes = [c.c_void_p, c.c_char_p, c.c_int32, c.c_char_p, c.c_int64]
    lib.ref_biaser_add.argtypes = [c.c_void_p, I32P, c.c_int32]
    lib.ref_biaser_advance.argtypes = [c.c_void_p, c.c_int32]
    lib.ref_biaser_apply.argtypes = [c.c_void_p, F32P, c.c_int32]
    lib.ref_biaser_variants.restype = c.c_int32
    lib.ref_biaser_variants.argtypes = [c.c_char_p, c.c_char_p, c.c_int64]
    lib.ref_vad_new.argtypes = [c.c_float, c.c_int32, c.c_int32, c.c_uint64, c.c_uint64]
    lib.ref_vad_process.argtypes = [c.c_void_p, F32P, c.c_uint64, c.c_int32]
    lib.ref_vad_segment_count.restype = c.c_int32
    lib.ref_vad_segment_count.argtypes = [c.c_void_p]
    lib.ref_vad_segment.restype = c.c_int64
    lib.ref_vad_segment.argtypes = [c.c_void_p, c.c_int32, F32P, F32P, c.c_int64]
    return lib


def helpers(ref):
    out = {}
    blob, _, trials = th.detok_inputs()
    h = ref.ref_tokenizer_new(blob, len(blob))
    out["detokeniser"] = []
    for ids in trials:
        buf = c.create_string_buffer(4096)
        nr = ref.ref_tokens_to_text(h, i32(ids), len(ids), buf, 4096)
        out["detokeniser"].append([nr, digest(buf.raw[:nr])])
    ref.ref_tokenizer_free(h)

    out["resample"] = {}
    for rate in th.RESAMPLE_RATES:
        rows = []
        for x in th.resample_inputs(rate):
            cap = len(x) * 3 + 16
            o = np.zeros(cap, np.float32)
            nr = ref.ref_resample(f32(x), len(x), float(rate), 16000.0, f32(o), cap)
            rows.append([nr, digest(o[:nr])])
        out["resample"][str(rate)] = rows

    blob, cases = th.align_inputs()
    h = ref.ref_tokenizer_new(blob, len(blob))
    out["align_words"] = []
    for layers, heads, steps, frames, x, toks, tpf in cases:
        st, en = np.zeros(64, np.float32), np.zeros(64, np.float32)
        txt = c.create_string_buffer(8192)
        n = ref.ref_align_words(h, f32(x), layers, heads, steps, frames, i32(toks), len(toks), tpf, f32(st), f32(en),
                                txt, 8192, 64)
        k = max(n, 0)
        out["align_words"].append({"n": n, "words": [w.hex() for w in txt.raw.split(b"\0")[:k]],
                                   "start": st[:k].tolist(), "end": en[:k].tolist()})
    ref.ref_tokenizer_free(h)

    blob, _ = th.bpe_vocab()
    out["text_to_tokens"] = {}
    for make, key in ((ref.ref_tokenizer_new_bpe, "bpe"), (ref.ref_tokenizer_new, "longest_match")):
        h = make(blob, len(blob))
        rows = []
        for t in th.TEXTS:
            a = np.zeros(128, np.int32)
            nr = ref.ref_text_to_tokens(h, th.text_bytes(t), i32(a), 128)
            rows.append({"n": nr, "ids": a[:nr].tolist() if nr > 0 else []})
        out["text_to_tokens"][key] = rows
        ref.ref_tokenizer_free(h)

    out["biaser"] = []
    for seqs, path, lr0 in th.biaser_inputs():
        b = ref.ref_biaser_new()
        for s in seqs:
            ref.ref_biaser_add(b, i32(s), len(s))
        ref.ref_biaser_reset(b)
        for t in path:
            ref.ref_biaser_advance(b, int(t))
        lr = lr0.copy()
        ref.ref_biaser_apply(b, f32(lr), th.BIASER_VOCAB)
        ref.ref_biaser_free(b)
        idx = np.flatnonzero(lr != lr0)
        out["biaser"].append({"index": idx.tolist(), "value": lr[idx].tolist()})

    def terms(h, text, max_terms):
        buf = c.create_string_buffer(1 << 14)
        nr = ref.ref_extract_terms(h, text, max_terms, buf, 1 << 14)
        return {"n": nr, "terms": [t.hex() for t in buf.raw.split(b"\0")[:max(nr, 0)]]}

    h = ref.ref_tokenizer_new_bpe(blob, len(blob))
    out["extract_terms"] = {"passage": {str(m): terms(h, th.PASSAGE.encode("utf-8"), m) for m in th.MAX_TERMS}}
    ref.ref_tokenizer_free(h)
    blob2 = synth_tokenizer_bin(400)
    h = ref.ref_tokenizer_new_bpe(blob2, len(blob2))
    out["extract_terms"]["short"] = terms(h, th.SHORT_PASSAGE, 0)
    ref.ref_tokenizer_free(h)
    return out


def make_vad(ref, opts):
    hop = int(opts.get("vad_hop_size", 512))
    window = math.ceil(float(opts.get("vad_window_duration", 0.5)) * 16000 / hop)       # transcriber.cpp
    max_seg = int(round(float(opts.get("vad_max_segment_duration", 15.0)) * 16000))
    return ref.ref_vad_new(float(opts.get("vad_threshold", 0.5)), window, hop,
                           int(opts.get("vad_look_behind_sample_count", 8192)), max_seg)


def vad_segments(ref, v):
    out = []
    for i in range(ref.ref_vad_segment_count(v)):
        info = np.zeros(4, np.float32)
        n = ref.ref_vad_segment(v, i, f32(info), None, 0)
        audio = np.zeros(max(n, 1), np.float32)
        ref.ref_vad_segment(v, i, f32(info), f32(audio), n)
        out.append([float(info[0]), float(info[1]), bool(info[2]), int(n), digest(audio[:n])])
    return out


def segmentation(ref):
    out = {"one_shot": {}, "streamed": {}, "restarted": {}}
    for (opts, n, rate), case in zip(ts.CASES, ts.CASE_IDS):
        audio = ts.one_shot_audio(n)
        v = make_vad(ref, opts)
        ref.ref_vad_start(v)
        ref.ref_vad_process(v, f32(audio), n, rate)
        ref.ref_vad_stop(v)
        out["one_shot"][case] = vad_segments(ref, v)
        ref.ref_vad_free(v)
    for name, opts in ts.STREAM_OPTS.items():
        v = make_vad(ref, opts)
        ref.ref_vad_start(v)
        rows = []
        for p in ts.streamed_pieces():
            ref.ref_vad_process(v, f32(p), len(p), 16000)
            rows.append(vad_segments(ref, v))
        out["streamed"][name] = rows
        ref.ref_vad_free(v)
        v = make_vad(ref, opts)
        rows = []
        for audio in ts.restart_sessions():
            ref.ref_vad_start(v)
            ref.ref_vad_process(v, f32(audio), len(audio), 16000)
            rows.append(vad_segments(ref, v))
            ref.ref_vad_stop(v)
        out["restarted"][name] = rows
        ref.ref_vad_free(v)
    return out


def oracle_words(ref, o, d, memory, tokens_budget, seg_samples):
    """Greedy decode on `memory` collecting cross-attention, then the reference's align_words."""
    cross = o.cross_kv(memory)
    cache = o.new_self_cache()
    toks, cur, att = [d.bos], d.bos, []
    for t in range(tokens_budget):
        lg, xa = o.decoder_step([cur], t, cache, cross, want_cross_attn=True)
        att.append(np.stack([a[:, 0, :] for a in xa]))          # [L, H, T]
        nxt = int(np.argmax(lg[0]))
        toks.append(nxt)
        if nxt == d.eos:
            break
        cur = nxt
    steps, T = len(att), memory.shape[0]
    x = np.ascontiguousarray(np.stack(att, 2).reshape(d.dec_layers * d.heads, steps, T).astype(np.float32))
    blob = synth_tokenizer_bin(d.vocab)
    h = ref.ref_tokenizer_new(blob, len(blob))
    ids = np.asarray(toks, np.int32)
    st, en = np.zeros(256, np.float32), np.zeros(256, np.float32)
    txt = c.create_string_buffer(1 << 16)
    tpf = np.float32(np.float32(seg_samples) / np.float32(16000.0)) / np.float32(T)
    n = ref.ref_align_words(h, f32(x), d.dec_layers, d.heads, steps, T, i32(ids), len(ids), tpf, f32(st), f32(en),
                            txt, 1 << 16, 256)
    ref.ref_tokenizer_free(h)
    return {"words": [w.decode("utf-8") for w in txt.raw.split(b"\0")[:n]], "start": st[:n].tolist(),
            "end": en[:n].tolist(), "time_per_frame": float(tpf)}


def word_timestamps(ref):
    out = {"classic": {}}
    for arch, seed, n in tw.CLASSIC_CASES:
        seg = synth_audio(7, n)
        seg = seg[: len(seg) // 512 * 512]
        o = oracle_for(arch, seed)
        out["classic"][f"{arch}_s{seed}_{n}"] = oracle_words(ref, o, ARCHS[arch], o.encoder(seg), o.max_len(len(seg)), len(seg))
    arch = "test_streaming"
    d = ARCHS[arch]
    seg = synth_audio(*tw.STREAMING_AUDIO)
    seg = seg[: len(seg) // 512 * 512]
    o = StreamingOracle(SDims.from_product(d), synth_weights(arch, 0))
    n_feat = len(seg) // 1280 * 4
    out["streaming"] = oracle_words(ref, o, d, o.memory_stateless(seg, n_feat, n_feat), o.max_tokens_greedy(len(seg)), len(seg))
    return out


def keyterms(ref):
    arch = "test_streaming"
    d = ARCHS[arch]
    blob = synth_tokenizer_bin(d.vocab)
    vocab = orc.load_tokenizer_bin(blob)
    seg = synth_audio(*tk.KEYTERM_AUDIO)
    seg = seg[: len(seg) // 512 * 512]
    o = StreamingOracle(SDims.from_product(d), synth_weights(arch, 0))
    n_feat = len(seg) // 1280 * 4
    mem = o.memory_stateless(seg, n_feat, n_feat)
    budget = o.max_tokens_greedy(len(seg))
    plain, _ = o.greedy_memory(mem, budget, keep_logits=False)
    # key terms spelled from vocabulary pieces the unbiased decode does not produce; each starts with the
    # word-boundary marker, so it has exactly one spelling (ContextBiaser::variants_for_term)
    marker = "▁".encode()
    starts = [i for i in range(10, d.vocab - 3) if vocab[i].startswith(marker)
              and all(j not in plain for j in (i, i + 1, i + 2))]
    a, b = starts[0], starts[5]
    terms = [(vocab[a] + vocab[a + 1]).decode(), (vocab[b] + vocab[b + 1] + vocab[b + 2]).decode()]
    tok = ref.ref_tokenizer_new_bpe(blob, len(blob))
    biaser = ref.ref_biaser_new()
    for term in terms:
        buf = c.create_string_buffer(1024)
        n = ref.ref_biaser_variants(term.encode(), buf, 1024)
        for variant in buf.raw.split(b"\0")[:n]:
            ids = np.zeros(64, np.int32)
            k = ref.ref_text_to_tokens(tok, variant, i32(ids), 64)
            assert k > 0
            ref.ref_biaser_add(biaser, i32(ids), k)
    ref.ref_tokenizer_free(tok)
    # greedy decode with the reference biaser (default boost 2) applied to the oracle's logits before each argmax
    cross = o.cross_kv(mem)
    cache = o.new_self_cache()
    biased, cur = [d.bos], d.bos
    ref.ref_biaser_reset(biaser)
    for t in range(budget):
        lg = np.ascontiguousarray(o.decoder_step([cur], t, cache, cross)[0], np.float32)
        ref.ref_biaser_apply(biaser, f32(lg), d.vocab)
        nxt = int(np.argmax(lg))
        biased.append(nxt)
        if nxt == d.eos:
            break
        ref.ref_biaser_advance(biaser, nxt)
        cur = nxt
    ref.ref_biaser_free(biaser)
    return {"terms": terms, "plain": [int(t) for t in plain], "biased": biased}


def python_binding():
    ref_py = os.path.join(build_ref.REF, "language-bindings", "python", "src")
    c.CDLL(api.lib_path(), mode=c.RTLD_GLOBAL)          # same SONAME as the name the binding dlopens
    sys.path.insert(0, ref_py)
    from moonshine_voice import moonshine_api            # runs the binding's struct-size guard
    lib = moonshine_api._MoonshineLib().lib             # binds every symbol the binding declares
    assert hasattr(lib, "moonshine_b200_transcribe_device")
    structs = ("TranscriptWordC", "SpeakerSpanC", "TranscriptLineC", "TranscriptC", "TranscriberOptionC")
    return {"structs": {s: tb.layout(getattr(moonshine_api, s)) for s in structs},
            "sizes": {s: c.sizeof(getattr(moonshine_api, s)) for s in structs},
            "symbols": sorted(k for k, v in vars(lib).items() if isinstance(v, c._CFuncPtr)),
            "header_version": moonshine_api.MOONSHINE_HEADER_VERSION,
            "flag_force_update": moonshine_api.MOONSHINE_FLAG_FORCE_UPDATE}


def write(name, obj):
    path = os.path.join(GOLD, name)
    with open(path, "w", encoding="utf-8") as f:
        json.dump(obj, f, ensure_ascii=False, separators=(",", ":"))
        f.write("\n")
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    ref = load_ref()
    write("ref_helpers.json", helpers(ref))
    write("ref_segmentation.json", segmentation(ref))
    write("ref_keyterms.json", keyterms(ref))
    write("ref_python_binding.json", python_binding())
    write("ref_word_timestamps.json", word_timestamps(ref))
