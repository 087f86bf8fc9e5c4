"""BPE tokenizers (csrc/tokenizer.cpp through the C ABI) — bit-exact token ids.

Pinning chain: the reference's known-answer vector (src/token/clip.rs:232-249) pins the Python oracle
(oracle/tokenizer_oracle.py, a line-by-line restatement); the oracle generated tests/golden/tokenizer_vectors.json; the C++
tokenizer must reproduce those vectors and agree with the oracle on a seeded fuzz corpus. The real CLIP / OpenCLIP vocabularies
(3 MB of third-party data) are not stored whole: tests/golden/tokenizer_ref_subset.json keeps every entry this file's corpus
reaches at its original position (tests/golden/make_tokenizer_golden.py says why that tokenizes the corpus exactly as the full
files do), and the `real` fixture writes it back out as vocabulary files. CPU only, no GPU call.
"""
import json
import os
import random

import pytest

from oracle import tokenizer_oracle as TO
from sdxl_b200.tokenizer import ClipTokenizer, OpenClipTokenizer
from sdxl_b200 import SdxlError

GOLD = os.path.join(os.path.dirname(__file__), "golden")
MINI = os.path.join(GOLD, "mini_bpe")
VEC = json.load(open(os.path.join(GOLD, "tokenizer_vectors.json"), encoding="utf-8"))

KAT_TEXT = "Hello world! <|startoftext|>asdf<|startoftext|>"
KAT_IDS = [3306, 1002, 256, 49406, 587, 10468, 49406]
KAT_DECODE = "hello world ! <|startoftext|>asdf <|startoftext|>"


@pytest.fixture(scope="module")
def mini():
    return (OpenClipTokenizer(os.path.join(MINI, "mini_merges.txt"), os.path.join(MINI, "mini_vocab.txt")),
            TO.OpenClipTokenizer(os.path.join(MINI, "mini_merges.txt"), os.path.join(MINI, "mini_vocab.txt")))


def _write_subset(path, table, placeholder):
    """One line per position: the kept entry, or a placeholder on U+E000 that no byte-level piece can equal."""
    keep = table["keep"]
    with open(path, "w", encoding="utf-8", newline="\n") as f:
        f.writelines((keep[str(i)] if str(i) in keep else placeholder(i)) + "\n" for i in range(table["n"]))
    return path


@pytest.fixture(scope="module")
def real(tmp_path_factory):
    sub = json.load(open(os.path.join(GOLD, "tokenizer_ref_subset.json"), encoding="utf-8"))
    d = tmp_path_factory.mktemp("ref_vocab")
    c = _write_subset(str(d / "bpe_simple_vocab_16e6.txt"), sub["clip_merges"], lambda i: f"\ue000{i} \ue001")
    m = _write_subset(str(d / "merges.txt"), sub["open_clip_merges"], lambda i: f"\ue000{i} \ue001")
    v = _write_subset(str(d / "vocab.txt"), sub["open_clip_vocab"], lambda i: f"\ue000{i}")
    return {"clip": (ClipTokenizer(c), TO.ClipTokenizer(c)), "open_clip": (OpenClipTokenizer(m, v), TO.OpenClipTokenizer(m, v))}


def test_reference_known_answer_pins_the_oracle(real):
    """src/token/clip.rs:232-249, verbatim."""
    _, oracle = real["clip"]
    enc = oracle.encode(KAT_TEXT, False, False)
    assert enc == KAT_IDS
    assert oracle.decode(enc) == KAT_DECODE


def test_reference_known_answer_cxx(real):
    tok, _ = real["clip"]
    enc = tok.encode(KAT_TEXT, False, False)
    assert enc == KAT_IDS
    assert tok.decode(enc) == KAT_DECODE
    assert (tok.start_of_text_token(), tok.end_of_text_token(), tok.padding_token()) == (49406, 49407, 49407)
    otok, _ = real["open_clip"]
    assert otok.padding_token() == 0   # open_clip.rs:218-220


@pytest.mark.parametrize("which", ["clip", "open_clip"])
def test_real_vocab_vectors(real, which):
    tok, oracle = real[which]
    for i, p in enumerate(VEC["prompts"]):
        assert oracle.encode(p, False, False) == VEC[which]["encode"][i], p      # fixture is what the oracle says
        assert tok.encode(p, False, False) == VEC[which]["encode"][i], p
        assert tok.tokenize_text(p, 77) == VEC[which]["tokenize_text_77"][i], p
        assert tok.decode(VEC[which]["encode"][i]) == VEC[which]["decode"][i], p


def test_mini_vocab_vectors(mini):
    tok, oracle = mini
    for i, p in enumerate(VEC["prompts"]):
        assert oracle.encode(p, False, False) == VEC["mini"]["encode"][i], p
        assert tok.encode(p, False, False) == VEC["mini"]["encode"][i], p
        assert tok.tokenize_text(p, 77) == VEC["mini"]["tokenize_text_77"][i], p
        assert tok.decode(VEC["mini"]["encode"][i]) == VEC["mini"]["decode"][i], p


def test_case_fold_closure_of_letter_class():
    """The only code point outside L/N whose simple case variants are letters is U+0345 (see the oracle's PAT comment)."""
    import unicodedata as U
    found = set()
    for cp in range(0x110000):
        if 0xD800 <= cp <= 0xDFFF:
            continue
        c = chr(cp)
        for v in {c.lower(), c.upper(), c.title(), c.casefold()}:
            if len(v) == 1 and v != c and (U.category(c)[0] in "LN") != (U.category(v)[0] in "LN"):
                found.add(cp)
    assert found == {0x345}
    assert [m.group(0) for m in TO.regex.compile(TO.PAT).finditer("s\u0345 \u0345")] == ["s\u0345", "\u0345"]


def _fuzz_strings(n, seed):
    rng = random.Random(seed)
    pools = [
        (0x20, 0x7E), (0x20, 0x7E), (0x20, 0x7E), (0xA0, 0x24F), (0x370, 0x3FF), (0x400, 0x4FF), (0x5D0, 0x5EA), (0x660, 0x669),
        (0x900, 0x97F), (0x2000, 0x206F), (0x2150, 0x218F), (0x3040, 0x30FF), (0x4E00, 0x4E80), (0xFB00, 0xFB06), (0x1F600, 0x1F64F),
        (0x1D400, 0x1D433), (0x9, 0xD), (0x1C, 0x1F), (0x300, 0x36F),
    ]
    extra = ["'s", "'t", "'re", "'ve", "'m", "'ll", "'d", "<|startoftext|>", "<|endoftext|>", " ", "  ", "Σ", "ς", "İ", "ſ", "K", "'", "<|"]
    for _ in range(n):
        parts = []
        for _ in range(rng.randint(0, 24)):
            if rng.random() < 0.25:
                parts.append(rng.choice(extra))
            else:
                lo, hi = rng.choice(pools)
                parts.append("".join(chr(rng.randint(lo, hi)) for _ in range(rng.randint(1, 6))))
        s = "".join(parts).replace("\0", " ")
        yield "".join(ch for ch in s if not 0xD800 <= ord(ch) <= 0xDFFF)


def test_fuzz_cxx_equals_oracle_mini(mini):
    tok, oracle = mini
    n = 0
    for s in _fuzz_strings(400, 1234):
        assert tok.encode(s, True, True) == oracle.encode(s, True, True), repr(s)
        n += 1
    assert n == 400


def test_fuzz_cxx_equals_oracle_real(real):
    for which in ("clip", "open_clip"):
        tok, oracle = real[which]
        for s in _fuzz_strings(150, 99):
            try:
                want = oracle.encode(s, False, True)
            except KeyError:
                # piece not in the vocabulary: the reference panics (encoder[...] on a missing key); the library reports an error
                with pytest.raises(SdxlError, match="not in the vocabulary"):
                    tok.encode(s, False, True)
                continue
            assert tok.encode(s, False, True) == want, (which, repr(s))


def test_truncation_drops_end_of_text(mini):
    """tokenize_text resizes to seq_len (stablediffusion/mod.rs:787): a long prompt loses its <|endoftext|>."""
    tok, oracle = mini
    long = "cat " * 100
    got = tok.tokenize_text(long, 77)
    assert len(got) == 77 and got == TO.tokenize_text(long, oracle, 77) and 49407 not in got
    short = tok.tokenize_text("cat", 8)
    assert short[0] == 49406 and 49407 in short and short[-1] == 0


def test_errors_are_reported_not_thrown_across_the_abi():
    with pytest.raises(SdxlError, match="cannot open"):
        OpenClipTokenizer("/nonexistent/merges.txt", "/nonexistent/vocab.txt")
    with pytest.raises(SdxlError, match="cannot open"):
        ClipTokenizer("/nonexistent/bpe.txt")
    # a merges file that is too short for ClipTokenizer::new's hard-coded slice (clip.rs:98)
    with pytest.raises(SdxlError, match="needs"):
        ClipTokenizer(os.path.join(MINI, "mini_merges.txt"))


def test_invalid_utf8_is_replaced_like_from_utf8_lossy(mini):
    """The C ABI takes bytes: malformed UTF-8 decodes with U+FFFD per maximal invalid subpart (String::from_utf8_lossy, which a
    Rust caller converting from raw bytes would have applied) — same ids as the oracle on bytes.decode(errors="replace")."""
    import ctypes as C
    from sdxl_b200 import _lib
    tok, oracle = mini
    lib = _lib.load()
    for raw in (b"caf\xc3 au lait", b"\xff\xfe cat", b"x\xe2\x82 y", b"\xf0\x9f\x98 smile", b"ok \xed\xa0\x80 surrogate", b"\xc0\xaf overlong"):
        n = C.c_int(0)
        assert lib.sdxl_tokenizer_encode(tok.h, raw, 0, 0, None, 0, C.byref(n)) == 0
        buf = (C.c_uint32 * max(1, n.value))()
        assert lib.sdxl_tokenizer_encode(tok.h, raw, 0, 0, buf, n.value, C.byref(n)) == 0
        assert list(buf[:n.value]) == oracle.encode(raw.decode("utf-8", errors="replace"), False, False), raw


def test_open_clip_ids_match_huggingface_tokenizers(real):
    """Independent check: the ids the HuggingFace `tokenizers` runtime gives on the reference's own tokenizer.json (the file
    its vocab.txt / merges.txt were exported from, tokenizer/convert.py; stored in the vectors file) equal those of the oracle
    and the C++ tokenizer (NFC-stable prompts: tokenizer.json normalises with NFC, the reference's Rust code does not)."""
    tok, oracle = real["open_clip"]
    hf = VEC["huggingface_open_clip"]
    for p, want in zip(hf["prompts"], hf["encode"]):   # want includes <|startoftext|> / <|endoftext|>
        assert oracle.encode(p, True, True) == want, p
        assert tok.encode(p, True, True) == want, p
