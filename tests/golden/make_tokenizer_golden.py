"""Generates the tokenizer fixtures from the ORACLE (oracle/tokenizer_oracle.py — pinned by the reference's own
known-answer vector, see its header):

  tests/golden/mini_bpe/{mini_merges.txt,mini_vocab.txt}   a small synthetic BPE vocabulary (trained here on PROMPTS with a plain
                                                 most-frequent-pair loop) so the C++ tokenizer can be tested on machines that do
                                                 not have the reference's vocabulary files (the GPU box);
  tests/golden/tokenizer_vectors.json            prompt -> ids for (a) the mini vocabulary, (b) the reference's real CLIP and
                                                 OpenCLIP vocabularies, (c) the HuggingFace `tokenizers` runtime on the
                                                 reference's tokenizer.json (the file its OpenCLIP vocab.txt / merges.txt were
                                                 exported from);
  tests/golden/tokenizer_ref_subset.json         the entries of the real vocabularies that the test corpus reaches, at their
                                                 original positions (see `ref_subset`).

(b), (c) and the subset need the reference's tokenizer directory (the repository's tokenizer/ folder of
Gadersd/stable-diffusion-xl-burn), given as $SDXL_TOKENIZER_DIR; without it the committed copies are kept.

    SDXL_TOKENIZER_DIR=<reference>/tokenizer python tests/golden/make_tokenizer_golden.py
"""
import collections
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "stable-diffusion-xl-burn_b200"))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import tokenizer_oracle as T  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
REF_TOK = os.environ.get("SDXL_TOKENIZER_DIR")

PROMPTS = [
    "a photo of a cat",
    "Hello world! <|startoftext|>asdf<|startoftext|>",
    "  An   astronaut riding\ta horse\non Mars,  4k, highly-detailed!!  ",
    "it's the artist's 1st painting; they've said we'll see, I'm sure he'd've",
    "Ünïcödé façade — naïve café 北京 東京 \U0001F600\U0001F3A8 ﬁn ǅ İstanbul "
    "ΣΊΣΥΦΟΣ ΟΔΟΣ",
    "ſtart 'ſ <|ſtartoftext|> <|ENDOFTEXT|> Kelvin",
    "1234567890 ½ ٣ ² x²+y³",
    "",
    "   ",
    "\u00a0\u2003 weird\u3000spaces\u0085x tab\x1cseparator \u2028line\u200bzero",
    "a cinematic photograph of an elderly lighthouse keeper standing on a rocky cliff at dusk, dramatic storm clouds, "
    "crashing waves, volumetric light from the lamp room, 35mm film grain, shallow depth of field, award winning, "
    "ultra detailed, masterpiece, trending on artstation, by greg rutkowski and alphonse mucha and studio ghibli, 8k uhd",
    "don't can't won't 'tis 'twas 'll 're 'd!!! ??? ... --- ___ <<|>> <|endoftext|>",
]


def train_mini(corpus, n_merges):
    """Plain BPE training on byte-encoded words (ties broken by first occurrence); returns merges."""
    be = dict(T.bytes_to_unicode())
    pat = T.regex.compile(T.PAT)
    words = collections.Counter()
    for text in corpus:
        for m in pat.finditer(T.whitespace_clean(text).lower()):
            tok = [be[b] for b in m.group(0).encode("utf-8")]
            tok[-1] += "</w>"
            words[tuple(tok)] += 1
    merges = []
    for _ in range(n_merges):
        pairs = collections.Counter()
        for w, c in words.items():
            for p in zip(w, w[1:]):
                pairs[p] += c
        if not pairs:
            break
        best = max(pairs.items(), key=lambda kv: kv[1])[0]
        merges.append(best)
        nw = collections.Counter()
        for w, c in words.items():
            out, i = [], 0
            while i < len(w):
                if i < len(w) - 1 and (w[i], w[i + 1]) == best:
                    out.append(w[i] + w[i + 1])
                    i += 2
                else:
                    out.append(w[i])
                    i += 1
            nw[tuple(out)] += c
        words = nw
    return merges

# NFC-stable prompts: tokenizer.json normalises with NFC, the reference's Rust code does not
HF_PROMPTS = ["a photo of a cat", "An astronaut riding a horse on Mars, 4k, highly-detailed!!",
              "it's the artist's 1st painting; they've said we'll see", "Ünïcödé façade naïve café", "x²+y³ = 42 %"]


class _Seen(dict):
    """A dict that remembers which keys were read."""

    def __init__(self, d):
        super().__init__(d)
        self.seen = set()

    def __getitem__(self, k):
        v = super().__getitem__(k)
        self.seen.add(k)
        return v


def ref_subset(ref_dir):
    """The real vocabularies cut down to what the tests' corpus reaches, each kept entry at its original position.

    An encode reads only the ranks of merge pairs that occur side by side in a word and the ids of the pieces it emits. A
    file that keeps those entries where they were, and fills every other position with a placeholder built on U+E000 (a code
    point the byte-level alphabet never produces, so a placeholder can neither match a pair nor shadow a piece), tokenizes
    the corpus exactly as the full file does: the same merges in the same order, the same ids, the same missing-piece
    errors. The CLIP vocabulary is the merges file itself, so there a merge whose concatenation is an emitted piece stays too.
    """
    import test_tokenizer as TT
    corpus = PROMPTS + HF_PROMPTS + list(TT._fuzz_strings(150, 99))
    clip_path = os.path.join(ref_dir, "clip", "bpe_simple_vocab_16e6.txt")
    oc_merges, oc_vocab = os.path.join(ref_dir, "open_clip", "merges.txt"), os.path.join(ref_dir, "open_clip", "vocab.txt")
    c, o = T.ClipTokenizer(clip_path), T.OpenClipTokenizer(oc_merges, oc_vocab)
    for t in (c, o):
        t.bpe_ranks, t.encoder = _Seen(t.bpe_ranks), _Seen(t.encoder)
        for s in corpus:
            try:
                t.encode(s, True, True)
            except KeyError:   # a piece the vocabulary lacks: the tests expect the same error from the subset
                pass

    def table(keep, n=None):
        return {"n": n or max(keep) + 1, "keep": {str(i): keep[i] for i in sorted(keep)}}

    hi = 49152 - 256 - 2 + 1   # ClipTokenizer uses merges[1:hi]
    clip = {i: f"{a} {b}" for i, (a, b) in enumerate(T.load_merges(clip_path)[:hi])
            if i >= 1 and ((a, b) in c.bpe_ranks.seen or a + b in c.encoder.seen)}
    om = {i: f"{a} {b}" for i, (a, b) in enumerate(T.load_merges(oc_merges)) if (a, b) in o.bpe_ranks.seen}
    with open(oc_vocab, encoding="utf-8", newline="\n") as f:
        vocab = [ln[:-1] if ln.endswith("\n") else ln for ln in f]
    vocab = [v[:-1] if v.endswith("\r") else v for v in vocab]
    ov = {i: v for i, v in enumerate(vocab) if v in o.encoder.seen}
    return {"clip_merges": table(clip, hi), "open_clip_merges": table(om), "open_clip_vocab": table(ov)}


def main():
    mini = os.path.join(HERE, "mini_bpe")
    os.makedirs(mini, exist_ok=True)
    merges = train_mini(PROMPTS, 400)
    chars = [u for _, u in T.bytes_to_unicode()]
    vocab = ["<pad>"] + chars + [c + "</w>" for c in chars] + [a + b for a, b in merges]
    vocab += ["<|startoftext|>", "<|endoftext|>"]
    # ids 49406 / 49407 are hard-coded in the reference (clip.rs:215-221); the mini vocabulary is smaller, so sot/eot ids
    # simply do not decode — encode() never looks them up.
    with open(os.path.join(mini, "mini_merges.txt"), "w", encoding="utf-8", newline="\n") as f:
        f.write("#version:mini\n")  # a one-word line: load_merges skips it
        for a, b in merges:
            f.write(f"{a} {b}\n")
    with open(os.path.join(mini, "mini_vocab.txt"), "w", encoding="utf-8", newline="\n") as f:
        for v in vocab:
            f.write(v + "\n")
    out = {"prompts": PROMPTS, "mini": {}, "clip": {}, "open_clip": {}}
    tok = T.OpenClipTokenizer(os.path.join(mini, "mini_merges.txt"), os.path.join(mini, "mini_vocab.txt"))
    out["mini"]["encode"] = [tok.encode(p, False, False) for p in PROMPTS]
    out["mini"]["tokenize_text_77"] = [T.tokenize_text(p, tok, 77) for p in PROMPTS]
    out["mini"]["decode"] = [tok.decode(e) for e in out["mini"]["encode"]]
    if REF_TOK and os.path.isdir(REF_TOK):
        c = T.ClipTokenizer(os.path.join(REF_TOK, "clip", "bpe_simple_vocab_16e6.txt"))
        o = T.OpenClipTokenizer(os.path.join(REF_TOK, "open_clip", "merges.txt"), os.path.join(REF_TOK, "open_clip", "vocab.txt"))
        for name, t in (("clip", c), ("open_clip", o)):
            out[name]["encode"] = [t.encode(p, False, False) for p in PROMPTS]
            out[name]["tokenize_text_77"] = [T.tokenize_text(p, t, 77) for p in PROMPTS]
            out[name]["decode"] = [t.decode(e) for e in out[name]["encode"]]
        import tokenizers
        hf = tokenizers.Tokenizer.from_file(os.path.join(REF_TOK, "tokenizer.json"))
        out["huggingface_open_clip"] = {"prompts": HF_PROMPTS, "encode": [hf.encode(p).ids for p in HF_PROMPTS]}
        subset = ref_subset(REF_TOK)
        with open(os.path.join(HERE, "tokenizer_ref_subset.json"), "w", encoding="utf-8") as f:
            json.dump(subset, f, ensure_ascii=False, indent=0)
        print("subset entries", {k: len(v["keep"]) for k, v in subset.items()})
    else:
        print("WARNING: reference tokenizer files not found; real-vocabulary vectors not regenerated", file=sys.stderr)
        old = json.load(open(os.path.join(HERE, "tokenizer_vectors.json")))
        for k in ("clip", "open_clip", "huggingface_open_clip"):
            out[k] = old[k]
    with open(os.path.join(HERE, "tokenizer_vectors.json"), "w", encoding="utf-8") as f:
        json.dump(out, f, ensure_ascii=True, indent=0)
    print("mini merges", len(merges), "vocab", len(vocab), "prompts", len(PROMPTS))


if __name__ == "__main__":
    main()
