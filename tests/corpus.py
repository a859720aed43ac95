"""Shared test corpora: the fixture strings of BASELINE config #1 (SURVEY.md section 4 items 1-4 and
the quirk corpus of section 8c) and a seeded mixed-Unicode fuzz generator."""
from __future__ import annotations

import numpy as np

# strings the reference itself names (default_tokenizer.py:195-198, numpy_tokenizer.py:286,
# time_tokenizer.py:113) followed by the quirk corpus (SURVEY.md 8a Q1-Q12, 8c).
FIXTURES = [
    "This is a #test! Testing, Testing, 1 2 3",
    "can\u2019t wait to get my glasses back \U0001F913",
    "IKR!! IM LIKE \"WHERE'S MY DADDY AT? \U0001F440) https://t.co/jM3qLZijMc",
    "$#@^:a./",
    "This is a test line, just to get things warmed up...",
    " ",
    "a",
    "ab",
    "abc",
    "a b",
    "  ",
    "a  b",
    " a",
    "a ",
    "!",
    "!!",
    "! ",
    " !",
    "a@b",
    "#foo",
    " #a b,c",
    "#a,b c,d",
    "fooBar, a@b",
    "a@b.c,d@e.f fooBar, x-y z",
    "a@b,c@d,e@f one,two three,four five,six",
    "a@b,c@d,e@f  one,two   three,four five,six",
    "camelCaseWord HTTPServer XMLHttpRequest",
    "see http://foo.com/bar?x=1#frag and more",
    "email me at joe.blow@example.com or .@joe ok",
    ".@joe",
    "x .@joe, y",
    "@",
    "@a",
    "a@",
    "$AAPL ^GSPC #tag @user",
    "$ AAPL # tag",
    "http://",
    "a://b",
    "1://b ://",
    "\u65e5\u672c\u8a9e\u306e\u30c6\u30ad\u30b9\u30c8\u3001\u3067\u3059\u3002",
    "\u00dcn\u00efc\u00f6d\u00e9 \u01c4 \u01c5 \u01c6 \u00bd \u00b2 \u0663",
    "tab\tnew\nline\xa0nbsp\u3000ideo",
    "zero\u200bwidth\u00adsoft\ufeffbom",
    "\u24b6\u24d0 circled \u2160\u2170 roman",
    "lone \ud800 surrogate \udfff end",
    "\U0010ffff max \U000e0100 vs \U0003134f",
    "emoji\U0001F600\U0001F64Fend \U0001F1FA\U0001F1F8",
    "\u2028line\u2029para\u0085nel\u1680ogham\u205fmmsp",
    "a\u0301e\u0301 combining",
    "x" * 127,
    "y" * 128,
    "ab " * 85,            # 255 chars
    "ab " * 85 + "c",      # 256
    "ab " * 85 + "cd",     # 257
    "#" * 64,
    "a@b " * 70,
    "A" * 250,
    ("word " * 40 + "http://t.co/abc ") * 3,
]

EMPTY = ""  # Q1: reference raises IndexError; batch API returns zero characters / zero tokens

_ASCII_WORD = "abcdefghijklmnopqrstuvwxyz"
_POOLS = {
    "lower": _ASCII_WORD,
    "upper": _ASCII_WORD.upper(),
    "digit": "0123456789",
    "punct": ".,!?'\"():;-_/\\@#$^&*+=<>[]{}|~`%",
    "space": " \t\n\r\x0b\x0c\x1c\x1d\x1e\x1f\x85\xa0\u1680\u2000\u2005\u200a\u2028\u2029\u202f\u205f\u3000",
    "latin": "".join(chr(c) for c in range(0xC0, 0x250)),
    "cjk": "".join(chr(c) for c in list(range(0x4E00, 0x4E80)) + list(range(0x3040, 0x30FF)) + list(range(0xAC00, 0xAC40))),
    "emoji": "".join(chr(c) for c in range(0x1F600, 0x1F650)),
    "mbpunct": "\u3001\u3002\u300c\u300d\u2026\u2014\u2019\u201c\u201d\u00b7\u00a1\u00bf",
    "numeric": "\u00bd\u00b2\u0663\u2160\u2170\u3007\u0969\u2460",
    "odd": "\u200b\u00ad\ufeff\x00\x01\x7f\u0080\u009f\ud800\udfff\U0010ffff\U000e0100\U000e01ef\U0003134f\u01c5\u24b6\u24d0\u0345",
}
_SPECIALS = ["@", "#", "$", "^", ":", "/", ".", "://", ".@", " .@", " #", " @", "@@", "//"]


def fuzz_string(rng: np.random.Generator, max_len: int = 60, profile: str = "mixed") -> str:
    n = int(rng.integers(0, max_len + 1))
    if profile == "ascii":
        pools, weights = ["lower", "upper", "digit", "punct", "space"], [0.5, 0.1, 0.08, 0.12, 0.2]
    elif profile == "marks":
        pools, weights = ["lower", "upper", "digit", "punct", "space"], [0.45, 0.05, 0.05, 0.1, 0.1]
    else:
        pools = list(_POOLS)
        weights = [0.25, 0.06, 0.05, 0.1, 0.14, 0.08, 0.08, 0.05, 0.05, 0.04, 0.10]
    weights = np.array(weights) / np.sum(weights)
    out = []
    while len(out) < n:
        if profile != "ascii" and rng.random() < (0.25 if profile == "marks" else 0.08):
            out.extend(_SPECIALS[int(rng.integers(len(_SPECIALS)))])
            continue
        pool = _POOLS[pools[int(rng.choice(len(pools), p=weights))]]
        run = int(rng.integers(1, 5))
        for _ in range(run):
            out.append(pool[int(rng.integers(len(pool)))])
    return "".join(out[:n])


def fuzz_strings(seed: int, count: int, max_len: int = 60, profile: str = "mixed"):
    rng = np.random.default_rng(seed)
    return [fuzz_string(rng, max_len, profile) for _ in range(count)]


# ---- long-string scenarios of the tokenize kernel (test_gpu_parity.py, test_gpu_extended.py, test_gpu_rules.py) --------
# Bytes owned per unit of work (latok_internal.h): a range (one warp) and a tile (the ranges of one CTA, one look-back
# record) in both geometries of the tokenize kernel (long strings: 3 968-byte ranges x 9, short strings: 2 944 x 11);
# the scenarios place interesting things around multiples of each, and around 7 936 bytes, a size that cuts ranges at
# other phases.
RANGES = (3968, 2944)
UNITS = (3968, 7936, 9 * 3968, 2944, 11 * 2944)
ALIGN_PATTERNS = ["a@b.c", " #tag ", "x http://t.co/abc y", "fooBar", ".@joe ", "éè 日本 \U0001F600!", "a, b",
                  "  ", "!! ", "e@f,g@h,i@j one,two three,four "]
STRADDLE_CHARS = ["é", "日", "\U0001F600", "　", "\u2028"]


def long_doc(rng: np.random.Generator, n_chars: int, profile: str = "ascii") -> str:
    parts, total = [], 0
    while total < n_chars:
        s = fuzz_string(rng, 200, profile)
        parts.append(s)
        parts.append(" " if rng.random() < 0.7 else "\n")
        total += len(s) + 1
    return "".join(parts)[:n_chars]


def long_documents():
    """Fuzz documents of 70 000 characters and of a few bytes around 1, 2 and 3 times every unit of work."""
    rng = np.random.default_rng(42)
    sizes = [(70000, "ascii"), (50000, "mixed"), (33000, "marks"), (100, "ascii")]
    for u in UNITS:
        sizes += [(u, "ascii"), (u + 1, "ascii"), (u - 1, "ascii"), (2 * u, "ascii"), (3 * u + 5, "mixed")]
    return [long_doc(rng, int(n), p) for n, p in sizes]


def alignment_sweep(unit: int):
    """Every pattern of ALIGN_PATTERNS slid across byte `unit` one byte at a time, one string per case."""
    texts = []
    for pat in ALIGN_PATTERNS:
        for shift in range(-8, 6):
            pad = unit + shift - 3
            texts.append("w" * 5 + " " + "z" * (pad - 6) + pat + " tail end")
    return texts


def alignment_sweep_steps():
    """The same patterns against the 1 KB steps inside a range and against the 116-byte closer search windows."""
    texts = []
    for pat in ALIGN_PATTERNS:
        for base in (1024, 2048, 3072, 3968 + 116, 3968 + 128, 4096, 2 * 3968 + 116, 2944 + 116, 2944 + 128, 2 * 2944 + 116):
            for shift in range(-6, 5):
                texts.append("q r " + "z" * (base + shift - 8) + " " + pat + " tail end")
    return texts


def multibyte_straddle(ch: str):
    """40 copies of `ch` starting a few bytes before every unit and 1 KB step: the character straddles the boundary."""
    texts = []
    for unit in UNITS + (1024, 2048, 4096):
        for shift in range(0, 6):
            texts.append("a" * (unit - shift) + ch * 40 + " b")
            texts.append("a b " * ((unit - shift) // 4 - 1) + "a" * ((unit - shift) % 4 + 4) + ch * 40 + " b")
    return texts


def space_free_runs():
    """Chunks longer than the right halo (they force the look-ahead walk), with a mark at their start or end or none,
    after text that ends near a tile boundary."""
    cases = []
    for TILE, run in ((7936, 300), (7936, 1000), (7936, 7936 - 50), (7936, 7936 + 300), (7936, 2 * 7936 + 77), (7936, 40000),
                      (3968, 100), (3968, 130), (3968, 3968 + 300), (35712, 200), (35712, 35712 + 5000), (31744, 200), (3968, 70000),
                      (2944, 100), (2944, 130), (2944, 2944 + 300), (32384, 200), (32384, 32384 + 5000), (2944, 70000)):
        base = "x y " * ((TILE - 120) // 4)
        cases.append(base + " " + ",".join(["ab"] * (run // 3)) + " end")                    # no mark: commas split
        cases.append(base + " " + ",".join(["ab"] * (run // 3)) + ",q@r end")                # mark at the very end
        cases.append(base + " " + ",".join(["ab"] * (run // 3)) + ",http://x.y/z end")
        cases.append(base + " #" + ",".join(["ab"] * (run // 3)) + " end,more stuff")        # mark at the start
        cases.append(base + " " + ",".join(["ab"] * (run // 3)))                             # run reaches end of string
        cases.append(base + " " + ",".join(["ab"] * (run // 3)) + "@z")                      # mark, then end of string
    return cases


def cjk_runs():
    """A space-free run of multi-byte characters after every unit."""
    return ["y" * (u - 100) + " " + "日、" * 3000 + "a@b 日 end" for u in UNITS]


def backlog_across_tiles():
    """k marks in one whitespace chunk blank the following k-1 chunks too; the backlog crosses tile boundaries and
    string boundaries (it must reset at each string start)."""
    many = ",".join(f"a{i}@b" for i in range(40))
    words = " ".join(f"w{i},x" for i in range(60))
    texts = []
    for u in UNITS:
        texts += ["p" * (u - 200) + " " + many + " " + words, "p" * (u - 30) + " " + many + " " + words,
                  "p q " * ((u - 200) // 4) + many + " " + words, "p q " * ((u - 40) // 4) + many + " " + words]
    texts += [
        many + " " + " ".join(f"w{i},x" for i in range(3000)),
        ",".join(f"a{i}@b" for i in range(5000)) + " " + " ".join(f"w{i},x" for i in range(6000)),
        many, words, many + " " + words,
        many + "   " + words,       # empty chunks also consume backlog
    ]
    return texts


HANDOFF_MARKS = ["aa@bb,cc@dd xx", "aa@bb,cc@dd,ee@ff,gg@hh xx yy zz", "http://a.b/c,x@y,#t d@e.f,g@h uu vv ww",
                 "a@b,c@d,e@f,g@h,i@j,k@l,m@n one two three four five six seven"]


def handoff_between_ranges():
    """One multi-mark chunk near the end of each of 20+ ranges (2 tiles + 2), swept over the range end."""
    filler = "lorem ipsum dolor sit amet consectetur "
    texts = []
    for shift, R in [(sh, R) for R in RANGES for sh in range(0, 64, 3 if R == 3968 else 7)]:
        for m in HANDOFF_MARKS:
            parts, pos = [], 0
            for k in range(1, 21 if R == 3968 else 25):
                target = R * k - 20 + shift - len(m) // 2
                pad = max(target - pos, 1)
                fill = (filler * (pad // len(filler) + 1))[:pad - 1] + " "
                parts += [fill, m + " "]
                pos += len(fill) + len(m) + 1
            texts.append("".join(parts))
    return texts


def handoff_long_tail():
    """The chunks of HANDOFF_MARKS with no space after them for a long while: the backlog is carried through ranges."""
    return ["pre fix " + m + " " + ("word,word;word/" * 1200) + " end tail a b c" for m in HANDOFF_MARKS]


def token_over_whole_range():
    """Strings without a split point, of 4-byte characters a few bytes longer than a range: the token begins in one
    range, covers the next one and ends within the closer search window of the third, at every alignment."""
    texts = [chr(0x20000 + j) * n for j in range(700) for n in (997,)] + [chr(0x4E00 + j) * 1325 for j in range(500)]
    texts += [chr(0x20000 + j) * n for j in range(300) for n in (993, 1001, 1012)]
    return texts


def tokens_spanning_ranges(range_bytes: int):
    """One token that covers 2, 3 and 10 whole ranges (the last one crosses a tile boundary), started and ended at
    drifting offsets."""
    texts = []
    for k in range(40):
        for nr in (2, 3, 10):
            n = nr * range_bytes + (k * 53) % 257 - 128
            texts.append("lead " * (k % 7) + "x" * n + " tail word")
            texts.append("日" * (n // 3) + " z")
    return texts


def token_feature_rows(range_bytes: int):
    """Steps with few, many and more than 512 token ends, rows at every phase of a 16-byte chunk, tokens around the
    uint8 wrap of the sums, tokens that begin several lane-words / steps / ranges before they end."""
    texts = []
    for k in range(48):
        lead = "w " * k                                  # k tokens in front: the rows of what follows start at every phase
        texts.append(lead + "a,b" * 700)                 # one token end per character: > 512 per 1 KB step (fallback path)
        texts.append(lead + "!?" * (300 + 7 * k))        # symbols only
        texts.append(lead + "ab cd, " * (140 + k))       # ordinary density, ~170 rows per step
        texts.append(lead + ("x" * (250 + k) + " ") * 9) # tokens around the uint8 wrap (250..297 characters)
        texts.append(lead + "é" * (260 + 3 * k) + " 日本語 " + "y" * (1000 + 37 * k) + " z")
        texts.append(lead + "tok " * 3 + "q" * (range_bytes + 100 * k) + ",end")     # a token that began a range earlier
        texts.append("z" * k)                            # a few bytes, also the empty string
    return texts


def token_feature_rows_at_capacity():
    """505..520 token ends in the first step of a string, then sparse text."""
    return [(",a" * (250 + j) + " " + "word " * 300) for j in range(0, 12)]


TINY_BATCHES = (["a"], ["a b"], ["a b c d e f"], ["", "a", "", "b c"])
