"""Reference statement of translation (include/bsq.h, bsq_translate) in numpy, built from the rule itself, not from the
library's tables."""
import itertools

import numpy as np

CODES = {
    1: "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    2: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIMMTTTTNNKKSS**VVVVAAAADDEEGGGG",
    4: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
    5: "FFLLSSSSYY**CCWWLLLLPPPPHHQQRRRRIIMMTTTTNNKKSSSSVVVVAAAADDEEGGGG",
    6: "FFLLSSSSYYQQCC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG",
}
CODES[11] = CODES[1]

IUPAC = {"A": "A", "C": "C", "G": "G", "T": "T", "U": "T", "R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC",
         "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGT"}
COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}
TCAG = {"T": 0, "C": 1, "A": 2, "G": 3}
BIT = {"A": 1, "C": 2, "G": 4, "T": 8}


def code_string(code):
    return CODES[code] if isinstance(code, int) else (code.decode("latin-1") if isinstance(code, bytes) else code)


def base_set(byte):
    """The bases byte value ``byte`` stands for ("" = invalid)."""
    c = chr(byte).upper() if byte < 0x80 else ""
    return IUPAC.get(c, "") if c else ""


def codon_letter(s0, s1, s2, code):
    """The letter of a triple of base sets (strings of bases) under a 64-letter code."""
    if not (s0 and s1 and s2):
        return "X"
    letters = {code[16 * TCAG[a] + 4 * TCAG[b] + TCAG[c]] for a, b, c in itertools.product(s0, s1, s2)}
    return letters.pop() if len(letters) == 1 else "X"


def tables(code):
    """(masks[256], codons[4096]) as numpy uint8: what bsq_translate_table returns."""
    code = code_string(code)
    masks = np.array([sum(BIT[b] for b in base_set(x)) for x in range(256)], np.uint8)
    sets = ["".join(b for b in "ACGT" if m & BIT[b]) for m in range(16)]
    codons = np.array([ord(codon_letter(sets[i >> 8], sets[(i >> 4) & 15], sets[i & 15], code)) for i in range(4096)], np.uint8)
    return masks, codons


def frame_len(n, frame):
    k = abs(frame)
    return max(0, (n - (k - 1)) // 3)


def translate_seq(seq, frame, code=1):
    """One frame of one sequence (bytes or str), codon by codon, as the header words it -> str."""
    code = code_string(code)
    s = seq.encode("latin-1") if isinstance(seq, str) else bytes(seq)
    n, k = len(s), abs(frame)
    out = []
    for t in range(frame_len(n, frame)):
        if frame > 0:
            sets = [base_set(s[k - 1 + 3 * t + d]) for d in range(3)]
        else:
            sets = ["".join(COMP[b] for b in base_set(s[n - k - 3 * t - d])) for d in range(3)]
        out.append(codon_letter(*sets, code))
    return "".join(out)


_TABLE_CACHE = {}


def translate(buf, offs, frames, code=1):
    """-> (bytes, out_offsets) of a packed batch, vectorised in numpy (what the GPU tests compare bit for bit)."""
    key = code_string(code)
    if key not in _TABLE_CACHE:
        _TABLE_CACHE[key] = tables(key)
    masks, codons = _TABLE_CACHE[key]
    cmask = np.array([int(f"{m:04b}"[::-1], 2) for m in range(16)], np.uint8)[masks]
    buf = np.asarray(buf, np.uint8)
    offs = np.asarray(offs, np.int64)
    n, F = offs.size - 1, len(frames)
    lens = np.diff(offs)
    L = np.stack([np.maximum(0, (lens - (abs(f) - 1)) // 3) for f in frames], 1) if n else np.zeros((0, F), np.int64)
    out_o = np.zeros(n * F + 1, np.int64)
    np.cumsum(L.reshape(-1), out=out_o[1:])
    total = int(out_o[-1])
    out = np.zeros(total, np.uint8)
    for fi, f in enumerate(frames):
        rows = np.arange(n) * F + fi
        cnt = L[:, fi]
        if cnt.sum() == 0:
            continue
        row = np.repeat(np.arange(n), cnt)
        t = np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        dst = out_o[rows][row] + t
        k = abs(f)
        if f > 0:
            p = offs[row] + k - 1 + 3 * t
            m0, m1, m2 = masks[buf[p]], masks[buf[p + 1]], masks[buf[p + 2]]
        else:
            p = offs[row] + lens[row] - k - 3 * t
            m0, m1, m2 = cmask[buf[p]], cmask[buf[p - 1]], cmask[buf[p - 2]]
        out[dst] = codons[(m0.astype(np.int64) << 8) | (m1.astype(np.int64) << 4) | m2]
    return out, out_o
