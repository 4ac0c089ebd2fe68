"""Test infrastructure: the sequence-packing rule of include/bsq.h (bsq_seqpack_plan / bsq_tokenize_seqpack) stated
again in plain Python, one sequence and one row at a time.

``plan`` is best-fit decreasing exactly as the header words it (a quadratic scan over the open rows, which is what the
library's bucketed planner must agree with); ``pack`` lays given per-sequence token rows (for example the rows of
``batch_tokenize_varlen``) out in the planned rows with the padding value and the position ids.
"""
import numpy as np

INT32_MAX = 2 ** 31 - 1


def plan(lens, k, L, rows=None):
    """-> dict(R, starts, row_ptr, row_seq, cu_seqlens, max_seqlen) for sequence lengths ``lens`` (already cropped).
    ValueError where the header says BSQ_ERR_ARG."""
    lens = [int(x) for x in lens]
    need = [x + k for x in lens]
    for w in need:
        if w > L:
            raise ValueError(f"seq len + bos + eos > padlen: {w}, vs padlen {L}")
    order = sorted((i for i in range(len(need)) if need[i] > 0), key=lambda i: -need[i])  # stable: ties to the lower index
    fill, content = [], []  # per row: tokens used, sequences in column order
    starts = [-1] * len(need)
    for i in order:
        best = None
        for r in range(len(fill)):
            room = L - fill[r]
            if room >= need[i] and (best is None or room < L - fill[best]):
                best = r
        if best is None:
            fill.append(0)
            content.append([])
            best = len(fill) - 1
        starts[i] = best * L + fill[best]
        fill[best] += need[i]
        content[best].append(i)
    R = len(fill)
    if rows is not None:
        if R > rows:
            raise ValueError(f"the batch needs {R} rows, more than rows = {rows}")
        fill += [0] * (rows - R)
        content += [[] for _ in range(rows - R)]
        R = rows
    if R * L > INT32_MAX:
        raise ValueError("R * L exceeds 2^31 - 1")
    cu, longest = [], 0
    for r in range(R):
        for i in content[r]:
            cu.append(starts[i])
            longest = max(longest, need[i])
        if fill[r] < L:
            cu.append(r * L + fill[r])
            longest = max(longest, L - fill[r])
    cu.append(R * L)
    row_ptr = [0]
    for r in range(R):
        row_ptr.append(row_ptr[-1] + len(content[r]))
    return dict(R=R, starts=np.array(starts, np.int64), row_ptr=np.array(row_ptr, np.int64),
                row_seq=np.array([i for c in content for i in c], np.int64), cu_seqlens=np.array(cu, np.int32),
                max_seqlen=longest)


def pack(p, seq_rows, L, pad_value, dtype, pad_label=None, label_rows=None):
    """The expected ``(R, L)`` tokens and int32 position ids (and labels when ``label_rows`` is given) of plan ``p``
    with sequence ``i``'s tokens ``seq_rows[i]``."""
    R = p["R"]
    tokens = np.full(R * L, pad_value, dtype=dtype)
    labels = None if label_rows is None else np.full(R * L, pad_label, dtype=np.int64)
    pos = np.zeros(R * L, dtype=np.int32)
    cu = p["cu_seqlens"]
    for a, b in zip(cu[:-1], cu[1:]):
        pos[a:b] = np.arange(b - a, dtype=np.int32)
    for i, s in enumerate(p["starts"]):
        if s < 0:
            continue
        tokens[s:s + len(seq_rows[i])] = seq_rows[i]
        if labels is not None:
            labels[s:s + len(label_rows[i])] = label_rows[i]
    out = (tokens.reshape(R, L), pos.reshape(R, L))
    return out if labels is None else out + (labels.reshape(R, L),)
