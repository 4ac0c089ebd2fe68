"""Reference statement of sliding-window tiling and stitching (include/bsq.h, bsq_tile / bsq_untile_mean) in numpy."""
import numpy as np

SHORT, END, DROP = 0, 1, 2
TAILS = {"short": SHORT, "end": END, "drop": DROP}


def windows(n, W, S, tail):
    """[(start, length)] of one sequence of n residues."""
    tail = TAILS.get(tail, tail)
    if n <= W:
        return [(0, n)]
    if tail == DROP:
        m = (n - W) // S + 1
        return [(j * S, W) for j in range(m)]
    m = -(-(n - W) // S) + 1
    if tail == SHORT:
        return [(j * S, min(W, n - j * S)) for j in range(m)]
    return [(j * S, W) for j in range(m - 1)] + [(n - W, W)]


def tile(buf, offs, W, S, tail):
    """-> (bytes, out_offsets, seq_ptr, seq_index, starts) of a packed batch, all numpy."""
    offs = np.asarray(offs, np.int64)
    n = offs.size - 1
    parts, out_o, seq_ptr, seq_index, starts = [], [0], [0], [], []
    for i in range(n):
        s = int(offs[i])
        for st, ln in windows(int(offs[i + 1]) - s, W, S, tail):
            parts.append(np.asarray(buf[s + st:s + st + ln], np.uint8))
            out_o.append(out_o[-1] + ln)
            seq_index.append(i)
            starts.append(st)
        seq_ptr.append(len(seq_index))
    b = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
    return (b, np.array(out_o, np.int64), np.array(seq_ptr, np.int64), np.array(seq_index, np.int64),
            np.array(starts, np.int64))


def untile(y, lens, W, S, tail, row_base, col0, strands=1, flipped=None):
    """The per-residue mean of window outputs, as an explicit float32 loop in the header's order.

    y: 2-D (rows, C) view of the outputs (any float dtype, converted exactly to float32); row_base(w): window w's first
    row; lens: the source lengths; flipped: strands * M flags or None.  -> float32 (sum lens, C)."""
    y = np.asarray(y)
    C = y.shape[1]
    tail = TAILS.get(tail, tail)
    wins = [windows(int(n), W, S, tail) for n in lens]
    M = sum(len(w) for w in wins)
    out = np.empty((int(sum(lens)), C), np.float32)
    row, w0 = 0, 0
    for i, n in enumerate(lens):
        for p in range(int(n)):
            acc = np.zeros(C, np.float32)
            cnt = 0
            for strand in range(strands):
                for j, (st, ln) in enumerate(wins[i]):
                    if not st <= p < st + ln:
                        continue
                    w = w0 + j + strand * M
                    t = p - st
                    if flipped is not None and flipped[w]:
                        t = ln - 1 - t
                    acc = (acc + y[row_base(w) + col0 + t].astype(np.float32)).astype(np.float32)
                    cnt += 1
            out[row] = acc / np.float32(cnt) if cnt else np.float32(np.nan)
            row += 1
        w0 += len(wins[i])
    return out
