"""Read 2 of each ligation-oligo design beside M13 (collapse.py:172-189), made from read 2 as the synthetic generator writes
it -- TEST INFRASTRUCTURE for the GPU tests and the measuring tools.

The recorder of tests/golden/collapse_cases_oligos.json.gz (oracle/make_golden_collapse_oligos.py) holds the same table,
but importing it loads the reference environment, which exists only where the fixtures are recorded.
tests/test_oligo_layouts.py keeps the two tables identical."""
import numpy as np

# the generator writes read 2 as: M13 spacer (22), N6, I8 spacer (8), N6, the rest
LAYOUTS = {
    # oligo: (read 2 of that design from the generator's read 2, where its first hexamer starts)
    "I8": (lambda b: "GTCGTGAT" + b[22:] + b[:14][::-1], 8),
    "I8_single": (lambda b: b[22:28] + "ATCACGAC" + b[36:] + b[:22][::-1], 0),
    "NEBIO": (lambda b: b[22:28] + b[36:42] + b[42:47] + "A" + "TACGGG" + b[47:] + b[:23][::-1], 0),
    "TAKARA": (lambda b: b[22:28] + b[36:42] + "GTACGGG" + b[42:] + b[:23][::-1], 0),
}


def relayout_array(reads, oligo):
    """LAYOUTS[oligo] over many reads at once: uint8 array (n, width) of generator read 2 -> the same shape, re-laid out.
    The layout is applied once to a string of distinct placeholder characters, which says for every output column the
    input column it copies or the spacer base it holds."""
    n, width = reads.shape
    out_cols = LAYOUTS[oligo][0]("".join(chr(0x100 + k) for k in range(width)))[:width]
    out = np.empty((n, len(out_cols)), dtype=np.uint8)
    for j, ch in enumerate(out_cols):
        out[:, j] = reads[:, ord(ch) - 0x100] if ord(ch) >= 0x100 else ord(ch)
    return out
