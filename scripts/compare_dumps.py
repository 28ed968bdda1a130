"""Compare two `bench.py --dump-outputs` directories file by file, bitwise.

    python scripts/compare_dumps.py DIR_A DIR_B

Every .npy of either directory must exist in both with the same shape and the same bits (np.array_equal on the raw
64-bit words, so NaNs and signed zeros count too).  Prints one line per file; exit status 1 if any file differs or is
missing.  Use it for changes that must not move a single bit of what a Newton step computes."""
import os
import sys

import numpy as np


def main(a, b):
    names = sorted({f for d in (a, b) for f in os.listdir(d) if f.endswith(".npy")})
    if not names:
        print(f"no .npy files in {a} or {b}")
        return 1
    bad = 0
    for name in names:
        pa, pb = os.path.join(a, name), os.path.join(b, name)
        if not (os.path.exists(pa) and os.path.exists(pb)):
            print(f"MISSING  {name}")
            bad += 1
            continue
        x, y = np.load(pa), np.load(pb)
        same = x.shape == y.shape and x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))
        if same:
            print(f"equal    {name}  {x.shape}")
        else:
            if x.shape == y.shape and x.dtype == y.dtype:
                words = lambda v: v.reshape(-1).view(np.uint8).reshape(v.size, -1)  # noqa: E731
                print(f"DIFFERS  {name}  {int((words(x) != words(y)).any(axis=1).sum())} of {x.size} entries")
            else:
                print(f"DIFFERS  {name}  {x.shape} {x.dtype} vs {y.shape} {y.dtype}")
            bad += 1
    print(f"{len(names) - bad} of {len(names)} files bitwise equal")
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
