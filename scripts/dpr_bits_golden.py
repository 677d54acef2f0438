"""Write tests/golden/dpr_bits.npz: the outputs of the runs of tests/dpr_bits_cases.py, on a B200.

    python scripts/dpr_bits_golden.py [--lib PATH_TO_LIBAGT_SO] [--out PATH]

--lib runs another build of libagt.so (the golden file of the sample loop's pair body was written by the build before it,
so that the test holds the new loop to the old one's bits).  Prints the card it ran on."""
import argparse
import subprocess
import sys

import numpy as np

sys.path.insert(0, ".")
from accurate_aprilgroup_tracking_b200 import _lib, synth  # noqa: E402
from tests import dpr_bits_cases  # noqa: E402


def context_on(path, mtx):
    """AgtContext bound to the library at `path` (the in-tree one when None)."""
    from accurate_aprilgroup_tracking_b200.context import AgtContext
    if path is None:
        return AgtContext(0, mtx, None)
    import ctypes as C
    lib = C.CDLL(path)
    for name, (res, args) in _lib.PROTOTYPES.items():
        if hasattr(lib, name):
            getattr(lib, name).restype = res
            getattr(lib, name).argtypes = args
    saved, _lib._lib = _lib._lib, lib
    try:
        return AgtContext(0, mtx, None)
    finally:
        _lib._lib = saved


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None)
    ap.add_argument("--out", default=str(dpr_bits_cases.GOLDEN))
    args = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True).stdout)
    ctxs = [context_on(args.lib, cam.mtx) for cam in (synth.CAMERA_1080P, synth.CAMERA_VGA)]
    for c in ctxs:
        c.set_synthetic_model()
    arrays = dpr_bits_cases.run_all(*ctxs)
    np.savez_compressed(args.out, **arrays)
    print(f"wrote {len(arrays)} arrays to {args.out}")
    for c in ctxs:
        c.close()


if __name__ == "__main__":
    main()
