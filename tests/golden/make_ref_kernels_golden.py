"""Freeze the outputs of the REFERENCE's own kernels that tests/test_oracle_ref.py and tests/test_gpu_envshade.py compare with into
tests/golden/ref_compiled_kernels.npz.  The kernels are the unmodified sources of the reference (kernel.cu, denoising.cu, the
renderutils kernels) compiled for the host by oracle.build_ref(), which needs the reference tree; every case is defined once, by the
`ref_*` functions of those test modules.  usage: python tests/golden/make_ref_kernels_golden.py"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def main():
    from common import FROZEN_REFERENCE, oracle
    from oracle import Reference
    import test_gpu_envshade
    import test_oracle_ref
    ref = Reference(oracle())
    cases = test_oracle_ref.reference_cases() + [("product-" + b, test_gpu_envshade.ref_product_case, (b,)) for b in ("pbr", "diffuse")]
    out = {}
    for name, fn, args in cases:
        for field, value in fn(ref, *args).items():
            out["%s|%s" % (name, field)] = np.asarray(value)
    np.savez_compressed(FROZEN_REFERENCE, **out)
    print("wrote %s: %d cases, %d arrays, %d bytes" % (FROZEN_REFERENCE, len(cases), len(out), os.path.getsize(FROZEN_REFERENCE)))


if __name__ == "__main__":
    main()
