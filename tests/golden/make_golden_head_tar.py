"""Golden fixture of head.tar's parameter layout: name and shape of every parameter of the UNMODIFIED reference's
Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128), in named_parameters() order.  That order indexes the per-parameter
Adam state of head.tar's 'optimizer' entry (audio_exp_nerf.py:487-489, :584-591).

Run where the reference tree is present (oracle/ref_import.py finds it, $IDEAL_NERF_REFERENCE first):

    python tests/golden/make_golden_head_tar.py [OUT_DIR]          # writes OUT_DIR/head_tar_layout.npz (default: tests/golden)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_import  # noqa: E402


def main(out_dir):
    head = ref_import.import_head(force_cpu=True)
    named = list(head.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128).named_parameters())
    shapes = np.zeros((len(named), 4), np.int64)             # (ndim, d0, d1, d2): every parameter here has at most 3 dims
    for i, (_, p) in enumerate(named):
        shapes[i, 0] = p.dim()
        shapes[i, 1:1 + p.dim()] = p.shape
    np.savez_compressed(os.path.join(out_dir, "head_tar_layout.npz"), names=np.array([n for n, _ in named]), shapes=shapes)
    print(f"head_tar_layout.npz: {len(named)} parameters from {ref_import.REF_ROOT}")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
