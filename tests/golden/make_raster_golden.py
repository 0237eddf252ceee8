"""Generates tests/golden/raster_ref.json: SHA-256 digests of the inputs and of the outputs (face_index_map, weight_map,
depth_map, faces_inv) of the reference's own rasterizer kernels, oracle/_ref/libnmr_ref.so (built by oracle/build_ref.sh
from the reference tree), on every case of tests/test_raster_gpu.py's REF_CASES.  Needs an sm_100 GPU and that build.

  python tests/golden/make_raster_golden.py [OUT.json]       (default: tests/golden/raster_ref.json)
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

import torch  # noqa: E402

from oracle import raster  # noqa: E402
import test_raster_gpu as T  # noqa: E402


def main(out_path):
    if not raster.gpu_ref_available():
        raise SystemExit("oracle/_ref/libnmr_ref.so is missing: build it with oracle/build_ref.sh")
    dev = torch.device("cuda:0")
    out = {}
    for case, size in T.REF_CASES:
        faces = T.REF_FACES[case]().to(dev)
        fim, wim, depth, finv = raster.forward_face_index_map_gpu_ref(faces, size)
        torch.cuda.synchronize()
        out["%s@%d" % (case, size)] = dict(faces=T.digest(faces), covered=int((fim >= 0).sum()), fim=T.digest(fim),
                                           wim=T.digest(wim), depth=T.digest(depth), faces_inv=T.digest(finv))
        print(case, size, out["%s@%d" % (case, size)]["covered"])
    with open(out_path, "w") as fp:
        json.dump(out, fp, indent=1, sort_keys=True)
        fp.write("\n")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "raster_ref.json"))
