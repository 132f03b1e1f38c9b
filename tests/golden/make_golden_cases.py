"""Writes the stored outputs of tests/test_oracle.py's seeded random cases and 1080p frame:

    python tests/golden/make_golden_cases.py

  reference_random_cases.json  per case: sha256 of the input and of the blur / mag / ang / nms / edges planes; per sigma: sha256 of
                               the Gaussian kernel
  reference_1080p.npz          sha256 of the input, the edge map bit-packed (np.packbits, row-major), its edge-pixel count

The outputs come from the compiled reference (oracle/_ref/libcanny_ref.so) when it is built, otherwise from the C restatement
(oracle/liboracle.so); "source" in both files says which.  The tests check the oracle against them on every checkout and the compiled
reference against them wherever it is built.
"""
import hashlib
import importlib.util
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
sys.path.insert(0, str(ROOT))
from oracle.bindings import Oracle, Ref  # noqa: E402

spec = importlib.util.spec_from_file_location("test_oracle", ROOT / "tests" / "test_oracle.py")
T = importlib.util.module_from_spec(spec)
spec.loader.exec_module(T)


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


if Ref.available():
    impl, source = Ref(), "compiled reference (oracle/_ref/libcanny_ref.so)"

    def planes(img, sigma, lo, hi):
        return T.reference_planes(impl, img, sigma, lo, hi)
else:
    impl, source = Oracle(), "C restatement (oracle/liboracle.so)"

    def planes(img, sigma, lo, hi):
        return impl.canny(img, sigma, lo, hi, steps=True)

cases, kernels = [], {}
for t, img, sigma, lo, hi in T.reference_random_cases():
    case = {"img": sha(img), "sigma": sigma, "lo": lo, "hi": hi}
    case.update({name: sha(p) for name, p in zip(T.PLANES, planes(img, sigma, lo, hi))})
    cases.append(case)
    kernels[str(sigma)] = sha(impl.gaussian_kernel(sigma)[0])
(HERE / "reference_random_cases.json").write_text(json.dumps({"source": source, "kernels": kernels, "cases": cases}, indent=0) + "\n")

img = T.frame_1080p()
edges = impl.canny(img, 1.4, 20, 60)
np.savez_compressed(HERE / "reference_1080p.npz", source=np.array(source), img_sha256=np.array(sha(img)),
                    edges_bits=np.packbits(edges == 255), edge_pixels=np.array(int((edges == 255).sum())))
print(source, len(cases), "cases;", int((edges == 255).sum()), "edge pixels at 1080p")
