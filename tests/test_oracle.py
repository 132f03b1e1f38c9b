"""CPU tests that PIN the oracle (oracle/canny_oracle.c):
  1. every value-pinning vector of the reference's own tests/utils/test_utils.cpp;
  2. golden fixtures generated from the compiled, unmodified reference (tests/golden/make_golden.py);
  3. stored outputs on 400 seeded random cases and a 1080p frame (tests/golden/make_golden_cases.py), checked against the compiled
     reference itself wherever oracle/_ref/libcanny_ref.so is present.
"""
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

GOLD = Path(__file__).resolve().parent / "golden"
FLT_EPSILON = np.finfo(np.float32).eps
E = 255


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def impls(oracle, request):
    out = [oracle]
    from oracle.bindings import Ref
    if Ref.available():
        out.append(Ref())
    return out


@pytest.fixture(params=["oracle", "ref"])
def impl(request, oracle):
    if request.param == "oracle":
        return oracle
    from oracle.bindings import Ref
    if not Ref.available():
        pytest.skip("compiled reference not present")
    return Ref()


# ---- tests/utils/test_utils.cpp:7-45 -----------------------------------------------------------
def test_kernel_sum_one(impl):
    k, n = impl.gaussian_kernel(0.5)
    s = np.float32(0)
    for v in k:
        s = np.float32(s + v)
    assert abs(s - 1) < FLT_EPSILON


def test_kernel_values(impl):
    k, n = impl.gaussian_kernel(0.5)
    want = np.array([0.0002638651, 0.1064507720, 0.7865707259, 0.1064507720, 0.0002638651], np.float32)
    assert n == 5 and (np.abs(want - k) < FLT_EPSILON).all()


def test_kernel_creation(impl):
    k, n = impl.gaussian_kernel(2)
    assert n == 13
    for i in range(7):
        assert k[i] == k[12 - i]


# ---- :47-104 (sigma 0.5 on test.jpg) ------------------------------------------------------------
def test_gaussian_testjpg(impl, test_gray):
    out = impl.gaussian(test_gray, 0.5)
    assert out.shape == (256, 256)
    assert out.sum() != 0 and out.min() >= 0 and out.max() <= 255


# ---- :106-208 -------------------------------------------------------------------------------------
def test_gradient_vectors(impl):
    gx, gy = impl.xy_gradient(np.ones((3, 3), np.int16))
    assert gx.shape == (3, 3) and not gx.any() and not gy.any()
    img = np.array([1, 2, 1, 2, 3, 2, 3, 4, 3], np.int16).reshape(3, 3)
    gx, gy = impl.xy_gradient(img)
    assert gx.ravel().tolist() == [3, 0, -3, 4, 0, -4, 3, 0, -3]
    assert gy.ravel().tolist() == [3, 4, 3, 6, 8, 6, 3, 4, 3]


def test_sobel_dimensions(impl):
    m, a = impl.sobel(np.ones((3, 3), np.int16))
    assert m.shape == (3, 3) and a.shape == (3, 3)


# ---- :273-347 ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("grad,angle,expect", [
    ([0, 0, 0, 0, 10, 0, 50, 20, 50], [0] * 9, [0, 0, 0, 0, 10, 0, 50, 0, 50]),
    ([0, 1, 1, 0, 2, 0, 1, 1, 0], [0, 45, 45, 45, 45, 45, 45, 45, 0], [0, 1, 0, 0, 2, 0, 0, 1, 0]),
    ([1, 0, 0, 0, 1, 0, 0, 0, 1], [90] * 9, [1, 0, 0, 0, 1, 0, 0, 0, 1]),
    ([0, 1, 1, 0, 2, 0, 1, 1, 0], [135, 135, 0, 135, 135, 135, 0, 135, 135], [0, 1, 0, 0, 2, 0, 0, 1, 0]),
])
def test_nonmaximal_vectors(impl, grad, angle, expect):
    out = impl.nonmaximal(np.array(grad, np.int16).reshape(3, 3), np.array(angle, np.int16).reshape(3, 3))
    assert out.ravel().tolist() == expect


# ---- :349-397 ---------------------------------------------------------------------------------------
def test_find_edge_pixels_vector(impl):
    nms = np.array([5, 6, 0, 5, 5, 4, 1, 0, 1, 4, 1, 3, 7, 0, 0, 10, 9, 8, 0, 0, 0, 0, 0, 0, 0], np.int16).reshape(5, 5)
    want = [E, E, 0, 5, 5, E, 1, 0, 1, 4, 1, E, E, 0, 0, E, E, E, 0, 0, 0, 0, 0, 0, 0]
    out, _ = impl.find_edge_pixels(nms, np.zeros((5, 5), np.uint8), 1, 2, 10)
    assert out.ravel().tolist() == want


def test_hysteresis_vector(impl):
    nms = np.array([5, 6, 0, 5, 10, 4, 1, 0, 1, 4, 1, 3, 7, 0, 0, 10, 9, 8, 0, 0, 0, 0, 0, 0, 0], np.int16).reshape(5, 5)
    want = [E, E, 0, E, E, E, 0, 0, 0, E, 0, E, E, 0, 0, E, E, E, 0, 0, 0, 0, 0, 0, 0]
    assert impl.hysteresis(nms, 2, 10).ravel().tolist() == want


def test_angle_vector_commented_out_in_reference(oracle):
    # tests/utils/test_utils.cpp:253-271 (commented out there, still the documented binning):
    # gx = 1, gy = {0,-1,1,3,-3} -> {0,135,45,90,90}
    t = oracle.angle_table(3)
    assert [int(t[gy + 3, 1 + 3]) for gy in (0, -1, 1, 3, -3)] == [0, 135, 45, 90, 90]


def test_missing_link_quirk(impl):
    # src/utils.cpp:399: (1,0) does not propagate to (0,1); the reverse direction works
    a = np.array([[0, 30, 0], [100, 0, 0], [0, 0, 0]], np.int16)
    assert impl.hysteresis(a, 20, 60).ravel().tolist() == [0, 0, 0, E, 0, 0, 0, 0, 0]
    b = np.array([[0, 100, 0], [30, 0, 0], [0, 0, 0]], np.int16)
    assert impl.hysteresis(b, 20, 60).ravel().tolist() == [0, E, 0, E, 0, 0, 0, 0, 0]


# ---- golden fixtures from the compiled reference -----------------------------------------------------
def test_golden_testjpg(oracle, test_gray):
    man = json.loads((GOLD / "manifest.json").read_text())
    assert sha(test_gray) == man["test_gray_sha256"]
    n = 0
    for key, want in man.items():
        if not key.startswith("testjpg_"):
            continue
        _, s, lo, hi = key.split("_")
        blur, mag, ang, nms, edges = oracle.canny(test_gray, float(s[1:]), int(lo), int(hi), steps=True)
        assert sha(blur) == want["blur_sha256"] and sha(mag) == want["mag_sha256"] and sha(ang) == want["ang_sha256"]
        assert sha(nms) == want["nms_sha256"] and sha(edges) == want["edges_sha256"]
        assert int((edges == 255).sum()) == want["edge_pixels"]
        assert {str(a): int((ang == a).sum()) for a in (0, 45, 90, 135)} == want["angle_counts"]
        n += 1
    assert n == 4
    # BASELINE config 1: sigma 1.4, 20/60 on tests/test.jpg -> 3466 edge pixels (SURVEY 8c)
    assert man["testjpg_s1.4_20_60"]["edge_pixels"] == 3466


def test_golden_small_cases(oracle):
    z = np.load(GOLD / "golden_small_cases.npz")
    keys = sorted(k[:-4] for k in z.files if k.endswith("_img"))
    assert len(keys) == 66
    for k in keys:
        sigma = float(k.split("_s")[1])
        lo, hi = (int(v) for v in z[k + "_par"])
        blur, mag, ang, nms, edges = oracle.canny(z[k + "_img"], sigma, lo, hi, steps=True)
        assert (blur == z[k + "_blur"]).all() and (mag == z[k + "_mag"]).all() and (ang == z[k + "_ang"]).all(), k
        assert (nms == z[k + "_nms"]).all() and ((edges == 255) == (z[k + "_edges"] == 1)).all(), k


def test_golden_hysteresis_cases(oracle):
    z = np.load(GOLD / "golden_hysteresis_cases.npz")
    for i in range(200):
        assert ((oracle.hysteresis(z[f"h{i}_in"], 20, 60) == 255) == (z[f"h{i}_out"] == 1)).all(), i


# ---- seeded random cases and a 1080p frame: stored outputs, and the compiled reference where it is built ----------
# tests/golden/reference_random_cases.json and reference_1080p.npz hold, for every case, sha256 digests of the five planes (and
# the 1080p edge map bit-packed); tests/golden/make_golden_cases.py writes them.  Both tests compare the oracle with those stored
# outputs on every checkout and, where oracle/_ref/libcanny_ref.so is built, also check the stored outputs against the compiled
# reference itself.
PLANES = ("blur", "mag", "ang", "nms", "edges")


def reference_random_cases():
    """The 400 seeded cases: (t, img, sigma, lo, hi)."""
    rng = np.random.default_rng(1)
    for t in range(400):
        h, w = (int(v) for v in rng.integers(2, 48, 2))
        sigma = float(rng.choice([0.5, 0.8, 1.0, 1.4, 2.0, 3.0, 5.0]))
        kind = t % 3
        if kind == 0:
            img = rng.integers(0, 256, (h, w))
        elif kind == 1:
            img = rng.integers(100, 140, (h, w))
        else:
            img = (rng.random((h, w)) < 0.3) * 255
        img = img.astype(np.uint8)
        lo = int(rng.integers(0, 100))
        hi = int(rng.integers(lo + 1, 256))
        yield t, img, sigma, lo, hi


def reference_planes(ref, img, sigma, lo, hi):
    """The compiled reference's five planes, stage by stage, with its whole-pipeline edge map checked against the staged one."""
    blur = ref.gaussian(img, sigma)
    mag, ang = ref.sobel(blur)
    nms = ref.nonmaximal(mag, ang)
    edges = ref.canny(img, sigma, lo, hi)
    assert (ref.hysteresis(nms, lo, hi) == edges).all()
    return blur, mag, ang, nms, edges


def frame_1080p():
    import canny_edge_b200 as cb
    return cb.synth_host(1, 1080, 1920, kind=0, seed=1234)[0]


def test_oracle_equals_reference_random(oracle):
    from oracle.bindings import Ref
    ref = Ref() if Ref.available() else None
    gold = json.loads((GOLD / "reference_random_cases.json").read_text())
    assert len(gold["cases"]) == 400
    for t, img, sigma, lo, hi in reference_random_cases():
        want = gold["cases"][t]
        assert (sha(img), sigma, lo, hi) == (want["img"], want["sigma"], want["lo"], want["hi"]), f"case {t}: the seeded input changed"
        got = oracle.canny(img, sigma, lo, hi, steps=True)
        for name, plane in zip(PLANES, got):
            assert sha(plane) == want[name], f"case {t} {img.shape} sigma={sigma} {lo}/{hi}: {name} differs from the stored output"
        assert sha(oracle.gaussian_kernel(sigma)[0]) == gold["kernels"][str(sigma)]
        if ref is not None:
            for name, plane in zip(PLANES, reference_planes(ref, img, sigma, lo, hi)):
                assert sha(plane) == want[name], f"case {t}: the compiled reference's {name} differs from the stored output"
            assert sha(ref.gaussian_kernel(sigma)[0]) == gold["kernels"][str(sigma)]


def test_oracle_equals_reference_1080p(oracle):
    from oracle.bindings import Ref
    z = np.load(GOLD / "reference_1080p.npz")
    img = frame_1080p()
    assert sha(img) == str(z["img_sha256"]), "the seeded 1080p input changed"
    want = np.unpackbits(z["edges_bits"])[: img.size].reshape(img.shape).astype(np.int16) * 255
    assert int((want == 255).sum()) == int(z["edge_pixels"])
    got = oracle.canny(img, 1.4, 20, 60)
    assert (got == want).all(), f"{int((got != want).sum())} pixels differ from the stored edge map"
    if Ref.available():
        assert (Ref().canny(img, 1.4, 20, 60) == want).all(), "the compiled reference differs from the stored edge map"


def test_oracle_workload_generator_matches_product_generator():
    """bench.py's CPU legs build their frames with oracle_synth_rows (no product code loaded); the GPU arm with the library's
    generator.  Both must be the same bytes."""
    import canny_edge_b200 as cb
    from oracle.bindings import synth_frames
    for kind in (0, 1, 2):
        a = cb.synth_host(2, 70, 300, kind=kind, seed=1234, first_frame=5)
        b = synth_frames(2, 70, 300, kind=kind, seed=1234, first_frame=5, threads=2)
        assert (a == b).all(), kind
