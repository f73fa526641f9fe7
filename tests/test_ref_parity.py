"""Parity pinned by the REFERENCE itself (SURVEY.md 8c): oracle/_ref is /root/reference/src/ORBextractor.cc compiled
unmodified (plus ORBmatcher's DescriptorDistance / ComputeThreeMaxima) -- `make -C oracle ref`.  Three legs:

  * committed reference vectors (tests/golden/ref_*.npz, scripts/make_golden_ref.py) == the restated oracle,
    with no reference tree needed;
  * the reference's object code == the oracle on many more frames, where oracle/_ref is present (built here from
    /root/reference, shipped prebuilt to the GPU box);
  * GPU: the CUDA path == the reference vectors and == the reference's object code on BASELINE.json configs[0] and [1].
"""
import hashlib
import json
import os

import numpy as np
import pytest

from orb_slam3_b200.synth import synth_frame, shifted_frame

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIELDS = ("x", "y", "size", "angle", "response", "octave", "class_id")


def _load(name):
    return np.load(os.path.join(G, name), allow_pickle=False)


def _same(k, d, mono, rk, rd, rmono, ctx=""):
    assert len(k) == len(rk) and mono == rmono, (ctx, len(k), len(rk), mono, rmono)
    for f in FIELDS:
        assert np.array_equal(k[f], rk[f]), (ctx, f)
    assert np.array_equal(d, rd), ctx


@pytest.fixture(scope="module")
def ref():
    from oracle import ref as R
    if not R.available():
        pytest.skip("oracle/_ref is not built and /root/reference is absent")
    R.lib()
    return R


# ------------------------------------------------------------------ committed reference vectors vs the oracle
def test_oracle_equals_reference_vectors(oracle):
    z = _load("ref_extract_640x480.npz")
    k, d, mono = oracle.OracleExtractor(1000).extract(synth_frame(480, 640, 1))
    _same(k, d, mono, z["kps"], z["desc"], int(z["mono"]), "configs[0]")
    z = _load("ref_extract_lowtex.npz")
    k, d, mono = oracle.OracleExtractor(1000).extract(synth_frame(480, 640, 11, low_texture=True), lap=tuple(z["lap"]))
    _same(k, d, mono, z["kps"], z["desc"], int(z["mono"]), "low texture + lapping area")
    assert 0 < mono < len(k)
    z = _load("ref_extract_1280x720.npz")
    k, d, mono = oracle.OracleExtractor(2000).extract(synth_frame(720, 1280, 3))
    assert len(k) == int(z["n"]) and mono == int(z["mono"])
    assert hashlib.sha256(k.tobytes()).hexdigest() == str(z["sha_kps"])
    assert hashlib.sha256(d.tobytes()).hexdigest() == str(z["sha_desc"])


def test_oracle_match_helpers_equal_reference_vectors(oracle):
    z = _load("ref_match_helpers.npz")
    got = np.array([oracle.ham_distance(a, b) for a, b in zip(z["a"], z["b"])], np.int32)
    assert np.array_equal(got, z["dist"])
    assert (z["dist"][:16] == 0).all() and (z["dist"][16:32] == 256).all()   # SURVEY 8c known answers
    pop = np.unpackbits(z["a"] ^ z["b"], axis=1).sum(1)
    assert np.array_equal(pop, z["dist"])
    tm = np.array([oracle.three_maxima(h) for h in z["hist"]], np.int32)
    assert np.array_equal(tm, z["three"])
    # the product's host-side Hamming entry point (no GPU involved)
    from orb_slam3_b200 import _lib
    L = _lib.lib()
    got = np.array([L.ham_distance(_lib.ptr(np.ascontiguousarray(a)), _lib.ptr(np.ascontiguousarray(b)))
                    for a, b in zip(z["a"], z["b"])], np.int32)
    assert np.array_equal(got, z["dist"])


# ------------------------------------------------------------------ the reference's object code vs the oracle
def test_reference_tables(ref, oracle):
    for nf, nl in ((1000, 8), (2000, 8), (1250, 8)):
        r = ref.RefExtractor(nf, 1.2, nl).tables()
        o = oracle.OracleExtractor(nf, 1.2, nl)
        assert np.array_equal(r["umax"], o.umax())
        assert list(r["umax"]) == [15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3]  # SURVEY 8c
        pat = np.zeros(1024, np.int32)
        oracle.lib().orc_pattern(pat.ctypes.data_as(__import__("ctypes").c_void_p))
        assert np.array_equal(r["pattern"], pat)
        assert r["quota"].sum() == nf
        # the product's constructor tables (host side of the C ABI, no device needed)
        from orb_slam3_b200.extractor import ORBextractor
        e = ORBextractor(nf, 1.2, nl, 20, 7)
        assert np.array_equal(np.asarray(e.GetScaleFactors(), np.float32), r["scale"])
        assert np.array_equal(np.asarray(e.GetInverseScaleFactors(), np.float32), r["inv_scale"])
        assert np.array_equal(np.asarray(e.GetScaleSigmaSquares(), np.float32), r["sigma2"])
        assert np.array_equal(np.asarray(e.GetInverseScaleSigmaSquares(), np.float32), r["inv_sigma2"])
        assert np.array_equal(np.asarray(e.features_per_level(), np.int32), r["quota"])


CASES = [  # (h, w, nfeatures, seed, low_texture, lap)
    (480, 640, 1000, 1, False, (0, 0)), (480, 640, 1000, 2, False, (100, 300)), (480, 640, 1000, 11, True, (0, 0)),
    (480, 752, 1200, 3, False, (0, 0)),      # EuRoC geometry
    (376, 1241, 2000, 4, False, (0, 0)),     # KITTI geometry (nIni = 4 root nodes)
    (512, 512, 1500, 5, False, (0, 511)),    # TUM-VI geometry, everything inside the lapping area
    (720, 1280, 2000, 3, False, (0, 0)), (720, 1280, 2000, 6, True, (400, 900)),
    (480, 640, 5000, 7, False, (0, 0)),      # initialisation extractor (5 x nFeatures): quota rarely reached
    (240, 320, 300, 8, False, (0, 0)),
]


@pytest.mark.parametrize("h,w,nf,seed,low,lap", CASES)
def test_reference_object_code_equals_oracle(ref, oracle, h, w, nf, seed, low, lap):
    img = synth_frame(h, w, seed, low_texture=low)
    r, o = ref.RefExtractor(nf), oracle.OracleExtractor(nf)
    rk, rd, rm = r.extract(img, lap)
    ok, od, om = o.extract(img, lap)
    _same(ok, od, om, rk, rd, rm, (h, w, nf, seed))
    for l in range(8):
        assert np.array_equal(r.level_image(l), o.level_image(l)), l
    # the reference keeps its state between calls (mvImagePyramid is overwritten): a second frame on the same object
    img2 = shifted_frame(img, 3, -2, seed + 100)
    _same(*o.extract(img2, lap), *r.extract(img2, lap), "second frame")


def test_reference_pyramid_border_is_reflect101(ref):
    """ComputePyramid's 19-px frame (ORBextractor.cc:1185-1191): not read by the path (SURVEY A.2), checked so the
    stand-in's copyMakeBorder is known to behave like OpenCV's documented BORDER_REFLECT_101."""
    img = synth_frame(240, 320, 9)
    r = ref.RefExtractor(300)
    r.extract(img)
    for l in (0, 3):
        inner = r.level_image(l)
        assert np.array_equal(r.level_image(l, border=19), np.pad(inner, 19, mode="reflect"))


def test_reference_descriptor_distance_and_three_maxima(ref, oracle):
    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, (2000, 32), dtype=np.uint8)
    b = rng.integers(0, 256, (2000, 32), dtype=np.uint8)
    for x, y in zip(a, b):
        assert ref.descriptor_distance(x, y) == oracle.ham_distance(x, y)
    assert ref.descriptor_distance(np.zeros(32, np.uint8), np.full(32, 255, np.uint8)) == 256
    for _ in range(500):
        h = rng.integers(0, rng.integers(1, 50), 30).astype(np.int32)
        if rng.random() < 0.3:
            h[rng.random(30) < 0.8] = 0
        assert ref.three_maxima(h) == oracle.three_maxima(h)


def test_reference_empty_image_returns_minus_one(ref):
    """operator() on an empty image (ORBextractor.cc:1090-1091); the C ABI returns ORB_E_EMPTY for it."""
    import ctypes as C
    r = ref.RefExtractor(500)
    n = C.c_int(7)
    rc = ref.lib().ref_extract(r._h, None, 0, 0, 0, 0, 0, None, None, 0, C.byref(n))
    assert rc == -1


# ------------------------------------------------------------------ GPU: CUDA path vs the reference
@pytest.mark.gpu
def test_cuda_equals_reference_vectors():
    from orb_slam3_b200.extractor import ORBextractor
    z = _load("ref_extract_640x480.npz")
    mono, k, d = ORBextractor(1000, 1.2, 8, 20, 7)(synth_frame(480, 640, 1))
    _same(k, d, mono, z["kps"], z["desc"], int(z["mono"]), "configs[0]")
    z = _load("ref_extract_lowtex.npz")
    mono, k, d = ORBextractor(1000, 1.2, 8, 20, 7)(synth_frame(480, 640, 11, low_texture=True), None, tuple(int(v) for v in z["lap"]))
    _same(k, d, mono, z["kps"], z["desc"], int(z["mono"]), "low texture + lapping")
    z = _load("ref_extract_1280x720.npz")
    mono, k, d = ORBextractor(2000, 1.2, 8, 20, 7)(synth_frame(720, 1280, 3))
    assert len(k) == int(z["n"]) and mono == int(z["mono"])
    assert hashlib.sha256(np.ascontiguousarray(k).tobytes()).hexdigest() == str(z["sha_kps"])
    assert hashlib.sha256(np.ascontiguousarray(d).tobytes()).hexdigest() == str(z["sha_desc"])


def digest(*arrays):
    """sha256 over dtype, shape and bytes: what tests/golden/ref_gpu.json records of an output."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(repr((a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def recorded(key):
    """The reference's results for one GPU case, as committed by scripts/make_golden_ref_gpu.py."""
    with open(os.path.join(G, "ref_gpu.json")) as f:
        return json.load(f)["cases"][key]


def extract_key(h, w, nf, seed, low, lap):
    return "extract_%d_%d_%d_%d_%d_%d_%d" % (h, w, nf, seed, int(low), lap[0], lap[1])


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,nf,seed,low,lap", CASES)
def test_cuda_equals_reference_object_code(h, w, nf, seed, low, lap):
    """Against the reference's object code where oracle/_ref is present, else against its committed results."""
    from oracle import ref as R
    from orb_slam3_b200.extractor import ORBextractor
    img = synth_frame(h, w, seed, low_texture=low)
    e = ORBextractor(nf, 1.2, 8, 20, 7)
    mono, k, d = e(img, None, lap)
    if not R.available():
        z = recorded(extract_key(h, w, nf, seed, low, lap))
        assert (len(k), mono) == (z["n"], z["mono"])
        assert digest(k) == z["kps"] and digest(d) == z["desc"]
        assert [digest(e.image_pyramid(l)) for l in range(8)] == z["levels"]
        return
    R.lib()
    r = R.RefExtractor(nf)
    rk, rd, rm = r.extract(img, lap)
    _same(k, d, mono, rk, rd, rm, (h, w, nf, seed))
    for l in range(8):
        assert np.array_equal(e.image_pyramid(l), r.level_image(l)), l
