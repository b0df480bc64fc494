"""CPU: on-disk formats (a-tvsnet_b200/preprocess.py, SURVEY.md 8(f) N3) - camera text, PFM, pair.txt - round trips
and hand-written files; the bundled example cameras (example/*/N_cam.npy) survive write_cam -> load_cam."""
import importlib.util
import io
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location('atvs_preprocess', os.path.join(ROOT, 'a-tvsnet_b200', 'preprocess.py'))
P = importlib.util.module_from_spec(spec)
spec.loader.exec_module(P)

CAM_TXT = """extrinsic
1 0 0 0.5
0 1 0 -2
0 0 1 3.25
0 0 0 1

intrinsic
500.5 0 320
0 501.5 240
0 0 1

%s
"""


def test_load_cam_depth_field_variants():
    c = P.load_cam(io.StringIO(CAM_TXT % '425.0 2.5'), max_d=192)                 # 29 words: num = max_d
    assert c.shape == (2, 4, 4) and c[0, 0, 3] == 0.5 and c[0, 2, 3] == 3.25 and c[1, 1, 1] == 501.5
    assert list(c[1, 3]) == [425.0, 2.5, 192.0, 425.0 + 2.5 * 192]
    c = P.load_cam(io.StringIO(CAM_TXT % '425.0 2.5 64'), interval_scale=2)       # 30 words: end derived
    assert list(c[1, 3]) == [425.0, 5.0, 64.0, 425.0 + 5.0 * 64]
    c = P.load_cam(io.StringIO(CAM_TXT % '0.05 0.0033 128 0.4724'))               # 31 words
    assert list(c[1, 3]) == [0.05, 0.0033, 128.0, 0.4724]
    assert list(P.load_cam(io.StringIO(CAM_TXT % ''))[1, 3]) == [0, 0, 0, 0]
    assert np.all(c[1, :3, 3] == 0) and np.all(c[0, 3] == [0, 0, 0, 1])


def test_write_cam_round_trip(tmp_path):
    bundled = np.load(os.path.join(ROOT, 'tests', 'golden', 'example', '0', '2_cam.npy')).astype(np.float64)
    rng = np.random.default_rng(0)
    posed = np.zeros((2, 4, 4))         # random pose, all four depth fields set
    posed[0] = np.eye(4)
    posed[0, :3] = rng.standard_normal((3, 4))
    posed[1, :3, :3] = [[131.7, 0, 120], [0, 132.1, 80], [0, 0, 1]]
    posed[1, 3] = [0.05, 0.0033, 128, 0.4724]
    for cam in (bundled, posed):
        f = str(tmp_path / 'c_cam.txt')
        P.write_cam(f, cam)
        back = P.load_cam(f)
        assert np.array_equal(back[0], cam[0]) and np.array_equal(back[1, :3, :3], cam[1, :3, :3])
        assert np.array_equal(back[1, 3], cam[1, 3])
        s = P.scale_camera(cam, 0.25)
        assert s[1, 0, 0] == cam[1, 0, 0] * 0.25 and s[1, 1, 2] == cam[1, 1, 2] * 0.25 and s[1, 2, 2] == cam[1, 2, 2]
        assert np.array_equal(s[0], cam[0]) and s is not cam


def test_pfm_round_trip_and_layout(tmp_path):
    rng = np.random.default_rng(1)
    for shape in ((5, 7), (4, 6, 1), (3, 5, 3)):
        img = rng.standard_normal(shape).astype(np.float32)
        f = str(tmp_path / 'a.pfm')
        P.write_pfm(f, img)
        back = P.load_pfm(f)
        assert np.array_equal(back, img.reshape(back.shape))
    raw = open(f, 'rb').read()
    assert raw.startswith(b'PF\n5 3\n-1.000000\n')                                # colour, width height, little endian
    # rows are stored bottom-up: the first stored row is the LAST image row
    first_row = np.frombuffer(raw[len(b'PF\n5 3\n-1.000000\n'):][:5 * 3 * 4], '<f4').reshape(5, 3)
    assert np.array_equal(first_row, img[-1])
    # big-endian file written by hand
    g = np.arange(6, dtype='>f4').reshape(2, 3)
    open(f, 'wb').write(b'Pf\n3 2\n1.0\n' + g.tobytes())
    assert np.array_equal(P.load_pfm(f), np.float32([[3, 4, 5], [0, 1, 2]]))
    with pytest.raises(Exception):
        P.write_pfm(f, img.astype(np.float64))
    open(f, 'wb').write(b'P5\n3 2\n1.0\n')
    with pytest.raises(Exception):
        P.load_pfm(f)


def test_pair_txt(tmp_path):
    d = tmp_path / 'dense'
    d.mkdir()
    (d / 'pair.txt').write_text('2\n0\n3 1 0.9 2 0.8 5 0.1\n7\n1 0 0.5\n')
    lst = P.gen_pipeline_mvs_list(str(d), view_num=3)
    assert len(lst) == 2
    assert [os.path.basename(p) for p in lst[0]] == ['00000000.jpg', '00000000_cam.txt', '00000001.jpg', '00000001_cam.txt',
                                                      '00000002.jpg', '00000002_cam.txt']
    assert [os.path.basename(p) for p in lst[1]] == ['00000007.jpg', '00000007_cam.txt', '00000000.jpg', '00000000_cam.txt']
    assert lst[0][1].endswith(os.path.join('cams', '00000000_cam.txt'))


def test_center_image():
    rng = np.random.default_rng(2)
    img = (rng.uniform(0, 255, (20, 30, 3))).astype(np.uint8)
    c = P.center_image(img)
    assert c.dtype == np.float32 and np.allclose(c.mean(axis=(0, 1)), 0, atol=1e-5) and np.allclose(c.std(axis=(0, 1)), 1, atol=1e-4)


# ------------------------------------------------------------------ resize / crop / mask helpers (preprocess.py:39-100)
@pytest.fixture(scope='module')
def pgold():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_golden_preprocess.npz'))


def test_scale_image_equals_reference_cv2(pgold):
    """scale_image against the reference's own scale_image (= cv2.resize) run by tests/golden/make_golden_preprocess.py:
    bit-exact for 8-bit images (OpenCV's fixed-point bilinear) and for 'nearest', 1e-6 for float images."""
    from atvsnet_b200 import preprocess as P
    img8, dep = pgold['img8'], pgold['dep']
    for sc in (0.25, 0.5, 0.55, 0.8):
        assert np.array_equal(P.scale_image(img8, sc), pgold['lin8_%g' % sc]), sc
        assert np.array_equal(P.scale_image(img8, sc, 'nearest'), pgold['nn8_%g' % sc]), sc
        assert np.array_equal(P.scale_image(dep, sc, 'nearest'), pgold['nnf_%g' % sc]), sc
        got = P.scale_image(dep, sc)
        assert got.dtype == np.float32 and got.shape == pgold['linf_%g' % sc].shape
        assert np.abs(got - pgold['linf_%g' % sc]).max() <= 2e-6 * np.abs(dep).max(), sc
    assert P.scale_image(img8, 0.5, 'cubic') is None          # the reference falls through for other modes
    with pytest.raises(ValueError):
        P.scale_image(img8[:1, :1], 0.25)


def test_scale_image_live_cv2():
    """where OpenCV is importable: random even-sized images and odd scales, bit-exact (8-bit) / 2e-6 (float)."""
    cv2 = pytest.importorskip('cv2')
    from atvsnet_b200 import preprocess as P
    rng = np.random.default_rng(5)
    for shape in ((48, 64, 3), (270, 480, 3), (64, 48), (120, 90, 1)):
        img = rng.integers(0, 256, size=shape, dtype=np.uint8)
        f = rng.standard_normal(shape).astype(np.float32)
        for sc in (0.25, 0.5, 0.3, 0.4666666, 0.7, 0.9, 1.0):
            ref = cv2.resize(img, None, fx=sc, fy=sc, interpolation=cv2.INTER_LINEAR).reshape(P.scale_image(img, sc).shape)
            assert np.array_equal(P.scale_image(img, sc), ref), (shape, sc)
            ref = cv2.resize(f, None, fx=sc, fy=sc, interpolation=cv2.INTER_LINEAR).reshape(P.scale_image(f, sc).shape)
            assert np.abs(P.scale_image(f, sc) - ref).max() < 2e-6 * np.abs(f).max(), (shape, sc)


def test_scale_crop_mask_equal_reference(pgold):
    from atvsnet_b200 import preprocess as P
    imgs, cams, depth = list(pgold['mvs_imgs']), list(pgold['mvs_cams']), pgold['mvs_depth']
    si, sc, sd = P.scale_mvs_input([i.copy() for i in imgs], [c.copy() for c in cams], depth.copy(), scale=0.5)
    assert np.array_equal(np.stack(si), pgold['mvs_scaled_imgs'])
    assert np.array_equal(np.stack(sc), pgold['mvs_scaled_cams'])
    assert np.array_equal(sd, pgold['mvs_scaled_depth'])
    ci, cc, cd = P.crop_mvs_input([i.copy() for i in si], [c.copy() for c in sc], sd.copy(), base_image_size=32, max_h=64,
                                  max_w=96)
    assert np.array_equal(np.stack(ci), pgold['mvs_crop_imgs'])
    assert np.array_equal(np.stack(cc), pgold['mvs_crop_cams'])
    assert np.array_equal(cd, pgold['mvs_crop_depth'])
    assert np.array_equal(np.stack(P.scale_mvs_camera([c.copy() for c in cc], 0.25)), pgold['mvs_scaled_cams_quarter'])
    assert np.array_equal(P.mask_depth_image(pgold['dep'], 2.0, 8.0), pgold['mask_2_8'])
    two = P.scale_mvs_input([imgs[0].copy()], [cams[0].copy()], scale=0.5)
    assert len(two) == 2


def test_crop_to_32_python2_arithmetic():
    """BASELINE cfg3: a 1080 x 1920 frame is legal only after the crop to 1056 x 1920 (SURVEY.md F9).  The reference
    is Python 2: ``int(math.ceil(h / 32) * 32)`` floors first, so 1080 -> 1056 with 12 rows cut above and below, and
    sizes above (max_h, max_w) are centre-cropped to them; the principal point follows the crop."""
    from atvsnet_b200 import preprocess as P
    img = np.zeros((1080, 1920, 3), np.uint8)
    img[12:1068] = 7
    cam = np.zeros((2, 4, 4))
    cam[1, :3, :3] = [[1000.0, 0, 960.0], [0, 1000.0, 540.0], [0, 0, 1]]
    (out,), (c,) = P.crop_mvs_input([img], [cam.copy()], base_image_size=32, max_h=2000, max_w=2000)
    assert out.shape == (1056, 1920, 3) and (out == 7).all()
    assert c[1][1][2] == 540.0 - 12 and c[1][0][2] == 960.0
    (out,), (c,), d = P.crop_mvs_input([img], [cam.copy()], np.ones((1080, 1920)), base_image_size=32, max_h=480, max_w=896)
    assert out.shape == (480, 896, 3) and d.shape == (480, 896)
    assert c[1][1][2] == 540.0 - 300 and c[1][0][2] == 960.0 - 512
