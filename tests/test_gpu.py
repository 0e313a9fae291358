"""GPU parity suite (-m gpu): every stage and the whole path through the C ABI against the CPU oracle
(cv2 4.13 for the OpenCV pieces, numpy f64 for the filter) and against the committed golden vectors."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "oracle_seq.npz")


@pytest.fixture(scope="module")
def batch(cfg, lib_built):
    from larvio_b200 import api
    b = api.Batch(cfg, n_seq=2)
    yield b
    b.close()


@pytest.fixture(scope="module")
def clahe_imgs(seqs):
    import cv2
    cl = cv2.createCLAHE(3.0, (8, 8))
    return np.stack([cl.apply(seqs[s].images[j]) for s in range(2) for j in range(2)])   # s0f0 s0f1 s1f0 s1f1


def test_pyramid_bit_exact(batch, seqs):
    import cv2
    imgs = np.stack([seqs[0].images[0], seqs[1].images[0], seqs[0].images[3], seqs[1].images[5]])
    clahe, l1, l2, blur = batch.k_pyramid(imgs)
    cl = cv2.createCLAHE(3.0, (8, 8))
    for i in range(4):
        ref = cl.apply(imgs[i]); r1 = cv2.pyrDown(ref); r2 = cv2.pyrDown(r1)
        rb = cv2.GaussianBlur(ref, (7, 7), 2, sigmaY=2, borderType=cv2.BORDER_REFLECT_101)
        assert np.array_equal(ref, clahe[i]) and np.array_equal(r1, l1[i]) and np.array_equal(r2, l2[i])
        assert np.array_equal(rb, blur[i])


def test_pyramid_edge_images(batch):
    """constant, saturated and checkerboard inputs (CLAHE clip/redistribution corner cases)."""
    import cv2
    imgs = np.zeros((4, 480, 752), np.uint8)
    imgs[1] = 255
    imgs[2] = ((np.indices((480, 752)).sum(0) % 2) * 255).astype(np.uint8)
    imgs[3] = np.random.default_rng(0).integers(0, 256, (480, 752)).astype(np.uint8)
    clahe, l1, l2, blur = batch.k_pyramid(imgs)
    cl = cv2.createCLAHE(3.0, (8, 8))
    for i in range(4):
        ref = cl.apply(imgs[i])
        assert np.array_equal(ref, clahe[i]), i
        assert np.array_equal(cv2.pyrDown(cv2.pyrDown(ref)), l2[i]), i


def test_lk_matches_opencv(batch, clahe_imgs):
    import cv2
    A = clahe_imgs[[0, 2]]; B = clahe_imgs[[1, 3]]
    rng = np.random.default_rng(0)
    P = []
    for s in range(2):
        p = cv2.goodFeaturesToTrack(A[s], 200, 0.01, 20).reshape(-1, 2)
        extra = np.array([[0.3, 0.2], [751.0, 479.0], [5.5, 470.2], [745.1, 3.9], [-3.0, 100.0], [760.0, 200.0]], np.float32)
        p = np.concatenate([p, extra])[:206]
        while len(p) < 206:
            p = np.concatenate([p, rng.uniform(0, 470, (206 - len(p), 2)).astype(np.float32)])
        P.append(p)
    P = np.stack(P).astype(np.float32)
    init = P + rng.normal(0, 1.5, P.shape).astype(np.float32)
    out, st = batch.k_lk(A, B, P, init)
    crit = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 30, 0.01)
    for s in range(2):
        ref, rst, _ = cv2.calcOpticalFlowPyrLK(A[s], B[s], P[s].reshape(-1, 1, 2), init[s].reshape(-1, 1, 2).copy(), winSize=(21, 21),
                                               maxLevel=2, criteria=crit, flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
        ref = ref.reshape(-1, 2); rst = rst.reshape(-1)
        assert np.array_equal(rst, st[s])                              # status bit-exact
        ok = rst == 1
        # positions bit-exact: the kernel replays OpenCV's SSE accumulation order (oracle/lk_exact.py)
        assert np.array_equal(ref[ok], out[s][ok])


def test_orb_bit_exact(batch, clahe_imgs):
    import cv2
    from oracle.orb import OrbOracle
    img = clahe_imgs[0]
    rng = np.random.default_rng(1)
    pts = cv2.goodFeaturesToTrack(img, 196, 0.01, 20).reshape(-1, 2)
    pts = pts + rng.uniform(-0.5, 0.5, pts.shape).astype(np.float32)
    pts = np.concatenate([pts, np.array([[0.2, 0.3], [751, 479], [3.4, 476.5], [748.2, 2.2]], np.float32)])
    ang, desc = batch.k_orb(img[None], pts[None])
    o = OrbOracle(img)
    assert np.array_equal(o.angles(pts), ang[0])
    assert np.array_equal(o.compute(pts), desc[0])


def test_detector_identical_corners(batch, clahe_imgs):
    import cv2
    imgs = clahe_imgs[[1, 3]]
    det, eig = batch.k_detect(imgs, None, 200, return_eig=True)
    mask = np.full(imgs.shape, 255, np.uint8)
    for s in range(2):
        ref = cv2.goodFeaturesToTrack(imgs[s], 200, 0.01, 20).reshape(-1, 2)
        assert np.array_equal(ref, det[s])                            # same corners, same order
        re = cv2.cornerMinEigenVal(imgs[s], 3, ksize=3)
        # response map: OpenCV sums the 3x3 box in a running double; we sum 9 terms -> <=1 ulp on a few pixels
        assert (re != eig[s]).mean() < 1e-4 and np.abs(re - eig[s]).max() < 1e-7
        for p in ref[:120]:
            x, y = int(round(p[0])), int(round(p[1]))
            mask[s, max(y - 20, 0):min(y + 20, 479) + 1, max(x - 20, 0):min(x + 20, 751) + 1] = 0
    det = batch.k_detect(imgs, mask, [80, 57])
    for s, want in enumerate([80, 57]):
        ref = cv2.goodFeaturesToTrack(imgs[s], want, 0.01, 20, mask=mask[s]).reshape(-1, 2)
        assert np.array_equal(ref, det[s])
    empty = batch.k_detect(imgs, np.zeros(imgs.shape, np.uint8), 50)     # fully masked image
    assert all(len(e) == 0 for e in empty)


def test_undistort_bit_exact(batch, cfg):
    import cv2
    K = np.array([[cfg['intrinsics']['fx'], 0, cfg['intrinsics']['cx']], [0, cfg['intrinsics']['fy'], cfg['intrinsics']['cy']], [0, 0, 1.0]])
    D = np.array([cfg['distortion_coeffs'][k] for k in ('k1', 'k2', 'p1', 'p2')])
    p = np.random.default_rng(2).uniform([0, 0], [752, 480], (500, 2)).astype(np.float32)
    for to_px in (False, True):
        ref = cv2.undistortPoints(p.reshape(-1, 1, 2), K, D, R=np.eye(3), P=(K if to_px else np.eye(3))).reshape(-1, 2)
        assert np.array_equal(ref, batch.k_undistort(p, to_px))


def test_undistort_equidistant_matches_cv2_fisheye(lib_built):
    """SURVEY 8(f-3): distortion_model "equidistant" (config/mynteye.yaml) -> cv::fisheye::undistortPoints
    (image_processor.cpp:1063-1065).  Same Newton iteration, clamp and stop rule; double tan/sqrt of the device may differ
    from glibc in the last bit before the float cast, hence "nearly all identical, none off by more than a float ulp"."""
    import cv2
    from larvio_b200 import api
    from larvio_b200.config import Config
    D = dict(k1=-0.015661749636940888, k2=0.0028974710951617955, p1=0.0034539528765559204, p2=-0.006466223707507623)
    c = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), distortion_model="equidistant", distortion_coeffs=D)
    b = api.Batch(c, n_seq=1)
    K = np.array([[c['intrinsics']['fx'], 0, c['intrinsics']['cx']], [0, c['intrinsics']['fy'], c['intrinsics']['cy']], [0, 0, 1.0]])
    Dv = np.array([D[k] for k in ('k1', 'k2', 'p1', 'p2')])
    p = np.random.default_rng(2).uniform([0, 0], [752, 480], (2000, 2)).astype(np.float32)
    for to_px in (False, True):
        ref = cv2.fisheye.undistortPoints(p.reshape(-1, 1, 2), K, Dv, R=np.eye(3), P=(K if to_px else np.eye(3))).reshape(-1, 2)
        got = b.k_undistort(p, to_px)
        assert (ref == got).all(1).mean() > 0.995
        assert np.abs(ref - got).max() <= (1e-4 if to_px else 1e-6)
    b.close()


def test_ransac_masks_match_opencv(batch):
    import cv2
    rng = np.random.default_rng(5)
    K = np.array([[458.654, 0, 367.215], [0, 457.296, 248.375], [0, 0, 1]])
    P1, P2, REF = [], [], []
    for trial in range(150):
        n = int(rng.integers(15, 220)) if trial % 5 else int(rng.integers(1, 8))
        X = np.stack([rng.uniform(-4, 4, n), rng.uniform(-3, 3, n), rng.uniform(2, 9, n)], 1)
        R, _ = cv2.Rodrigues(rng.normal(0, 0.03, 3)); t = rng.normal(0, 0.08, 3)
        x1 = (K @ X.T).T; x1 = x1[:, :2] / x1[:, 2:]
        x2 = (K @ ((R @ X.T).T + t).T).T; x2 = x2[:, :2] / x2[:, 2:]
        x1 += rng.normal(0, 0.15, x1.shape); x2 += rng.normal(0, 0.15, x2.shape)
        oi = rng.choice(n, int(n * rng.uniform(0, 0.3)), replace=False)
        x2[oi] += rng.uniform(-15, 15, (len(oi), 2))
        p1, p2 = x1.astype(np.float32), x2.astype(np.float32)
        m = None
        if n >= 7:
            _, m = cv2.findFundamentalMat(p1, p2, cv2.FM_RANSAC, 1.0, 0.99)
        REF.append(np.ones(n, np.uint8) if m is None else m.reshape(-1))     # no mask => the reference keeps all
        P1.append(p1); P2.append(p2)
    masks = batch.k_ransac(P1, P2)
    bad = sum(not np.array_equal(a, b) for a, b in zip(REF, masks))
    assert bad == 0, bad          # same RNG stream, same acceptance rule, same candidate order as OpenCV


def _drive(cfg, seqs, nf, mode, S=2):
    """Run oracle and GPU side by side. mode: 'fe' (processImage only), 'be' (oracle messages -> GPU back end),
    'step' (fused)."""
    from larvio_b200 import api, harness
    from oracle.frontend import ImageProcessorOracle
    from oracle.backend import LarVioOracle
    b = api.Batch(cfg, n_seq=S)
    fes = [ImageProcessorOracle(cfg.raw) for _ in range(S)]
    bes = [LarVioOracle(cfg.raw) for _ in range(S)]
    feed = harness.ImuFeeder(seqs[:S], stride=256 if mode != 'fe' else 1024)     # 'fe' mode never erases consumed samples
    imu_o = [[] for _ in range(S)]; k = [0] * S
    inited = [False] * S
    rep = dict(msgs=0, id_mismatch=0, uv=0.0, vel=0.0, p=0.0, v=0.0, q=0.0, Prel=0.0, steps=0, ok_mismatch=0, imu_mismatch=0)
    from larvio_b200 import synth
    for j in range(nf):
        feed.push_until(j)
        msgs = []
        for s in range(S):
            k2 = synth.imu_window(seqs[s], k[s], seqs[s].img_t[j]); imu_o[s].extend(seqs[s].imu[k[s]:k2].tolist()); k[s] = k2
            msgs.append(fes[s].process_image(seqs[s].images[j], seqs[s].img_t[j], np.array(imu_o[s]).reshape(-1, 7)))
            if msgs[s] is not None and not inited[s]:
                a = (seqs[s].img_t[j], seqs[s].gt_q[j], seqs[s].gt_p[j], seqs[s].gt_v[j], np.zeros(3), np.zeros(3))
                bes[s].set_initial_state(*a); b.set_initial_state(s, *a); inited[s] = True
        imgs = np.stack([seqs[s].images[j] for s in range(S)]); t_img = np.array([seqs[s].img_t[j] for s in range(S)])
        ok = np.zeros(S, np.uint8)
        if mode == 'fe':
            feat, out_n, has = b.process_images(imgs, t_img, feed.buf, feed.n)
            for s in range(S):
                assert bool(has[s]) == (msgs[s] is not None)
                if msgs[s] is None:
                    continue
                rep['msgs'] += 1
                g = feat[s, :out_n[s]]
                if len(g) != len(msgs[s].ids) or not np.array_equal(g['id'], msgs[s].ids):
                    rep['id_mismatch'] += 1
                    continue
                if len(g) == 0:
                    continue                      # an empty message (every track lost): ids compared above, nothing else to compare
                uv = np.stack([g['u'], g['v'], g['u_init'], g['v_init']], 1); vel = np.stack([g['u_vel'], g['v_vel'], g['u_init_vel'], g['v_init_vel']], 1)
                rep['uv'] = max(rep['uv'], float(np.abs(uv - msgs[s].data[:, :4]).max())); rep['vel'] = max(rep['vel'], float(np.abs(vel - msgs[s].data[:, 4:]).max()))
            continue
        if mode == 'be':
            valid = np.array([m is not None for m in msgs], np.uint8)
            if valid.any():
                feat = np.zeros((S, b.cap), api.FEATURE_DTYPE); n_feat = np.zeros(S, np.int32); t_msg = np.zeros(S)
                for s, m in enumerate(msgs):
                    if m is None:
                        continue
                    n = len(m.ids); n_feat[s] = n; t_msg[s] = m.t; feat['id'][s, :n] = m.ids
                    for c, name in enumerate(['u', 'v', 'u_init', 'v_init', 'u_vel', 'v_vel', 'u_init_vel', 'v_init_vel']):
                        feat[name][s, :n] = m.data[:, c]
                ok = b.process_features(valid, t_msg, feat, n_feat, feed.buf, feed.n)
        else:
            ok = b.step(imgs, t_img, feed.buf, feed.n)
        for s in range(S):
            oko = bes[s].process_features(msgs[s], imu_o[s]) if msgs[s] is not None else False
            rep['ok_mismatch'] += bool(ok[s]) != bool(oko)
            rep['imu_mismatch'] += len(imu_o[s]) != int(feed.n[s])           # consumed samples erased like larvio.cpp:510-512
            if not oko:
                continue
            rep['steps'] += 1
            st = b.get_state(s); o = bes[s].imu_state
            rep['p'] = max(rep['p'], float(np.abs(st['p'] - o.p).max())); rep['v'] = max(rep['v'], float(np.abs(st['v'] - o.v).max()))
            gt = np.asarray(seqs[s].gt_p[j], np.float64)                      # trajectory error of both arms against the truth
            rep.setdefault('se_gpu', []).append(float(np.sum((st['p'] - gt) ** 2))); rep.setdefault('se_cpu', []).append(float(np.sum((o.p - gt) ** 2)))
            rep['q'] = max(rep['q'], float(min(np.abs(st['q'] - o.q).max(), np.abs(st['q'] + o.q).max())))
            P = b.get_covariance(s)
            assert P.shape == bes[s].P.shape
            rep['max_dim'] = max(rep.get('max_dim', 0), int(P.shape[0]))
            rep['max_slam'] = max(rep.get('max_slam', 0), len(getattr(bes[s], 'feature_states', [])))
            rep['anchor_changes'] = rep.get('anchor_changes', 0) + int(bes[s].stats.get('anchor_changes', 0) or 0)
            assert np.abs(P - P.T).max() == 0.0                               # symmetric by construction
            rep['Prel'] = max(rep['Prel'], float(np.linalg.norm(P - bes[s].P) / np.linalg.norm(bes[s].P)))
            cal = b.get_calibration(s)
            rep['calib'] = max(rep.get('calib', 0.0), float(max(np.abs(cal['Tg'] - bes[s].Tg).max(), np.abs(cal['As'] - bes[s].As).max(),
                               np.abs(cal['Ma'] - bes[s].Ma).max(), np.abs(cal['R_imu_cam0'] - o.R_imu_cam0).max(),
                               np.abs(cal['t_cam0_imu'] - o.t_cam0_imu).max(), abs(cal['td'] - bes[s].td))))
    b.close()
    if rep.get('se_gpu'):
        rep['rmse_gpu'] = float(np.sqrt(np.mean(rep['se_gpu']))); rep['rmse_cpu'] = float(np.sqrt(np.mean(rep['se_cpu'])))
    return rep


def test_ransac_tie_case_from_golden(batch):
    d = np.load(os.path.join(ROOT, "tests", "golden", "ransac_tie_case.npz"))
    got = batch.k_ransac([d["p1"].astype(np.float32)], [d["p2"].astype(np.float32)])[0]
    assert np.array_equal(got.astype(bool), d["cv"].reshape(-1).astype(bool))


def test_frontend_ids_bit_exact_short_sequences(cfg, seqs):
    rep = _drive(cfg, seqs, 14, 'fe')
    assert rep['msgs'] >= 10
    assert rep['id_mismatch'] == 0                    # feature ids and their order: bit-exact
    assert rep['uv'] == 0.0 and rep['vel'] == 0.0     # every stage bit-exact => identical messages


def test_backend_matches_oracle(cfg, seqs):
    rep = _drive(cfg, seqs, 14, 'be')
    assert rep['steps'] >= 10 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    # identical feature messages in: FP64 filter agrees to rounding (stated tolerance: 1e-9 relative per step)
    assert rep['p'] < 1e-9 and rep['v'] < 1e-9 and rep['q'] < 1e-9 and rep['Prel'] < 1e-9


def test_fused_step_tracks_oracle(cfg, seqs):
    rep = _drive(cfg, seqs, 14, 'step')
    assert rep['steps'] >= 10 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    # GPU front end (bit-exact messages) feeds the GPU filter
    assert rep['p'] < 1e-9 and rep['q'] < 1e-9 and rep['Prel'] < 1e-9


def test_zupt_static_start_matches_oracle(cfg):
    """checkZUPT / measurementUpdate_ZUPT_vpq (larvio.cpp:2751-2962): one second of standstill, then motion."""
    from larvio_b200 import synth
    zs = [synth.make_sequence(cfg.raw, 5 + s, 34, static_until=1.0) for s in range(2)]
    rep = _drive(cfg, zs, 34, 'step')
    assert rep['steps'] >= 14 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['p'] < 1e-9 and rep['v'] < 1e-9 and rep['q'] < 1e-9 and rep['Prel'] < 1e-9


def test_trajectory_rmse_within_one_percent_of_the_cpu_path(cfg):
    """north_star acceptance: per-sequence trajectory RMSE within 1 % of the CPU reference path on EuRoC-shaped synthetic
    inputs.  80 frames (4 s) of the fused GPU path and of the oracle, both started from the truth, both scored against
    the generator's ground truth."""
    from larvio_b200 import synth
    seqs80 = [synth.make_sequence(cfg.raw, s, 80) for s in range(2)]
    rep = _drive(cfg, seqs80, 80, 'step')
    assert rep['steps'] >= 70 and rep['ok_mismatch'] == 0
    assert rep['rmse_cpu'] > 1e-4                                  # a real, non-zero drift to compare
    assert abs(rep['rmse_gpu'] / rep['rmse_cpu'] - 1.0) < 0.01
    assert rep['p'] < 1e-8


def test_hybrid_slam_features_match_oracle(lib_built):
    """euroc defaults: hybrid MSCKF + 1-D inverse-depth EKF-SLAM features (one per cell of a 5x6 grid).  SLAM features
    enter the state 5 s after the start (larvio.cpp:1974), so the run is 130 frames long."""
    from larvio_b200 import synth
    from larvio_b200.config import Config
    hc = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), sw_size=16)
    hs = [synth.make_sequence(hc.raw, s, 130) for s in range(2)]
    rep = _drive(hc, hs, 130, 'step')
    assert rep['steps'] >= 60 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8


def test_hybrid_3d_inverse_depth_slam_features_match_oracle(lib_built):
    """feature_idp_dim: 3 - SLAM features carry (x/z, y/z, 1/z) in their anchor camera (3 state columns each): the anchor's
    own observation takes part in featureJacobian_ekf_new (larvio.cpp:1260-1262), three reflections split a new feature's
    block, H_2 is a 3x3 triangle (:1661-1676, :1821-1854), and when the anchor pose leaves the window the newest state
    becomes the anchor with updateFeatureCov_3didp (:2965-3122, including its old_state_id slip)."""
    from larvio_b200 import synth
    from larvio_b200.config import Config
    hc = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), sw_size=16, feature_idp_dim=3)
    hs = [synth.make_sequence(hc.raw, s, 130) for s in range(2)]
    rep = _drive(hc, hs, 130, 'step')
    assert rep['steps'] >= 60 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['max_slam'] >= 8 and rep['max_dim'] >= 22 + 6 * 15 + 3 * 8 and rep['anchor_changes'] >= 10
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8


def test_hybrid_3d_inverse_depth_with_online_calibration(lib_built):
    """configs[3]'s switches with the other parameterisation: 3-D inverse depth + estimate_extrin/td + IMU-intrinsic calibration
    (LEG_DIM 46: the feature blocks start behind 46 + 6N columns)."""
    from larvio_b200 import synth
    from larvio_b200.config import Config
    cc = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), sw_size=16, calib_imu_instrinsic=1, feature_idp_dim=3)
    cs = [synth.make_sequence(cc.raw, s, 124) for s in range(2)]
    rep = _drive(cc, cs, 124, 'step')
    assert rep['steps'] >= 58 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0 and rep['max_slam'] >= 5
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8 and rep['calib'] < 1e-9


def test_imu_intrinsic_calibration_matches_oracle(lib_built):
    """calib_imu_instrinsic: 1 -> LEG_DIM 46 (larvio.cpp:158-161): the 24 Tg/As/Ma states are propagated (calPhi
    :3532-3797) and corrected (:1497-1507) exactly like the oracle's, in pure-MSCKF mode."""
    from larvio_b200 import synth
    from larvio_b200.config import Config
    cc = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), sw_size=16, max_features_in_one_grid=0, calib_imu_instrinsic=1)
    cs = [synth.make_sequence(cc.raw, s, 70) for s in range(2)]
    rep = _drive(cc, cs, 70, 'step')
    assert rep['steps'] >= 40 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8 and rep['calib'] < 1e-9


def test_config_d_hybrid_with_online_calibration(lib_built):
    """BASELINE configs[3] per sequence: 1-D IDP hybrid + estimate_extrin/td + IMU-intrinsic calibration."""
    from larvio_b200 import synth
    from larvio_b200.config import Config
    cc = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), sw_size=16, calib_imu_instrinsic=1)
    cs = [synth.make_sequence(cc.raw, s, 124) for s in range(2)]
    rep = _drive(cc, cs, 124, 'step')
    assert rep['steps'] >= 58 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8 and rep['calib'] < 1e-9


def test_config_e_capacity_400_tracks_50_pose_window(lib_built):
    """BASELINE configs[4] per sequence: 400 tracks, 50-pose window, 4x5 SLAM grid (20 features).  46 frames fill 23 window
    slots; the run checks the capacities (feature table, raw/stacked Jacobian rows, d up to 22 + 6*51 + 20) and parity."""
    from larvio_b200 import synth
    from larvio_b200.config import Config
    ec = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_num=400, sw_size=50, aug_grid_rows=4, aug_grid_cols=5,
                     min_distance=14)
    es = [synth.make_sequence(ec.raw, s, 46) for s in range(2)]
    rep = _drive(ec, es, 46, 'step')
    assert rep['steps'] >= 40 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8


def test_self_start_with_the_static_initialiser(lib_built):
    """SURVEY 8(f-1): no injected state.  The sequence stands still for 1.4 s; the host-side inclinometer initialiser
    (lvb_static_init_*) watches the feature messages of lvb_process_images, starts the filter through
    lvb_set_initial_state, erases the consumed IMU samples, and lvb_process_features takes over (larvio.cpp:375-391).
    The oracle does the same with its own restatement of StaticInitializer.cpp."""
    from larvio_b200 import api, synth
    from larvio_b200.config import Config
    from oracle.frontend import ImageProcessorOracle
    from oracle.backend import LarVioOracle
    from oracle.initializer import StaticInitializerOracle
    c = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_in_one_grid=0, sw_size=16)
    NF = 56
    seq = synth.make_sequence(c.raw, 3, NF, static_until=1.4)
    b = api.Batch(c, n_seq=1)
    host_init = api.StaticInitializer(c); orc_init = StaticInitializerOracle(c.raw)
    fe = ImageProcessorOracle(c.raw); be = LarVioOracle(c.raw)
    imu_o = []; k = 0
    buf = np.zeros((1, 512), api.IMU_DTYPE); n_buf = np.zeros(1, np.int32)
    started = False; steps = 0; worst = 0.0
    for j in range(NF):
        k2 = synth.imu_window(seq, k, seq.img_t[j])
        new = seq.imu[k:k2]; k = k2
        imu_o.extend(new.tolist())
        m = len(new); n0 = int(n_buf[0])
        buf["t"][0, n0:n0 + m] = new[:, 0]; buf["gyro"][0, n0:n0 + m] = new[:, 1:4]; buf["acc"][0, n0:n0 + m] = new[:, 4:7]; n_buf[0] = n0 + m
        msg = fe.process_image(seq.images[j], seq.img_t[j], np.array(imu_o).reshape(-1, 7))
        feat, out_n, has = b.process_images(seq.images[j][None], np.array([seq.img_t[j]]), buf, n_buf)
        assert bool(has[0]) == (msg is not None)
        if msg is None:
            continue
        assert np.array_equal(feat[0, :out_n[0]]['id'], msg.ids)
        if not started:
            a = host_init.try_init(feat[0, :out_n[0]], seq.img_t[j], buf[0, :n_buf[0]])
            o = orc_init.try_inc_init(msg.ids, msg.data[:, :2], msg.t, np.array(imu_o).reshape(-1, 7))
            assert (a is None) == (o is None)
            if a is None:
                continue
            assert a["n_consumed"] == o["n_consumed"] and np.abs(a["q"] - o["q"]).max() < 1e-12
            b.set_initial_state(0, a["t"], a["q"], a["p"], a["v"], a["bg"], a["ba"])
            be.set_initial_state(o["t"], o["q"], o["p"], o["v"], o["bg"], o["ba"])
            nc = a["n_consumed"]                                          # StaticInitializer.cpp:149-150
            buf[0, :n_buf[0] - nc] = buf[0, nc:n_buf[0]].copy(); n_buf[0] -= nc
            del imu_o[:nc]
            started = True
        ok = b.process_features(has, np.array([seq.img_t[j]]), feat, out_n, buf, n_buf)
        oko = be.process_features(msg, imu_o)
        assert bool(ok[0]) == bool(oko) and int(n_buf[0]) == len(imu_o)
        if oko:
            st = b.get_state(0)
            worst = max(worst, float(np.abs(st['p'] - be.imu_state.p).max()), float(np.abs(st['v'] - be.imu_state.v).max()))
            P = b.get_covariance(0)
            assert P.shape == be.P.shape and np.linalg.norm(P - be.P) / np.linalg.norm(be.P) < 1e-8
            steps += 1
    assert started and steps >= 12 and worst < 1e-8
    # the filter started from gravity alone stays near the truth (the truth frame differs by the unobservable yaw only)
    assert abs(np.linalg.norm(be.imu_state.p) - np.linalg.norm(seq.gt_p[NF - 1] - seq.gt_p[0])) < 0.3
    b.close(); host_init.close()


def _blackout_sequences(cfg):
    """Sequence A loses every track for four frames mid-run (uniform grey images: LK's min-eigenvalue test fails for all
    points and the detector finds no corner), then has to repopulate from nothing; sequence B gets a grey SECOND image, so
    initializeFirstFeatures fails and the state machine falls back to FIRST_IMAGE (image_processor.cpp:160-172)."""
    import copy
    from larvio_b200 import synth
    a = synth.make_sequence(cfg.raw, 0, 44); b = synth.make_sequence(cfg.raw, 1, 44)
    a = copy.copy(a); b = copy.copy(b)
    a.images = a.images.copy(); b.images = b.images.copy()
    a.images[20:24] = 117
    b.images[1] = 117
    return [a, b]


def test_frontend_survives_blackout_and_failed_second_image(cfg):
    seqs2 = _blackout_sequences(cfg)
    rep = _drive(cfg, seqs2, 44, 'fe')
    assert rep['msgs'] >= 36 and rep['id_mismatch'] == 0       # ids and their order: bit-exact, before, during and after
    assert rep['uv'] < 1e-6 and rep['vel'] < 1e-4


def test_filter_runs_through_empty_feature_messages(cfg):
    """Same inputs through the fused path: during the blackout the published messages carry no feature at all, the filter
    keeps propagating and augmenting on IMU alone (larvio.cpp:394-461 with an empty message), then re-acquires."""
    seqs2 = _blackout_sequences(cfg)
    rep = _drive(cfg, seqs2, 44, 'step')
    assert rep['steps'] >= 36 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8


def _python_two_call_replay(c, mav_dir):
    """The replay driver's loop (larvio_b200/host/replay_main.cpp) through the Python mirror of the same C-ABI calls:
    returns the rows it would log (time since take-off, q w x y z, v, p, bg, ba)."""
    from larvio_b200 import api, euroc
    b = api.Batch(c, n_seq=1); init = api.StaticInitializer(c)
    buf = np.zeros((1, 4096), api.IMU_DTYPE); n_buf = np.zeros(1, np.int32)
    started = False; take_off = 0.0; ref = []
    for t, img, rows in euroc.Replay(mav_dir):
        m = len(rows); n0 = int(n_buf[0])
        buf["t"][0, n0:n0 + m] = rows[:, 0]; buf["gyro"][0, n0:n0 + m] = rows[:, 1:4]; buf["acc"][0, n0:n0 + m] = rows[:, 4:7]; n_buf[0] = n0 + m
        feat, out_n, has = b.process_images(img[None], np.array([t]), buf, n_buf)
        if not has[0]:
            continue
        if not started:
            a = init.try_init(feat[0, :out_n[0]], t, buf[0, :n_buf[0]])
            if a is None:
                continue
            b.set_initial_state(0, a["t"], a["q"], a["p"], a["v"], a["bg"], a["ba"])
            nc = a["n_consumed"]; buf[0, :n_buf[0] - nc] = buf[0, nc:n_buf[0]].copy(); n_buf[0] -= nc
            started = True; take_off = a["t"]
        ok = b.process_features(has, np.array([t]), feat, out_n, buf, n_buf)
        if ok[0]:
            st = b.get_state(0)
            ref.append(np.concatenate([[st["t"] - take_off, st["q"][3]], st["q"][:3], st["v"], st["p"], st["bg"], st["ba"]]))
    b.close(); init.close()
    return np.array(ref)


def _write_mav(tmp_path, seq):
    """A synthetic sequence as an EuRoC ASL directory (PNG + csv, ns stamps)."""
    import cv2
    mav = tmp_path / "mav0"
    (mav / "cam0" / "data").mkdir(parents=True); (mav / "imu0").mkdir(parents=True)
    with open(mav / "cam0" / "data.csv", "w") as f:
        f.write("#timestamp [ns],filename\n")
        for t, im in zip(seq.img_t, seq.images):
            ns = int(round(t * 1e9)); cv2.imwrite(str(mav / "cam0" / "data" / ("%d.png" % ns)), im); f.write("%d,%d.png\r\n" % (ns, ns))
    with open(mav / "imu0" / "data.csv", "w") as f:
        f.write("#timestamp [ns],w_x,w_y,w_z,a_x,a_y,a_z\n")
        for r in seq.imu:
            f.write("%d,%.17g,%.17g,%.17g,%.17g,%.17g,%.17g\r\n" % (int(round(r[0] * 1e9)), *r[1:]))
    return mav


def test_shim_facade_linked_and_run_matches_the_oracle(tmp_path, lib_built):
    """SURVEY 8(b): larvio_shim.hpp (the reference's ImageProcessor / LarVio classes over the C ABI) compiled, LINKED and RUN
    as the reference's own main loop (larvio_b200/bin/larvio_shim_demo <- host/shim_main.cpp, app/larvioMain.cpp:87-117) on an
    on-disk sequence; euroc.yaml defaults (hybrid, 5x6 SLAM grid), self-start from a standstill.  Every odometry line and
    every map-point list (getStableMapPointPositions / getActiveeMapPointPositions, larvio.h:86-87) is compared with the
    CPU oracle driven by the same files."""
    import subprocess
    from larvio_b200 import synth, euroc
    from larvio_b200.config import Config
    from oracle.frontend import ImageProcessorOracle
    from oracle.backend import LarVioOracle
    from oracle.initializer import StaticInitializerOracle
    cfg_path = os.path.join(ROOT, "configs", "euroc_mono.yaml")
    c = Config.load(cfg_path)
    NF = 150
    seq = synth.make_sequence(c.raw, 3, NF, static_until=1.4)
    mav = _write_mav(tmp_path, seq)
    exe = os.path.join(ROOT, "larvio_b200", "bin", "larvio_shim_demo")
    r = subprocess.run([exe, cfg_path, str(mav)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    odo = [np.array(l.split()[1:], float) for l in r.stdout.splitlines() if l.startswith("ODO ")]
    pts = [l.split() for l in r.stdout.splitlines() if l.startswith("PTS ")]
    # the oracle over the same files
    fe = ImageProcessorOracle(c.raw); be = LarVioOracle(c.raw); init = StaticInitializerOracle(c.raw)
    imu = []; started = False; ref = []; ref_pts = []
    for t, img, rows in euroc.Replay(str(mav)):
        imu.extend(rows.tolist())
        msg = fe.process_image(img, t, np.array(imu).reshape(-1, 7))
        if msg is None:
            continue
        if not started:
            o = init.try_inc_init(msg.ids, msg.data[:, :2], msg.t, np.array(imu).reshape(-1, 7))
            if o is None:
                continue
            be.set_initial_state(o["t"], o["q"], o["p"], o["v"], o["bg"], o["ba"])
            del imu[:o["n_consumed"]]
            started = True
        if be.process_features(msg, imu):
            st = be.imu_state
            ref.append(np.concatenate([[t], st.q, st.p, st.v]))
            if len(ref) % 10 == 0:
                for tag, m in (("S", be.get_stable_map_points()), ("A", be.get_active_map_points())):
                    if m:
                        ref_pts.append((tag, m))
    assert len(odo) == len(ref) >= 60
    odo = np.array(odo); ref = np.array(ref)
    assert np.abs(odo[:, 0] - ref[:, 0]).max() < 1e-9
    qd = np.minimum(np.abs(odo[:, 1:5] - ref[:, 1:5]).max(1), np.abs(odo[:, 1:5] + ref[:, 1:5]).max(1))
    assert qd.max() < 1e-8 and np.abs(odo[:, 5:] - ref[:, 5:]).max() < 1e-8
    assert len(pts) == len(ref_pts) >= 2 and any(p[1] == "S" for p in pts) and any(p[1] == "A" for p in pts)
    for got, (tag, m) in zip(pts, ref_pts):
        assert got[1] == tag and int(got[2]) == len(m)
        ids = [int(x) for x in got[3::4]]
        assert ids == sorted(m.keys())                                     # std::map order
        xyz = np.array(got[3:], float).reshape(-1, 4)[:, 1:]
        assert np.abs(xyz - np.array([m[k] for k in ids])).max() < 1e-7


def test_cpp_replay_driver_matches_the_python_two_call_path(tmp_path, lib_built):
    """larvio_b200/bin/larvio_replay on a synthetic EuRoC-layout directory (PNG + csv on disk, self-start from a
    standstill) must write the trajectory the Python mirror of the same calls produces."""
    import subprocess
    import cv2
    from larvio_b200 import api, synth, euroc
    from larvio_b200.config import Config
    cfg_path = os.path.join(ROOT, "configs", "euroc_mono.yaml")
    c = Config.load(cfg_path)
    NF = 40
    seq = synth.make_sequence(c.raw, 3, NF, static_until=1.4)
    mav = _write_mav(tmp_path, seq)
    exe = os.path.join(ROOT, "larvio_b200", "bin", "larvio_replay")
    r = subprocess.run([exe, cfg_path, str(tmp_path / "out"), str(mav)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = euroc.read_state_log(str(tmp_path / "out" / "seq0" / "msckf_2_state.txt"))
    ref = _python_two_call_replay(c, str(mav))
    assert got.shape[0] == ref.shape[0] >= 6
    assert np.allclose(got[:, :17], ref, rtol=2e-5, atol=2e-6)          # the log has 6 significant digits


def test_gpu_against_committed_golden(cfg, seqs):
    from larvio_b200 import api, harness
    g = np.load(GOLD)
    b = api.Batch(cfg, n_seq=2)
    feed = harness.ImuFeeder(seqs, stride=256)
    inited = [False, False]
    checked = 0
    for j in range(14):
        feed.push_until(j)
        imgs = np.stack([seqs[s].images[j] for s in range(2)]); t_img = np.array([seqs[s].img_t[j] for s in range(2)])
        feat, out_n, has = b.process_images(imgs, t_img, feed.buf, feed.n)
        for s in range(2):
            key = "ids_%d_%d" % (s, j)
            assert bool(has[s]) == (key in g.files)
            if has[s]:
                assert np.array_equal(feat[s, :out_n[s]]['id'], g[key])
                if not inited[s]:
                    b.set_initial_state(s, seqs[s].img_t[j], seqs[s].gt_q[j], seqs[s].gt_p[j], seqs[s].gt_v[j], np.zeros(3), np.zeros(3)); inited[s] = True
        if has.any():
            t_msg = np.where(has, t_img, 0.0)
            ok = b.process_features(has, t_msg, feat, out_n, feed.buf, feed.n)
            for s in range(2):
                key = "state_%d_%d" % (s, j)
                assert bool(ok[s]) == (key in g.files)
                if ok[s]:
                    st = b.get_state(s)
                    got = np.concatenate([st['q'], st['p'], st['v'], st['bg'], st['ba']])
                    assert np.abs(got - g[key]).max() < 1e-9
                    P = b.get_covariance(s)
                    assert P.shape[0] == int(g["Pfro_%d_%d" % (s, j)][1])
                    assert abs(np.linalg.norm(P) / g["Pfro_%d_%d" % (s, j)][0] - 1) < 1e-9
                    assert np.allclose(np.diag(P), g["Pdiag_%d_%d" % (s, j)], rtol=1e-8, atol=1e-14)
                    checked += 1
    b.close()
    assert checked >= 10


def test_batch_invariance_and_properties_at_full_batch(cfg, seqs):
    """Size-independent properties at BASELINE's batch size: 64 sequences (the same two inputs replicated)
    must give bit-identical results per replica; P stays symmetric PSD; quaternions stay unit."""
    from larvio_b200 import api, harness
    S = 64
    rep_seqs = [seqs[s % 2] for s in range(S)]
    b = api.Batch(cfg, n_seq=S)
    feed = harness.ImuFeeder(rep_seqs)
    for s in range(S):
        b.set_initial_state(s, rep_seqs[s].img_t[0], rep_seqs[s].gt_q[0], rep_seqs[s].gt_p[0], rep_seqs[s].gt_v[0], np.zeros(3), np.zeros(3))
    for j in range(12):
        feed.push_until(j)
        imgs = np.stack([rep_seqs[s].images[j] for s in range(S)]); t_img = np.array([rep_seqs[s].img_t[j] for s in range(S)])
        b.step(imgs, t_img, feed.buf, feed.n)
    st = b.get_states()
    for s in range(2, S):
        assert np.array_equal(st[s], st[s % 2]), s
    for s in (0, 1, 63):
        P = b.get_covariance(s)
        assert np.abs(P - P.T).max() == 0.0 and np.linalg.eigvalsh(P).min() > -1e-12
        assert abs(np.linalg.norm(st[s, 1:5]) - 1) < 1e-9
    b.close()


def _pool_sequences(cfg_raw, ids, n_frames):
    """Render sequences on all host cores.  bench.generate forks a worker pool; forking THIS process (CUDA initialised, BLAS
    and driver threads running) can deadlock, so a fresh child process renders into bench.py's on-disk input cache and this
    process only loads the result."""
    import json
    import subprocess
    import tempfile
    sys.path.insert(0, ROOT)
    import bench
    cache = tempfile.mkdtemp(prefix="lvb_test_cache_")
    code = ("import sys, json; sys.path.insert(0, %r); import bench\n"
            "a = json.load(open(sys.argv[1])); bench.generate(a['cfg'], a['ids'], a['nf'], bench.effective_cores())\n") % ROOT
    spec = os.path.join(cache, "spec.json")
    json.dump(dict(cfg=cfg_raw, ids=list(ids), nf=n_frames), open(spec, "w"))
    env = dict(os.environ, LVB_BENCH_CACHE=cache)
    r = subprocess.run([sys.executable, "-c", code, spec], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    old = os.environ.get("LVB_BENCH_CACHE")
    os.environ["LVB_BENCH_CACHE"] = cache
    try:
        # same key <=> same json round trip of the config as the child saw
        seqs = bench.generate(json.load(open(spec))["cfg"], list(ids), n_frames, 1)
    finally:
        if old is None:
            os.environ.pop("LVB_BENCH_CACHE", None)
        else:
            os.environ["LVB_BENCH_CACHE"] = old
    import shutil
    shutil.rmtree(cache, ignore_errors=True)
    return seqs


def test_baseline_config_c_full_window_matches_oracle(lib_built):
    """BASELINE configs[1]/[2] at steady state: sw_size 30, 200 tracks, MSCKF-only, 4 DISTINCT sequences, 84 frames - the
    30-pose window fills after ~60 frames, so QR compression and pruneImuStateBuffer (larvio.cpp:2310-2641) run on a
    full window (d = 202) for the last ~10 published frames.  Ids bit-exact, filter within 1e-8 of the oracle."""
    from larvio_b200.config import Config
    c = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_in_one_grid=0, sw_size=30)
    sq = _pool_sequences(c.raw, range(10, 14), 84)
    rep = _drive(c, sq, 84, 'step', S=4)
    assert rep['steps'] >= 4 * 38 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['max_dim'] >= 22 + 6 * 28                                # the window reached its capacity (pruned back to 28 after every second update)
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8
    rep_fe = _drive(c, sq[:2], 30, 'fe', S=2)
    assert rep_fe['id_mismatch'] == 0 and rep_fe['uv'] == 0.0


def test_baseline_config_e_with_slam_features_in_the_state(lib_built):
    """BASELINE configs[4] per sequence, long enough that it is what the config string says: 400 tracks, 50-pose window,
    4x5 grid -> SLAM features are promoted 5 s after the start (larvio.cpp:1974) and the window passes 40 poses."""
    from larvio_b200.config import Config
    ec = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_num=400, sw_size=50, aug_grid_rows=4, aug_grid_cols=5,
                     min_distance=14)
    es = _pool_sequences(ec.raw, range(2), 132)
    rep = _drive(ec, es, 132, 'step')
    assert rep['steps'] >= 2 * 60 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['max_slam'] >= 10 and rep['max_dim'] >= 22 + 6 * 40 + 10
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8


def test_full_batch_of_distinct_sequences_matches_oracle_on_a_sample(cfg):
    """BASELINE's batch size with 64 DISTINCT sequences: 24 frames through lvb_step, a sample of sequences spread over the
    batch (first, last, sub-batch seams) is compared with its own oracle run; every sequence must publish like its oracle twin."""
    from larvio_b200 import api, harness
    from oracle.frontend import ImageProcessorOracle
    from oracle.backend import LarVioOracle
    from larvio_b200 import synth
    S, NF = 64, 24
    sq = _pool_sequences(cfg.raw, range(100, 100 + S), NF)
    sample = [0, 15, 16, 31, 47, 63]
    b = api.Batch(cfg, n_seq=S)
    feed = harness.ImuFeeder(sq)
    fes = {s: ImageProcessorOracle(cfg.raw) for s in sample}; bes = {s: LarVioOracle(cfg.raw) for s in sample}
    imu_o = {s: [] for s in sample}; k = {s: 0 for s in sample}
    for s in range(S):
        b.set_initial_state(s, sq[s].img_t[0], sq[s].gt_q[0], sq[s].gt_p[0], sq[s].gt_v[0], np.zeros(3), np.zeros(3))
    for s in sample:
        bes[s].set_initial_state(sq[s].img_t[0], sq[s].gt_q[0], sq[s].gt_p[0], sq[s].gt_v[0], np.zeros(3), np.zeros(3))
    worst = 0.0; steps = 0
    for j in range(NF):
        feed.push_until(j)
        imgs = np.stack([sq[s].images[j] for s in range(S)]); t_img = np.array([sq[s].img_t[j] for s in range(S)])
        ok = b.step(imgs, t_img, feed.buf, feed.n)
        for s in sample:
            k2 = synth.imu_window(sq[s], k[s], sq[s].img_t[j]); imu_o[s].extend(sq[s].imu[k[s]:k2].tolist()); k[s] = k2
            msg = fes[s].process_image(sq[s].images[j], sq[s].img_t[j], np.array(imu_o[s]).reshape(-1, 7))
            oko = bes[s].process_features(msg, imu_o[s]) if msg is not None else False
            assert bool(ok[s]) == bool(oko), (j, s)
            if oko:
                st = b.get_state(s); o = bes[s].imu_state
                worst = max(worst, float(np.abs(st['p'] - o.p).max()), float(np.abs(st['v'] - o.v).max()))
                P = b.get_covariance(s)
                worst = max(worst, float(np.linalg.norm(P - bes[s].P) / np.linalg.norm(bes[s].P)))
                steps += 1
    b.close()
    assert steps >= len(sample) * 10 and worst < 1e-8


def test_more_than_64_pending_imu_samples_are_consumed_like_the_reference(lib_built):
    """pub_frequency 2 Hz with a 200 Hz IMU leaves ~100 samples in the caller's buffer per feature message.
    batchImuProcessing consumes the whole buffer (larvio.cpp:464-512); the per-call staging grows to hold it (it used to
    be capped at 64 samples, which would have stopped the propagation short of the message time)."""
    from larvio_b200 import synth
    from larvio_b200.config import Config
    c = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_in_one_grid=0, sw_size=12, pub_frequency=2)
    sq = [synth.make_sequence(c.raw, 20 + s, 64) for s in range(2)]
    rep = _drive(c, sq, 64, 'step')
    assert rep['steps'] >= 2 * 5 and rep['ok_mismatch'] == 0 and rep['imu_mismatch'] == 0
    assert rep['p'] < 1e-8 and rep['v'] < 1e-8 and rep['q'] < 1e-8 and rep['Prel'] < 1e-8


def test_sharded_batch_through_the_c_abi_matches_one_handle(cfg, seqs):
    """lvbm_* (SURVEY 8b/8e): 6 sequences split into 3 shards (all on GPU 0 here; one per GPU on a node), every shard stepped by
    its own host thread.  Sequences never interact, so the gathered states must be bit-identical to one 6-sequence handle."""
    from larvio_b200 import api, harness
    S = 6
    sq = [seqs[s % 2] for s in range(S)]
    one = api.Batch(cfg, n_seq=S)
    many = api.MultiBatch(cfg, S, [0, 0, 0])
    f1 = harness.ImuFeeder(sq); f2 = harness.ImuFeeder(sq)
    for s in range(S):
        a = (sq[s].img_t[0], sq[s].gt_q[0], sq[s].gt_p[0], sq[s].gt_v[0], np.zeros(3), np.zeros(3))
        one.set_initial_state(s, *a); many.set_initial_state(s, *a)
    for j in range(12):
        f1.push_until(j); f2.push_until(j)
        imgs = np.stack([sq[s].images[j] for s in range(S)]); t_img = np.array([sq[s].img_t[j] for s in range(S)])
        p1 = one.step(imgs, t_img, f1.buf, f1.n)
        p2 = many.step(imgs, t_img, f2.buf, f2.n)
        assert np.array_equal(p1, p2) and np.array_equal(f1.n, f2.n)
    assert np.array_equal(one.get_states(), many.get_states())
    assert many.launches > 0
    one.close(); many.close()


def test_unsupported_configs_fail_loudly(lib_built):
    from larvio_b200 import api
    from larvio_b200.config import Config
    c = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_in_one_grid=3)     # 3 x 30 cells: beyond the 64-feature SLAM block
    b = api.Batch(c, n_seq=1)
    imu = np.zeros((1, 8), api.IMU_DTYPE); n = np.zeros(1, np.int32)
    with pytest.raises(api.LarvioB200Error) as e:
        b.step(np.zeros((1, 480, 752), np.uint8), np.array([0.1]), imu, n)
    assert "more than 64 EKF-SLAM features" in str(e.value)
    b.close()


# ---- the CUDA back end against golden vectors the REFERENCE ITSELF produced (tests/golden/ref_*.npz) ---------------------------------
REF_CASES_GPU = ["msckf_sw30", "msckf_oldest", "hybrid_1d_oldest", "hybrid_3d", "config_d", "zupt", "self_start", "no_fej_no_calib", "calib_3d", "schmidt_1d_oldest",
                 "schmidt_3d_oldest", "hybrid_zupt", "self_start_jump"]


def _drive_fixture(name):
    """Replay the recorded processFeatures calls of one fixture through lvb_process_features (host feature messages + the
    caller's IMU buffer, consumed samples erased like larvio.cpp:510-512) and compare every call with what the compiled
    reference answered (tests/ref_runner.compare_with_fixture).  The self-start case runs the host-side static initialiser
    (lvb_static_init_*) on the same messages, as larvio.cpp:375-391 does."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_runner as rr
    from larvio_b200 import api
    from larvio_b200.config import Config
    ov, init, static_init, calls, ref = rr.load_fixture(os.path.join(ROOT, "tests", "golden", "ref_%s.npz" % name))
    c = Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), **ov)
    b = api.Batch(c, n_seq=1)
    host_init = api.StaticInitializer(c) if static_init else None
    cap = b.cap
    buf = np.zeros((1, 1024), api.IMU_DTYPE); n_buf = np.zeros(1, np.int32)
    started = False; first = False
    run = []
    for cl in calls:
        m = len(cl["imu"]); n0 = int(n_buf[0])
        buf["t"][0, n0:n0 + m] = cl["imu"][:, 0]; buf["gyro"][0, n0:n0 + m] = cl["imu"][:, 1:4]; buf["acc"][0, n0:n0 + m] = cl["imu"][:, 4:7]
        n_buf[0] = n0 + m
        n = len(cl["ids"])
        feat = np.zeros((1, cap), api.FEATURE_DTYPE)
        feat["id"][0, :n] = cl["ids"]
        for k, col in enumerate(["u", "v", "u_init", "v_init", "u_vel", "v_vel", "u_init_vel", "v_init_vel"]):
            feat[col][0, :n] = cl["data"][:, k]
        if not started:
            if init is not None:
                b.set_initial_state(0, *init); started = True
            else:
                if not first:                                            # bFirstFeatures gate, larvio.cpp:365-372 (td = 0 in the fixtures)
                    if n_buf[0] > 0 and buf["t"][0, 0] - cl["t"] <= 0.0:
                        first = True
                    else:
                        run.append(dict(ok=False)); continue
                a = host_init.try_init(feat[0, :n], cl["t"], buf[0, :n_buf[0]])
                if a is None:
                    run.append(dict(ok=False)); continue
                b.set_initial_state(0, a["t"], a["q"], a["p"], a["v"], a["bg"], a["ba"])
                nc = a["n_consumed"]                                     # StaticInitializer.cpp:149-150
                buf[0, :n_buf[0] - nc] = buf[0, nc:n_buf[0]].copy(); n_buf[0] -= nc
                started = True
        ok = b.process_features(np.ones(1, np.uint8), np.array([cl["t"]]), feat, np.array([n], np.int32), buf, n_buf)
        rec = dict(ok=bool(ok[0]))
        if rec["ok"]:
            st = b.get_state(0); cal = b.get_calibration(0); P = b.get_covariance(0)
            rec.update(q=st["q"], p=st["p"], v=st["v"], bg=st["bg"], ba=st["ba"], R_imu_cam0=cal["R_imu_cam0"], t_cam0_imu=cal["t_cam0_imu"],
                       td=float(cal["td"]), P=P, n_win=len(b.get_window(0)),
                       n_imu_left=int(n_buf[0]), Tg=cal["Tg"], As=cal["As"], Ma=cal["Ma"],
                       stable=b.get_points(0, 0), active=b.get_points(0, 1))          # larvio.h:86-87, read (and cleared) after every call like the fixture
        run.append(rec)
    b.close()
    if host_init is not None:
        host_init.close()
    w = rr.compare_with_fixture(run, ref)
    w["calib"] = max([float(max(np.abs(x["Tg"] - y["Tg"]).max(), np.abs(x["As"] - y["As"]).max(), np.abs(x["Ma"] - y["Ma"]).max()))
                      for x, y in zip(run, ref) if y["ok"] and "Tg" in x] or [0.0])
    return w


@pytest.mark.parametrize("name", REF_CASES_GPU)
def test_backend_matches_the_compiled_reference(name, lib_built):
    """The CUDA filter against the REFERENCE's own answers (not the numpy oracle): fixtures made by /root/reference/src/larvio.cpp
    compiled unmodified (oracle/_ref, tests/golden/make_ref_golden.py).  Per call: same return value, state dimension and IMU
    samples left; pose, velocity, biases, extrinsics, td within 1e-8; covariance fingerprints (P z, diag P, full P of the last
    call) within 1e-8 relative; IMU intrinsics within 1e-9."""
    w = _drive_fixture(name)
    assert w["n"] >= 18, w
    assert max(w["q"], w["p"], w["v"], w["bg"], w["ba"], w["ext"], w["td"]) < 1e-8, w
    assert max(w["Pz"], w["Pdiag"], w["P"]) < 1e-8 and w["calib"] < 1e-9, w
    assert w["pts"] < 1e-7 and (w["n_pts"] > 0) == (name in ("hybrid_1d_oldest", "hybrid_3d", "config_d", "calib_3d", "hybrid_zupt", "schmidt_1d_oldest", "schmidt_3d_oldest")), w   # map-point getters


# ---- the CUDA front end against the feature messages the REFERENCE's own front end published (tests/golden/ref_fe_*.npz) ------------
REF_FE_CASES_GPU = ["fe_plain", "fe_blackout", "fe_failed_second", "fe_400_tracks", "fe_static_start"]


def _drive_fe_fixture(name):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_runner as rr
    from larvio_b200 import api, harness
    cfg, seq, nf = rr.fe_case_sequence(name)
    ref, _ = rr.load_fe_fixture(os.path.join(ROOT, "tests", "golden", "ref_%s.npz" % name))
    b = api.Batch(cfg, n_seq=1)
    feed = harness.ImuFeeder([seq], stride=2048)            # the front end only reads the caller's buffer (processImage takes it const)
    msgs = []
    for j in range(nf):
        feed.push_until(j)
        feat, out_n, has = b.process_images(seq.images[j][None], np.array([seq.img_t[j]]), feed.buf, feed.n)
        if not has[0]:
            msgs.append(None); continue
        g = feat[0, :out_n[0]]
        msgs.append(dict(ids=g['id'].copy(), data=np.stack([g[c] for c in ['u', 'v', 'u_init', 'v_init', 'u_vel', 'v_vel', 'u_init_vel', 'v_init_vel']], 1)))
    b.close()
    return rr.compare_fe(msgs, ref)


@pytest.mark.parametrize("name", REF_FE_CASES_GPU)
def test_frontend_matches_the_compiled_reference(name, lib_built):
    """lvb_process_images against what the reference's own image_processor.cpp + ORBDescriptor.cpp published on the same images
    (compiled unmodified, OpenCV functions executed by cv2 4.13; tests/golden/make_ref_fe_golden.py): the same frames publish, ids
    and their order bit-exact, all eight message columns bit-identical."""
    n_pub, bad_ids, worst = _drive_fe_fixture(name)
    assert n_pub >= 10 and bad_ids == 0 and worst == 0.0, (n_pub, bad_ids, worst)


def test_shim_facade_matches_the_whole_reference_pipeline(tmp_path, lib_built):
    """The drop-in claim end to end: larvio_b200/bin/larvio_shim_demo (app/larvioMain.cpp's loop on the shim's ImageProcessor /
    LarVio over the CUDA library) against the reference's own five source files compiled unmodified behind the same loop
    (oracle/_ref/larvio_ref_main; tests/golden/ref_main_hybrid_selfstart.txt) on the same on-disk sequence: euroc.yaml defaults
    (hybrid, 5x6 SLAM grid), self start from a standstill.  Same publications, rotation / position / velocity within 1e-8,
    identical map-point lists within 1e-7."""
    import subprocess
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_runner as rr
    from larvio_b200 import synth
    from larvio_b200.config import Config
    cfg_path = os.path.join(ROOT, "configs", "euroc_mono.yaml")
    c = Config.load(cfg_path)
    seq = synth.make_sequence(c.raw, 3, 150, static_until=1.4)          # tests/golden/make_ref_main_golden.py: SPEC
    mav = rr.write_mav(tmp_path, seq)
    exe = os.path.join(ROOT, "larvio_b200", "bin", "larvio_shim_demo")
    r = subprocess.run([exe, cfg_path, str(mav)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    w = rr.compare_odometry(r.stdout, open(os.path.join(ROOT, "tests", "golden", "ref_main_hybrid_selfstart.txt")).read())
    assert w["n"] >= 60 and w["n_lists"] >= 2 and w["t"] < 1e-9 and max(w["R"], w["p"], w["v"]) < 1e-8 and w["pts"] < 1e-7, w


def test_replay_tool_writes_the_file_the_reference_writes(tmp_path, lib_built):
    """SURVEY 8(f-4), both directions of the on-disk formats: larvio_b200/bin/larvio_replay reads the EuRoC ASL directory (PNG + csv)
    and writes msckf_2_state.txt / msckf_2_takeoff.txt; the reference's own LarVio wrote the same two files while its whole
    pipeline (oracle/_ref/larvio_ref_main) ran on the same directory (tests/golden/ref_main_msckf_2_state.txt, _takeoff.txt).
    Same number of lines, same 24 columns, values equal to the 6 significant digits of the format."""
    import subprocess
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_runner as rr
    from larvio_b200 import synth
    from larvio_b200.config import Config
    cfg_path = os.path.join(ROOT, "configs", "euroc_mono.yaml")
    c = Config.load(cfg_path)
    seq = synth.make_sequence(c.raw, 3, 150, static_until=1.4)          # tests/golden/make_ref_main_golden.py: SPEC
    mav = rr.write_mav(tmp_path, seq)
    exe = os.path.join(ROOT, "larvio_b200", "bin", "larvio_replay")
    r = subprocess.run([exe, cfg_path, str(tmp_path / "out"), str(mav)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = np.loadtxt(str(tmp_path / "out" / "seq0" / "msckf_2_state.txt"), ndmin=2)
    ref = np.loadtxt(os.path.join(ROOT, "tests", "golden", "ref_main_msckf_2_state.txt"), ndmin=2)
    assert got.shape == ref.shape and ref.shape[1] == 24 and ref.shape[0] >= 60
    assert np.allclose(got, ref, rtol=2e-5, atol=2e-6)
    assert open(str(tmp_path / "out" / "seq0" / "msckf_2_takeoff.txt")).read().split() == open(os.path.join(ROOT, "tests", "golden", "ref_main_msckf_2_takeoff.txt")).read().split()
