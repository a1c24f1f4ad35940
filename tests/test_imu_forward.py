"""The IMU forward pass of kalman::EKF::motion_compensation_with_imu (L/src/kalman/ekf.cpp:292-418; SURVEY section 8f N1) --
limu_imu_forward_pass, HOST code inside liblimu_cuda (callable without a GPU) -- against the reference's own EKF compiled
unmodified (oracle/ref_ekf_driver.cpp): pose table, scan-end rotation and scan-end lidar position to 1e-12 (closed-form exp(S)
versus Eigen's Pade approximant), and the deskewed float points that come out of the per-point loop fed with OUR table:
identical through the C oracle's loop (CPU), <= 1 float ulp through the CUDA kernel (GPU).
"""
import numpy as np
import pytest


def window(rng, k=22, t0=50.0, n=4000, gyr=(0.02, -0.01, 0.35), acc=(0.3, -0.2, 9.81), dt=0.005, first_offset=-0.004):
    ts = t0 + first_offset + np.arange(k) * dt
    imu = np.concatenate([ts[:, None], np.array(gyr) + rng.normal(size=(k, 3)) * 0.002, np.array(acc) + rng.normal(size=(k, 3)) * 0.03], 1)
    curv = np.sort(rng.random(n) * 100.0).astype(np.float32)
    xyz = (rng.normal(size=(n, 3)) * 25).astype(np.float32)
    return imu, curv, xyz


def make_state(pkg, mean_acc, pil, bg, last_end=0.0, row0=None):
    st = pkg.ImuState()
    st.quat[:] = [1, 0, 0, 0]                     # the EKF constructor's ORI (ekf.cpp:101)
    st.bat[:] = [1, 1, 1]                         # BAT (:103); BAA, POS, VEL stay zero
    st.bga[:] = bg
    st.grav[:] = [0, 0, -9.81]                    # grav (:80)
    st.p_imu_lidar[:] = pil
    st.mean_acc_norm = float(np.linalg.norm(mean_acc))
    st.gravity_norm = 9.81
    st.last_lidar_end_time = last_end
    if row0 is not None:                          # the tracker's acc_s_last / ang_vel_last are uninitialised in a fresh reference EKF:
        st.acc_s_last[:] = row0[1:4]              # take whatever it put into row 0
        st.ang_vel_last[:] = row0[4:7]
    return st


def forward_and_reference(pkg, ref, rng, last_end=0.0, **kw):
    imu, curv, xyz = window(rng, **kw)
    t0 = kw.get("t0", 50.0)
    mean_acc, pil, bg = [0.3, -0.2, 9.81], [0.1, -0.05, 0.2], [0.001, 0.002, -0.001]
    ref.imu_set_last_lidar_end_time(last_end)
    r = ref.imu_deskew_reference(xyz, curv, imu, t0, mean_acc, pil, bg)
    ref.imu_set_last_lidar_end_time(0.0)
    st = make_state(pkg, mean_acc, pil, bg, last_end, r["table"][0])
    table, rot_end, ple = pkg.imu_forward_pass(st, imu, t0, float(curv[-1]))
    return r, table, rot_end, ple, st, (xyz, curv, pil)


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    return g.load_package()


@pytest.mark.parametrize("case", [dict(), dict(k=2, n=50), dict(k=41, dt=0.0025, n=300), dict(gyr=(1.2, -0.8, 2.5), acc=(2.0, 1.0, 9.0)),
                                  dict(gyr=(0.0, 0.0, 0.0)), dict(first_offset=-0.03)])
def test_forward_pass_matches_the_reference_ekf(pkg, ref, port, rng, case):
    r, table, rot_end, ple, st, (xyz, curv, pil) = forward_and_reference(pkg, ref, rng, **case)
    assert table.shape == r["table"].shape
    np.testing.assert_allclose(table, r["table"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(rot_end, r["rot_end"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(ple, r["pos_lidar_end"], rtol=0, atol=1e-12)
    assert st.last_lidar_end_time == 50.0 + float(curv[-1]) / 1000.0                      # ekf.cpp:413
    assert np.array_equal(np.array(st.acc_s_last), table[-1, 1:4]) and np.array_equal(np.array(st.ang_vel_last), table[-1, 4:7])
    out, wb = port.deskew_imu(xyz, curv, table, rot_end, ple, pil)                        # the per-point loop fed with OUR table
    ulp = np.spacing(np.abs(r["written_back"]).astype(np.float32))
    assert np.all(np.abs(wb - r["written_back"]) <= ulp) and (wb != r["written_back"]).mean() < 1e-3


def test_forward_pass_matches_golden_table(pkg, port):
    """The same checks against the reference's outputs recorded by tests/golden/make_golden.py on its IMU window (22 samples at 200 Hz,
    turning and accelerating platform) with the scan start, mean acceleration and gyro bias stored beside it: no compiled reference needed."""
    from test_golden import PA
    t0 = float(PA["imu_t0"])
    st = make_state(pkg, PA["imu_mean_acc"], PA["imu_pil"], PA["imu_bg"], 0.0, PA["imu_table"][0])
    curv = PA["imu_curv"]
    table, rot_end, ple = pkg.imu_forward_pass(st, PA["imu_samples"], t0, float(curv[-1]))
    assert table.shape == PA["imu_table"].shape
    np.testing.assert_allclose(table, PA["imu_table"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(rot_end, PA["imu_rot_end"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(ple, PA["imu_pos_lidar_end"], rtol=0, atol=1e-12)
    assert st.last_lidar_end_time == t0 + float(curv[-1]) / 1000.0
    assert np.array_equal(np.array(st.acc_s_last), table[-1, 1:4]) and np.array_equal(np.array(st.ang_vel_last), table[-1, 4:7])
    out, wb = port.deskew_imu(PA["imu_xyz"], curv, table, rot_end, ple, PA["imu_pil"])
    ulp = np.spacing(np.abs(PA["imu_written_back"]).astype(np.float32))
    assert np.all(np.abs(wb - PA["imu_written_back"]) <= ulp) and (wb != PA["imu_written_back"]).mean() < 1e-3


def _random_seeds_n():
    """4 seeds in the suite; LIMU_RANDOM_SEEDS_N="lo-hi" widens the campaign (profiles/r2_random_campaign.json)."""
    import os
    spec = os.environ.get("LIMU_RANDOM_SEEDS_N", "")
    if "-" in spec:
        lo, hi = spec.split("-")
        return range(int(lo), int(hi))
    return range(6000, 6004)


@pytest.mark.parametrize("seed", _random_seeds_n())
def test_forward_pass_matches_the_reference_ekf_on_random_windows(pkg, ref, port, seed):
    """Seeded random IMU windows (2 .. 60 samples at 100 / 200 / 400 Hz, rates up to ~3 rad/s, accelerations up to ~2 g, where the window
    starts before the scan) through limu_imu_forward_pass and through the compiled reference's own forward pass: pose table, scan-end
    rotation and lidar position to 1e-11; the per-point loop fed with OUR table writes the reference's floats back (<= 1 ulp)."""
    r_ = np.random.default_rng(seed)
    case = dict(k=int(r_.integers(2, 61)), dt=float(r_.choice([0.0025, 0.005, 0.01])), n=int(r_.integers(50, 3000)),
                gyr=tuple(r_.normal(size=3) * r_.choice([0.05, 0.5, 1.5])), acc=tuple(np.array([0.0, 0.0, 9.81]) + r_.normal(size=3) * r_.choice([0.3, 3.0])),
                first_offset=-float(r_.uniform(1e-4, 0.03)))
    r, table, rot_end, ple, st, (xyz, curv, pil) = forward_and_reference(pkg, ref, r_, **case)
    assert table.shape == r["table"].shape, case
    np.testing.assert_allclose(table, r["table"], rtol=0, atol=1e-11, err_msg=str(case))
    np.testing.assert_allclose(rot_end, r["rot_end"], rtol=0, atol=1e-11, err_msg=str(case))
    np.testing.assert_allclose(ple, r["pos_lidar_end"], rtol=0, atol=1e-11, err_msg=str(case))
    out, wb = port.deskew_imu(xyz, curv, table, rot_end, ple, pil)
    ulp = np.spacing(np.abs(r["written_back"]).astype(np.float32))
    assert np.all(np.abs(wb - r["written_back"]) <= ulp), case


@pytest.mark.parametrize("last_end", [50.013, 50.0301, 49.99, 50.0958])   # (with every pair skipped the reference reads uninitialised vectors)
def test_pairs_older_than_the_previous_scan_end(pkg, ref, rng, last_end):
    """ekf.cpp:322-323 (pairs entirely before the previous scan's end are skipped) and :340-341 (the straddling pair is cut)."""
    r, table, rot_end, ple, st, _ = forward_and_reference(pkg, ref, rng, last_end=last_end)
    assert table.shape == r["table"].shape and (len(table) < 22 or last_end < 50.0)
    np.testing.assert_allclose(table, r["table"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(rot_end, r["rot_end"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(ple, r["pos_lidar_end"], rtol=0, atol=1e-12)


def test_argument_checks(pkg, rng):
    imu, curv, _ = window(rng)
    st = make_state(pkg, [0, 0, 9.81], [0, 0, 0], [0, 0, 0])
    with pytest.raises(pkg.LimuError):
        pkg.imu_forward_pass(st, imu[:1], 50.0, 10.0)          # a window needs the previous sample and at least one new one
    st.mean_acc_norm = 0.0
    with pytest.raises(pkg.LimuError):
        pkg.imu_forward_pass(st, imu, 50.0, 10.0)


@pytest.mark.gpu
def test_forward_pass_feeds_the_cuda_deskew(pkg, ref, rng):
    r, table, rot_end, ple, st, (xyz, curv, pil) = forward_and_reference(pkg, ref, rng)
    ctx = pkg.Context(0)
    out, wb = ctx.deskew_imu(np.concatenate([xyz, curv[:, None]], 1).astype(np.float32), table, rot_end, ple, pil)
    ulp = np.spacing(np.abs(r["written_back"]).astype(np.float32))
    assert np.all(np.abs(wb - r["written_back"]) <= ulp) and (wb != r["written_back"]).mean() < 1e-3
    assert np.array_equal(out, wb.astype(np.float64))
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", _random_seeds_n())
def test_cuda_deskew_on_random_windows(pkg, ref, seed):
    """The same random windows through the CUDA per-point loop (limu_deskew_imu, csrc/imu_deskew.cu) fed with OUR forward pass:
    the reference's written-back floats within 1 ulp."""
    r_ = np.random.default_rng(seed)
    case = dict(k=int(r_.integers(2, 61)), dt=float(r_.choice([0.0025, 0.005, 0.01])), n=int(r_.integers(50, 3000)),
                gyr=tuple(r_.normal(size=3) * r_.choice([0.05, 0.5, 1.5])), acc=tuple(np.array([0.0, 0.0, 9.81]) + r_.normal(size=3) * r_.choice([0.3, 3.0])),
                first_offset=-float(r_.uniform(1e-4, 0.03)))
    r, table, rot_end, ple, st, (xyz, curv, pil) = forward_and_reference(pkg, ref, r_, **case)
    ctx = pkg.Context(0)
    out, wb = ctx.deskew_imu(np.concatenate([xyz, curv[:, None]], 1).astype(np.float32), table, rot_end, ple, pil)
    ulp = np.spacing(np.abs(r["written_back"]).astype(np.float32))
    assert np.all(np.abs(wb - r["written_back"]) <= ulp), case
    assert np.array_equal(out, wb.astype(np.float64))
    ctx.close()
