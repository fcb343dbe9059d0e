"""The C++ readers / writers of the reference's file formats (include/b200ba_io.hpp) and the C++ outlier deletion /
metric rescaling (include/b200ba_pipeline.hpp) against their Python mirrors (io.py, pipeline.py): files written by
one side are read by the other. Host logic only -- no device work."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    from camera_calibration_b200 import build
    build.build()
    path = str(tmp_path_factory.mktemp("io_example") / "b200ba_io_example")
    lib_dir = os.path.join(ROOT, "camera_calibration_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "io_example.cc"), "-o", path, "-L", lib_dir, "-lb200ba",
                           f"-Wl,-rpath,{lib_dir}"])
    return path


def _problem(cfg, **kw):
    """(dataset, state) of a small synthetic problem with one known geometry (the pattern lattice)."""
    from camera_calibration_b200 import api, io, synthetic
    sp = synthetic.make_problem(cfg, **kw)
    ds, st = api.dataset_from_flat(sp.problem, sp.init_state)
    for i in range(ds.ImagesetCount()):
        ds.GetImageset(i).SetFilename(f"image{i:04d}.png")
    g = io.KnownGeometry()
    g.cell_length_in_meters = float(np.float32(0.024))
    nx = kw.get("lattice", (10, 10))[0]
    for fid, idx in st.feature_id_to_points_index.items():
        g.feature_id_to_position[int(fid)] = (int(idx) % nx, int(idx) // nx)
    ds.known_geometries = [g]
    return ds, st


def _run(exe, *args, rc=0):
    r = subprocess.run([exe, *args], capture_output=True, text=True)
    assert r.returncode == rc, (args, r.stdout, r.stderr)
    return r.stdout


def _states_equal(a, b, tol=1e-13):
    assert list(a.image_used) == list(b.image_used)
    assert np.allclose(a.rig_tr_global, b.rig_tr_global, rtol=0, atol=tol)
    assert np.allclose(a.camera_tr_rig, b.camera_tr_rig, rtol=0, atol=tol)
    assert np.allclose(a.points, b.points, rtol=0, atol=tol)
    assert dict(a.feature_id_to_points_index) == dict(b.feature_id_to_points_index)
    assert len(a.intrinsics) == len(b.intrinsics)
    for m, k in zip(a.intrinsics, b.intrinsics):
        assert type(m) is type(k)
        assert (m.width(), m.height()) == (k.width(), k.height())
        assert np.allclose(m.flat_intrinsics(), k.flat_intrinsics(), rtol=0, atol=tol)


@pytest.mark.parametrize("cfg", [1, 2, 3, 4])
def test_dataset_and_state_round_trip_through_cpp(exe, tmp_path, cfg):
    from camera_calibration_b200 import io
    ds, st = _problem(cfg, n_imagesets=6, lattice=(8, 7), image_size=(410, 290))
    st.image_used[2] = False
    src, dst = tmp_path / "py", tmp_path / "cpp"
    assert io.SaveDataset(str(src / "dataset.bin"), ds)
    assert io.SaveBAState(str(src / "state"), st)
    out = _run(exe, "dataset", str(src / "dataset.bin"), str(dst / "dataset.bin"))
    assert f"cameras {ds.num_cameras()} imagesets {ds.ImagesetCount()} geometries 1" in out
    # dataset.bin is byte-exact (integers big-endian, floats raw)
    assert (src / "dataset.bin").read_bytes() == (dst / "dataset.bin").read_bytes()
    out = _run(exe, "state", str(src / "state"), str(dst / "state"), str(src / "dataset.bin"))
    assert f"cameras {ds.num_cameras()} imagesets {ds.ImagesetCount()} points {len(st.points)}" in out
    # ComputeFeatureIdToPointsIndex ran on the C++ side: same indices as the Python dataset carries
    index_sum = sum(int(ds.GetImageset(i).FeaturesOfCamera(c)["index"].sum())
                    for i in range(ds.ImagesetCount()) for c in range(ds.num_cameras()))
    assert f"index_sum {index_sum}" in out
    ref = io.LoadBAState(str(src / "state"))
    got = io.LoadBAState(str(dst / "state"))
    assert ref is not None and got is not None
    _states_equal(ref, got)
    # the text the two writers produce for poses is identical (same 14-digit formatting)
    assert (src / "state" / "rig_tr_global.yaml").read_text() == (dst / "state" / "rig_tr_global.yaml").read_text()
    assert (src / "state" / "camera_tr_rig.yaml").read_text() == (dst / "state" / "camera_tr_rig.yaml").read_text()


def test_cpp_loaders_reject_malformed_files(exe, tmp_path):
    from camera_calibration_b200 import io
    ds, st = _problem(2, n_imagesets=4, lattice=(8, 7), image_size=(410, 290))
    io.SaveDataset(str(tmp_path / "dataset.bin"), ds)
    data = (tmp_path / "dataset.bin").read_bytes()
    cases = {"truncated.bin": data[:len(data) // 2], "foreign.bin": b"not_calib_" + data[10:], "empty.yaml": b"",
             "garbage.yaml": b"pose_count: x\nposes: 3\npoints : [1, 2\n", "missing": None}
    for name, content in cases.items():
        p = tmp_path / name
        if content is not None:
            p.write_bytes(content)
        assert _run(exe, "malformed", str(p)).strip() == "0 0 0 0", name
    # a state directory whose mapping does not cover the dataset's feature ids is rejected, not dereferenced
    io.SaveBAState(str(tmp_path / "state"), st)
    text = (tmp_path / "state" / "points.yaml").read_text()
    (tmp_path / "state" / "points.yaml").write_text(text[:text.rindex("  - feature_id")])
    out = _run(exe, "state", str(tmp_path / "state"), str(tmp_path / "out"), str(tmp_path / "dataset.bin"), rc=1)
    assert "load failed" in out


def test_cpp_scale_to_metric_matches_python(exe, tmp_path):
    from camera_calibration_b200 import io, pipeline
    ds, st = _problem(3, n_imagesets=5, lattice=(8, 7), image_size=(410, 290))
    io.SaveDataset(str(tmp_path / "dataset.bin"), ds)
    io.SaveBAState(str(tmp_path / "state"), st)
    out = _run(exe, "scale", str(tmp_path / "dataset.bin"), str(tmp_path / "state"), str(tmp_path / "scaled"))
    cpp_factor = float(out.split("factor")[1].split()[0])
    ref = io.LoadBAState(str(tmp_path / "state"), ds)
    factor = pipeline.ScaleToMetric(ds, ref)
    assert abs(cpp_factor - factor) <= 1e-13 * factor
    got = io.LoadBAState(str(tmp_path / "scaled"))
    # the non-central model's line origins scale with the state (noncentral_generic.cc:148-154)
    _states_equal(ref, got, tol=1e-12)


def test_cpp_delete_outlier_features_matches_python(exe, tmp_path):
    from camera_calibration_b200 import io, pipeline
    ds, st = _problem(2, n_imagesets=6, lattice=(8, 7), image_size=(410, 290))

    def pinhole(model, lp):  # the stand-in projector of tests/io_example.cc
        z = lp[:, 2]
        with np.errstate(divide="ignore", invalid="ignore"):
            u, v = 400.0 * lp[:, 0] / z + 320.0, 400.0 * lp[:, 1] / z + 240.0
        ok = (z > 0) & (u >= 0) & (v >= 0) & (u < 640) & (v < 480)
        px = np.stack([np.where(z > 0, u, 0.0), np.where(z > 0, v, 0.0)], -1)
        return px, ok

    # observations = the pinhole projection + noise, a few gross outliers, one imageset nearly wiped out
    rng = np.random.default_rng(5)
    for i in range(ds.ImagesetCount()):
        f = ds.GetImageset(i).FeaturesOfCamera(0)
        T = st.image_tr_global(0, i)
        from camera_calibration_b200 import synthetic
        px, ok = pinhole(None, synthetic.pose_apply(T, st.points[f["index"]]))
        xy = px + rng.normal(0, 0.05, px.shape)
        bad = rng.random(len(xy)) < (0.9 if i == 4 else 0.04)
        xy[bad] += rng.normal(0, 30.0, (int(bad.sum()), 2))
        f["xy"] = xy.astype(np.float32)
    io.SaveDataset(str(tmp_path / "dataset.bin"), ds)
    io.SaveBAState(str(tmp_path / "state"), st)
    out = _run(exe, "outliers", str(tmp_path / "dataset.bin"), str(tmp_path / "state"), "0", "1.5", str(tmp_path / "pruned.bin"))
    ref_ds = io.LoadDataset(str(tmp_path / "dataset.bin"))
    ref_st = io.LoadBAState(str(tmp_path / "state"), ref_ds)
    removed = pipeline.DeleteOutlierFeatures(0, ref_ds, ref_st, 1.5, project_many=pinhole)
    assert removed > 0
    assert f"removed {removed}\n" in out
    assert "used " + " ".join("1" if u else "0" for u in ref_st.image_used) in out
    got = io.LoadDataset(str(tmp_path / "pruned.bin"))
    for i in range(ref_ds.ImagesetCount()):
        a, b = ref_ds.GetImageset(i).FeaturesOfCamera(0), got.GetImageset(i).FeaturesOfCamera(0)
        assert np.array_equal(a["id"], b["id"]) and np.array_equal(a["xy"], b["xy"])


def test_cpp_pyramid_helpers_match_python(exe, tmp_path):
    from camera_calibration_b200 import io, pipeline
    for w, h, ext, approx, level in ((640, 480, 1, 50, 0), (1207, 933, 1, 37, 2), (1999, 1499, 0, 30, 4), (410, 290, 1, 20, 1)):
        rx, ry = pipeline.ComputeGridResolution(w, h, ext, approx)
        lx, ly = pipeline.CalcGridResolutionForLevel(level, rx, ry)
        assert _run(exe, "gridres", str(w), str(h), str(ext), str(approx), str(level)).split() == [str(v) for v in (rx, ry, lx, ly)]
    ds, st = _problem(4, n_imagesets=5, lattice=(8, 7), image_size=(410, 290))
    io.SaveDataset(str(tmp_path / "dataset.bin"), ds)
    used = [True] * ds.ImagesetCount()
    used[1] = False
    for cam in (0, 1):
        rect = pipeline.ComputeIntegerBoundingRectForFeatures(ds, cam, used)
        assert _run(exe, "bounds", str(tmp_path / "dataset.bin"), str(cam)).split() == [str(int(v)) for v in rect]


def _pinhole_unproject(model, px):
    """The stand-in of tests/io_example.cc for the device un-projection."""
    x, y = px[:, 0], px[:, 1]
    d = np.stack([(x - 320.0) / 400.0, (y - 240.0) / 400.0, np.ones_like(x)], -1)
    d = d / np.sqrt(d[:, 0] ** 2 + d[:, 1] ** 2 + 1.0)[:, None]
    ok = ~((x < 7.0) | ((x > 200) & (x < 204) & (y > 100) & (y < 104)))
    return d, None, ok


@pytest.mark.parametrize("source,target", [("central", 0), ("central", 1), ("noncentral", 1), ("noncentral", 0)])
def test_cpp_resample_model_matches_python(exe, tmp_path, source, target):
    """ResampleModel (calibration.cc:373-522): the host logic -- grid initialisation from the dense direction image
    incl. the closest-valid-pixel search and the linear extrapolation, the sample selection, the bilinear re-sampling of
    a non-central model -- with the two device calls replaced by the same stand-ins on both sides."""
    from camera_calibration_b200 import api, io, pipeline
    ds, st = _problem(2 if source == "central" else 3, n_imagesets=4, lattice=(8, 7), image_size=(410, 290))
    model = st.intrinsics[0]
    io.SaveCameraModel(model, str(tmp_path / "model.yaml"))
    model = io.LoadCameraModel(str(tmp_path / "model.yaml"))  # what the C++ side reads (14 digits, re-normalised)
    T = api.CameraModel.Type
    samples = []

    def no_fit(gw, gh, grid, gp, d, iterations):
        samples.append((len(gp), len(d)))
        return grid, None

    ok, new = pipeline.ResampleModel(model, np.array([1.0, 0, 0, 0, 0, 0, 0]), model.calibration_min_x(), model.calibration_min_y(),
                                     model.calibration_max_x(), model.calibration_max_y(), T.CentralGeneric if target == 0 else T.NoncentralGeneric,
                                     13, 11, fit_fn=no_fit, unproject_many=_pinhole_unproject)
    out = _run(exe, "resample", str(tmp_path / "model.yaml"), str(target), "13", "11", str(tmp_path / "new.yaml"), "-")
    if not ok:
        assert "not resampled" in out
        return
    if samples:
        assert f"samples {samples[0][0]} {samples[0][1]}" in out
    # un-normalised comparison of what was written: read the flow lists directly (LoadCameraModel re-normalises directions)
    import yaml
    got = yaml.safe_load(open(tmp_path / "new.yaml"))
    assert got["type"] == type(new).__name__ and (got["grid_width"], got["grid_height"]) == (13, 11)
    if isinstance(new, api.CentralGenericModel):
        assert np.allclose(np.array(got["grid"]), new.grid().reshape(-1), rtol=0, atol=2e-14)
    else:
        assert np.allclose(np.array(got["direction_grid"]), new.direction_grid().reshape(-1), rtol=0, atol=2e-14)
        assert np.allclose(np.array(got["point_grid"]), new.point_grid().reshape(-1), rtol=0, atol=2e-14)
