"""CPU-only checks: the C-ABI library loads and exports every symbol include/b200ba.h declares,
fails loudly without a GPU, and the host-side flattening / sharding logic is right."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from camera_calibration_b200 import api, cabi, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from camera_calibration_b200 import build
    build.build()
    return cabi.load_library()


def test_header_symbols_are_exported_and_bound():
    lib = _lib()
    header = open(os.path.join(ROOT, "include", "b200ba.h")).read()
    declared = set(re.findall(r"B200BA_API [\w\s\*]+?\b(b200ba_\w+)\(", header))
    assert declared, "no declarations found"
    assert declared == set(cabi.SYMBOLS.keys())
    for name in declared:
        assert getattr(lib, name) is not None
    assert b"b200ba" in lib.b200ba_version()


def test_struct_layouts_match_header(tmp_path):
    """sizeof of the ctypes mirrors equals what the C compiler lays out."""
    src = r'''
#include <stdio.h>
#include "b200ba.h"
int main(){printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(b200ba_camera), sizeof(b200ba_problem), sizeof(b200ba_state),
 sizeof(b200ba_options), sizeof(b200ba_report), sizeof(b200ba_timings), sizeof(b200ba_fit_report));return 0;}'''
    exe = str(tmp_path / "b200ba_sizes")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
    sizes = [int(v) for v in subprocess.check_output([exe]).split()]
    mine = [C.sizeof(t) for t in (cabi.Camera, cabi.Problem, cabi.State, cabi.Options, cabi.Report, cabi.Timings, cabi.FitReport)]
    assert sizes == mine


def test_default_options_match_reference_constants():
    lib = _lib()
    o = cabi.Options()
    lib.b200ba_default_options(C.byref(o))
    p = cabi.default_options()
    for f, _ in cabi.Options._fields_:
        assert getattr(o, f) == getattr(p, f), f
    assert o.max_lm_attempts == 50 and o.init_lambda_factor == 1e-5 and o.huber_parameter == 1.0


def test_sizes_helpers():
    lib = _lib()
    for mt, gw, gh, n_intr, n_upd in ((0, 84, 60, 3 * 5040, 2 * 5040), (1, 50, 40, 6 * 2000, 5 * 2000), (3, 0, 0, 12, 12)):
        c = cabi.Camera()
        c.model_type, c.grid_width, c.grid_height = mt, gw, gh
        assert lib.b200ba_intrinsics_size(C.byref(c)) == n_intr == c.intrinsics_size()
        assert lib.b200ba_update_parameter_count(C.byref(c)) == n_upd == c.update_parameter_count()


def test_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    sp = synthetic.make_problem(1, n_imagesets=2, lattice=(4, 4))
    with pytest.raises(api.B200BAError):
        api.BundleAdjuster(sp.problem)
    with pytest.raises(api.B200BAError):
        api.schur_solve(2, np.zeros((1, 2, 2)), np.zeros((2, 1)), np.ones((1, 1)), [0, 0], [1])


def test_missing_library_is_an_error(tmp_path):
    with pytest.raises(cabi.LibraryMissing):
        cabi.load_library(str(tmp_path / "nope.so"))


def test_product_does_not_import_oracle():
    """The product package must never route through the oracle."""
    pkg = os.path.join(ROOT, "camera_calibration_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "ba_oracle" not in text, f
    for f in ("b200ba.h", "b200ba_shim.hpp"):
        p = os.path.join(ROOT, "include", f)
        if os.path.exists(p):
            assert "oracle" not in open(p).read().replace("CPU oracle only", "")


def test_flat_problem_validation_and_sharding():
    sp = synthetic.make_problem(2, n_imagesets=7, lattice=(6, 5), image_size=(300, 220))
    p = sp.problem
    assert np.all(np.diff(p.obs_imageset.astype(np.int64)) >= 0)
    shards = [p.shard(r, 3) for r in range(3)]
    assert sum(s.n_obs for s in shards) == p.n_obs
    for r, s in enumerate(shards):
        assert np.all(s.obs_imageset % 3 == r)
        assert s.n_imagesets == p.n_imagesets and s.n_points == p.n_points
    idx = np.concatenate([p.shard_indices(r, 3) for r in range(3)])
    assert np.array_equal(np.sort(idx), np.arange(p.n_obs))
    with pytest.raises(ValueError):
        cabi.FlatProblem(p.cameras, p.n_imagesets, p.n_points, p.obs_imageset[::-1], p.obs_camera, p.obs_point, p.obs_xy)
    with pytest.raises(ValueError):
        cabi.FlatProblem(p.cameras, p.n_imagesets, 3, p.obs_imageset, p.obs_camera, p.obs_point, p.obs_xy)


def test_dataset_roundtrip_through_reference_containers():
    sp = synthetic.make_problem(4, n_imagesets=5, lattice=(6, 5), image_size=(300, 220))
    ds, st = api.dataset_from_flat(sp.problem, sp.init_state)
    assert ds.ImagesetCount() == 5 and ds.num_cameras() == 2
    # flatten again the way api._Context does, without touching the GPU
    used = [i for i, u in enumerate(st.image_used) if u]
    oi, oc, op, oxy = [], [], [], []
    for seq, i in enumerate(used):
        for c in range(ds.num_cameras()):
            f = ds.GetImageset(i).FeaturesOfCamera(c)
            oi.append(np.full(len(f["id"]), seq, np.uint32)); oc.append(np.full(len(f["id"]), c, np.uint32))
            op.append(f["index"].astype(np.uint32)); oxy.append(f["xy"])
    assert np.array_equal(np.concatenate(oi), sp.problem.obs_imageset)
    assert np.array_equal(np.concatenate(oc), sp.problem.obs_camera)
    assert np.array_equal(np.concatenate(op), sp.problem.obs_point)
    assert np.array_equal(np.concatenate(oxy), sp.problem.obs_xy)
    assert st.intrinsics[0].update_parameter_count() == sp.problem.cameras[0].update_parameter_count()
    assert api.CameraModel.IsCentral(api.CameraModel.Type.CentralGeneric)
    assert not api.CameraModel.IsCentral(api.CameraModel.Type.NoncentralGeneric)


def _gloo_worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from camera_calibration_b200 import distributed
    from oracle import oracle
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sp = synthetic.make_problem(2, n_imagesets=8, lattice=(8, 6), image_size=(300, 220))
    opt = cabi.default_options()
    shard, idx = distributed.shard_problem(sp.problem, rank, world)
    st = distributed.shard_state(sp.init_state, idx)
    H, b, c = oracle.build_system(shard, st, opt)
    t = torch.from_numpy(np.concatenate([H.reshape(-1), b, [c]]))
    dist.all_reduce(t)  # what the NCCL all-reduce of the partial normal equations computes
    if rank == 0:
        Hf, bf, cf = oracle.build_system(sp.problem, sp.init_state, opt)
        full = np.concatenate([Hf.reshape(-1), bf, [cf]])
        q.put(float(np.abs(t.numpy() - full).max() / np.abs(full).max()))
    dist.destroy_process_group()


def test_sharded_partial_systems_allreduce_to_full_gloo():
    """world_size-2 gloo run of the N>1 host logic: imageset sharding + sum-all-reduce of the
    per-rank partial H, b, cost equals the single-rank system (oracle as the per-rank evaluator)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 300
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    err = q.get(timeout=300)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert err < 1e-12
