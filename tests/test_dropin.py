"""The drop-in surface of INTEGRATION.md section 1.

CPU: with ``buffer-x_b200`` and the repository root ahead of a reference checkout on ``sys.path``, the module names the
reference's ``test.py`` imports (:9-22) resolve as documented -- ``models.*`` to this package's mirrors (a regular package
beats the reference's namespace package ``models/``), ``utils.*``, ``dataset.*`` and ``config`` to the REFERENCE (its
``config`` is a regular package in the script directory, which precedes PYTHONPATH; its ``utils`` is a namespace package
without ``__init__.py``, so a regular ``utils`` package of ours would hide ``utils.timer`` etc. -- the round-1 defect).
GPU: the model exactly as ``test.py`` drives it -- ``nn.DataParallel(model, [0])``, ``model.eval()``, ``torch.no_grad()``,
the collate-shaped dict of CPU tensors (dataset/dataloader.py:108-122), NumPy's global RNG for the permutations,
``torch.cuda.empty_cache()`` between pairs, a new (Ns, Nt) for every pair -- against the oracle, eager and in graph mode
(12 shapes > the 8 cached graph shapes, so the LRU eviction runs).
"""
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fake_reference(tmp_path):
    """A directory tree shaped like the reference checkout (names only, no reference code)."""
    ref = tmp_path / "BUFFER-X"
    for d, files in {"utils": ["timer.py", "gpu_timer.py", "SE3.py", "tools.py", "result_io.py", "test_args.py", "progress_format.py", "common.py"],
                     "models": ["BUFFERX.py", "patch_embedder.py", "patchnet.py", "pose_estimator.py"],
                     "dataset": ["dataloader.py"]}.items():
        (ref / d).mkdir(parents=True)
        for f in files:
            (ref / d / f).write_text(f"ORIGIN = 'reference:{d}/{f}'\n")
    (ref / "config").mkdir()
    (ref / "config" / "__init__.py").write_text("ORIGIN = 'reference:config'\n")
    return ref


def test_documented_pythonpath_resolves_reference_and_mirror_modules(tmp_path):
    ref = _fake_reference(tmp_path)
    code = textwrap.dedent("""
        import importlib.util as u, json, os
        names = ["utils.timer", "utils.gpu_timer", "utils.SE3", "utils.tools", "utils.result_io", "utils.test_args",
                 "utils.progress_format", "dataset.dataloader", "models.BUFFERX", "models.patchnet", "models.patch_embedder",
                 "models.pose_estimator", "config"]
        out = {}
        for n in names:
            s = u.find_spec(n)
            out[n] = None if s is None else os.path.realpath(s.origin)
        print(json.dumps(out))
    """)
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "buffer-x_b200"), ROOT])      # as documented, then the checkout = cwd
    out = subprocess.run([sys.executable, "-c", code], cwd=str(ref), env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    import json
    res = json.loads(out.stdout.strip().splitlines()[-1])
    ours = os.path.realpath(os.path.join(ROOT, "buffer-x_b200"))
    for n in ("utils.timer", "utils.gpu_timer", "utils.SE3", "utils.tools", "utils.result_io", "utils.test_args", "utils.progress_format",
              "dataset.dataloader", "config"):
        assert res[n] is not None and res[n].startswith(os.path.realpath(str(ref))), f"{n} must come from the reference checkout, got {res[n]}"
    for n in ("models.BUFFERX", "models.patchnet", "models.patch_embedder", "models.pose_estimator"):
        assert res[n] is not None and res[n].startswith(ours), f"{n} must resolve to the B200 mirror, got {res[n]}"


def test_real_reference_checkout_utils_are_not_shadowed(tmp_path):
    """The same resolution in a tree with every Python file of the real reference checkout, by name
    (tests/golden/reference_layout.json, written by tests/tools/gen_reference_golden.py), none of its code."""
    ref = tmp_path / "BUFFER-X"
    for rel in json.load(open(os.path.join(ROOT, "tests", "golden", "reference_layout.json"))):
        (ref / rel).parent.mkdir(parents=True, exist_ok=True)
        (ref / rel).write_text(f"ORIGIN = 'reference:{rel}'\n")
    code = ("import importlib.util as u, os; "
            "print([os.path.realpath(u.find_spec(n).origin) for n in ('utils.timer','utils.SE3','utils.tools','models.BUFFERX')])")
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "buffer-x_b200"), ROOT])
    out = subprocess.run([sys.executable, "-c", code], cwd=str(ref), env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    paths = eval(out.stdout.strip().splitlines()[-1])
    utils = os.path.join(os.path.realpath(str(ref)), "utils") + os.sep
    assert all(p.startswith(utils) for p in paths[:3]) and paths[3].startswith(os.path.realpath(ROOT))


# ------------------------------------------------------------------------------------------------ GPU
def _collate_dict(d):
    """dataset/dataloader.py:108-122 ``collate_fn_descriptor``: CPU tensors + python scalars / strings."""
    return {"src_fds_pcd": torch.from_numpy(d["src_fds_pcd"]), "tgt_fds_pcd": torch.from_numpy(d["tgt_fds_pcd"]),
            "relt_pose": torch.from_numpy(d["relt_pose"]), "src_id": d["src_id"], "tgt_id": d["tgt_id"], "scene_name": d["scene_name"],
            "sensor": d["sensor"], "voxel_sizes": torch.from_numpy(d["voxel_sizes"]), "dataset_names": list(d["dataset_names"]),
            "sphericity": torch.from_numpy(d["sphericity"]), "is_aligned_to_global_z": d["is_aligned_to_global_z"]}


@pytest.mark.gpu
def test_dataparallel_loop_like_test_py_against_oracle(oracle):
    import bufferx_b200 as bx
    from bufferx_b200.se3 import compute_rre, compute_rte
    from bufferx_b200.synth import init_synthetic_weights, make_pair, workload_cfg
    assert torch.cuda.is_available()
    dev = torch.device("cuda:0")
    cfg = workload_cfg("C2")
    cfg.patch.num_fps, cfg.patch.num_points_radius_estimate, cfg.match.iter_n = 384, 512, 5000
    base = init_synthetic_weights(bx.BufferX(cfg), trained_pose=True)
    sd = {k: v.detach().clone() for k, v in base.state_dict().items()}
    base = base.to(dev)
    model = torch.nn.DataParallel(base, device_ids=[0])          # test.py:105
    model.eval()
    rng = np.random.default_rng(7)
    shapes = [(int(rng.integers(4200, 6000)), int(rng.integers(4200, 6000))) for _ in range(12)]
    assert len(set(shapes)) == 12
    pairs = [make_pair("C1", 20 + i, n_src=a, n_tgt=b) for i, (a, b) in enumerate(shapes)]
    expect = []
    for i, d in enumerate(pairs):
        perms = oracle.draw_perms(cfg, len(d["src_fds_pcd"]), len(d["tgt_fds_pcd"]), 100 + i)
        expect.append(oracle.register_pair(sd, cfg, d, perms, 0))
    for graphs in (False, True):
        base.enable_cuda_graphs(graphs, slots_per_shape=1)
        for i, d in enumerate(pairs):
            np.random.seed(100 + i)                              # the reference's host permutations come from the global RNG
            with torch.no_grad():
                pose, times, ninl, nmut, nind, su = model(_collate_dict(d))
            torch.cuda.empty_cache()                             # test.py:192
            o_pose, o_ninl, o_nmut, o_nind, o_su, _ = expect[i]
            assert isinstance(pose, np.ndarray) and pose.shape == (4, 4) and len(times) == 3
            assert (nmut, nind, ninl, su) == (o_nmut, o_nind, o_ninl, o_su), f"pair {i} graphs={graphs}: counts {(nmut, nind, ninl)} vs {(o_nmut, o_nind, o_ninl)}"
            if ninl >= 3:
                assert compute_rre(pose, o_pose) < 0.1 and compute_rte(pose, o_pose) < 0.005
            else:
                assert np.allclose(pose, o_pose, atol=1e-5)
        if graphs:
            assert len(base._slots) <= base.MAX_GRAPH_SHAPES
    base.enable_cuda_graphs(False)


@pytest.mark.gpu
def test_load_state_dict_and_to_drop_captured_graphs(oracle):
    """ADVICE r1: captured graphs bake in weight pointers; load_state_dict()/.to() must drop them (and results must follow
    the NEW weights)."""
    import bufferx_b200 as bx
    from bufferx_b200.synth import init_synthetic_weights, make_pair, workload_cfg
    dev = torch.device("cuda:0")
    cfg = workload_cfg("C1")
    a = init_synthetic_weights(bx.BufferX(cfg), seed=123).to(dev)
    b = init_synthetic_weights(bx.BufferX(cfg), seed=321)
    d = make_pair("C1", 3)
    perms = oracle.draw_perms(cfg, 5000, 5000, 3)
    with torch.no_grad():
        eager_b = b.to(dev)(d, perms=perms)
        a.enable_cuda_graphs(True, slots_per_shape=1)
        out_a = a(d, perms=perms)
        assert len(a._slots) == 1
        a.load_state_dict(b.state_dict())
        assert len(a._slots) == 0
        out_ab = a(d, perms=perms)
    assert out_ab[2:] == eager_b[2:] and np.array_equal(out_ab[0], eager_b[0])
    assert out_a[3] != out_ab[3] or not np.array_equal(out_a[0], out_ab[0])
    a.enable_cuda_graphs(False)


@pytest.mark.gpu
def test_fp16_range_flag_reruns_the_pair_on_the_tf32_kernel(oracle):
    """The shifted-descriptor conv kernel's sticky fp16-range flag rides in the pair's result block: when it is set, forward()
    (eager and graph mode) recomputes the pair on the TF32 tensor-core kernel, keeps the model on it and clears the flag --
    same counts, pose within rounding of the fp16-split path."""
    import bufferx_b200 as bx
    from bufferx_b200.se3 import compute_rre, compute_rte
    from bufferx_b200.synth import init_synthetic_weights, make_pair, workload_cfg
    dev = torch.device("cuda:0")
    cfg = workload_cfg("C2")
    cfg.patch.num_fps, cfg.patch.num_points_radius_estimate, cfg.match.iter_n = 384, 512, 5000
    d = make_pair("C1", 31)
    perms = oracle.draw_perms(cfg, 5000, 5000, 31)
    for graphs in (False, True):
        model = init_synthetic_weights(bx.BufferX(cfg), trained_pose=True).to(dev)
        model.enable_cuda_graphs(graphs, slots_per_shape=1)
        with torch.no_grad():
            ref = model(d, perms=perms)
            assert not model.Desc.conv_net.force_tf32
            model.Desc.conv_net.overflow_flag(dev).fill_(1)          # as if an activation had left fp16 range
            out = model(d, perms=perms)
            assert model.Desc.conv_net.force_tf32 and model.Pose.conv.force_tf32
            assert int(model.Desc.conv_net.overflow_flag(dev).item()) == 0
            again = model(d, perms=perms)                            # stays on the TF32 kernel, no rerun needed
        assert out[2:] == again[2:] and np.array_equal(out[0], again[0])
        assert out[3] == ref[3] and abs(out[2] - ref[2]) <= 1 and out[4] == ref[4]
        if ref[2] >= 3:
            assert compute_rre(out[0], ref[0]) < 0.5 and compute_rte(out[0], ref[0]) < 0.01
        model.enable_cuda_graphs(False)


@pytest.mark.gpu
def test_inputs_produced_on_another_stream_are_ordered(oracle):
    """ADVICE r1: forward_async copies CUDA inputs on the slot stream; it must wait for the producer stream."""
    import bufferx_b200 as bx
    from bufferx_b200.synth import init_synthetic_weights, make_pair, workload_cfg
    dev = torch.device("cuda:0")
    cfg = workload_cfg("C1")
    model = init_synthetic_weights(bx.BufferX(cfg)).to(dev)
    d = make_pair("C1", 4)
    perms = oracle.draw_perms(cfg, 5000, 5000, 4)
    with torch.no_grad():
        ref = model(d, perms=perms)
        model.enable_cuda_graphs(True, slots_per_shape=1)
        src_h = torch.from_numpy(d["src_fds_pcd"]).pin_memory()
        tgt_h = torch.from_numpy(d["tgt_fds_pcd"]).pin_memory()
        burn = torch.empty(64 * 1024 * 1024, device=dev)
        for _ in range(3):
            for _ in range(20):
                burn.normal_()                                   # keep the producer stream busy before the H2D copies
            g = dict(d)
            g["src_fds_pcd"] = src_h.to(dev, non_blocking=True)
            g["tgt_fds_pcd"] = tgt_h.to(dev, non_blocking=True)
            out = model.forward_async(g, perms=perms).result()
            del g
            assert out[2:] == ref[2:] and np.array_equal(out[0], ref[0])
    model.enable_cuda_graphs(False)


@pytest.mark.gpu
def test_radius_neighbors_beyond_the_shared_memory_sort(oracle):
    """Balls with more than 4096 neighbours (round 1: hard failure) take the global rank-sort path: same rows as the oracle,
    including the exact-tie order (duplicated supports), next to small balls in the same call."""
    from bufferx_b200 import ops
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(2)
    dense = (rng.random((6000, 3)) * 0.02).astype(np.float32)
    dense[3000:3500] = dense[:500]                                   # exact distance ties
    sparse = (rng.random((3000, 3)) * 5 + 1).astype(np.float32)
    sup = np.concatenate([dense, sparse]).astype(np.float32)
    qry = np.concatenate([dense[:5], sparse[:40]]).astype(np.float32)
    with torch.cuda.device(dev):
        got = ops.radius_neighbors(torch.from_numpy(qry).to(dev), torch.from_numpy(sup).to(dev), [len(qry)], [len(sup)], 0.5).cpu().numpy()
    exp = oracle.radius_neighbors(qry, sup, [len(qry)], [len(sup)], 0.5)
    assert got.shape == exp.shape and got.shape[1] >= 6000 and (got == exp).all()
