"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares (no compute without a GPU), the
synthetic reference generator mirrors the reference's gait / swing-spline rules, and the N>1 sharding + gather logic works
with world_size 2 over gloo."""
import ctypes as C
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HUNTER_CONFIG = os.path.join(ROOT, "tests", "golden", "hunter")        # hunter.urdf, task.info, reference.info of the original project


def test_abi_exports_every_declared_symbol():
    import hunter_bipedal_control_b200 as hb
    lib = hb.load_library()
    hdr = open(os.path.join(ROOT, "include", "hunter_b200.h")).read()
    names = set(re.findall(r"\b(hb_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), n
    assert names == set(hb.EXPORTED_SYMBOLS)


def test_abi_config_and_error_strings():
    import hunter_bipedal_control_b200 as hb
    lib = hb.load_library()
    cfg = hb.HbConfig()
    assert lib.hb_default_config(C.byref(cfg)) == 0
    assert cfg.horizon_N == 100 and abs(cfg.dt - 0.01) < 1e-15 and cfg.wbc_rho == 1e-8
    assert lib.hb_default_config(None) < 0
    assert lib.hb_strerror(0) == b"ok" and b"invalid" in lib.hb_strerror(-1)
    assert C.sizeof(hb.HbSolveInfo) == 56
    # misuse never crashes: null context
    assert lib.hb_sync(None) < 0 and lib.hb_destroy(None) < 0


def test_no_cpu_fallback_without_gpu():
    """The product path fails loudly when no B200 is visible (this container has none)."""
    import torch
    import hunter_bipedal_control_b200 as hb
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(hb.HunterB200Error):
        hb.Context(max_batch=1)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "hunter_bipedal_control_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                s = open(os.path.join(dp, f)).read()
                assert "oracle" not in s.lower().replace("the oracle", "").replace("cpu oracle", "") or f == "__init__.py" or "import" not in s, f
                assert not re.search(r"^\s*(from|import)\s+oracle", s, re.M), f
                assert "hb_oracle" not in s and "libhb_oracle" not in s, f


def test_gait_schedule_and_swing_splines():
    from hunter_bipedal_control_b200 import scenarios as S
    N, dt = 100, 0.01
    x0 = S.INITIAL_STATE.copy()
    x_ref, swing, mode, c = S.make_reference(x0, (0.2, 0, 0, 0), "trot", N, dt)
    # 0.1 s transition stance, then L 0.3 s / R 0.3 s (reference.info:67-80, task.info:11)
    assert (mode[:10] == 3).all() and (mode[10:40] == 2).all() and (mode[40:70] == 1).all() and (mode[70:100] == 2).all()
    sw = swing.reshape(N + 1, 4, 6)
    # stance feet: z reference = 0.02, zero velocity; swing feet lift to <= 0.02 + swingHeight and land at 0.02
    for k in range(N + 1):
        fl = S.mode_flags(int(mode[k]))
        for cc in range(4):
            if fl[cc]:
                assert abs(sw[k, cc, 2] - 0.02) < 1e-12 and np.abs(sw[k, cc, 3:]).max() < 1e-12
            else:
                assert 0.02 - 1e-9 <= sw[k, cc, 2] <= 0.02 + 0.04 + 1e-9
    # spline continuity across segments
    for cc in range(4):
        for a in range(3):
            segs = c["segments"][cc][a]
            for s0, s1 in zip(segs[:-1], segs[1:]):
                assert abs(s0[1] - s1[0]) < 1e-12 and abs(s0[4] - s1[2]) < 1e-12 and abs(s0[5] - s1[3]) < 1e-12
    # swing apex constants of genSwingTrajs (SwingTrajectoryPlanner.cpp:331-346)
    zsegs = [s for s in c["segments"][1][2] if abs(s[3]) + abs(s[5]) > 0]
    assert abs(zsegs[0][4] - 0.749 * 0.06) < 1e-12
    for g in ("stance", "standing_trot", "flying_trot"):
        _, _, md, _ = S.make_reference(x0, (0, 0, 0, 0), g, N, dt)
        assert set(md.tolist()) <= {0, 1, 2, 3}
    assert (S.make_reference(x0, (0, 0, 0, 0), "stance", N, dt)[2] == 3).all()
    assert 0 in S.make_reference(x0, (0, 0, 0, 0), "flying_trot", N, dt)[2]


def test_partition_and_sort():
    from hunter_bipedal_control_b200 import sharding as sh
    for total in (0, 1, 7, 8, 65536):
        for ws in (1, 2, 4, 8):
            blocks = [sh.partition(total, ws, r) for r in range(ws)]
            assert blocks[0][0] == 0 and blocks[-1][1] == total
            assert all(b[1] == n[0] for b, n in zip(blocks[:-1], blocks[1:]))
            assert max(b[1] - b[0] for b in blocks) - min(b[1] - b[0] for b in blocks) <= 1
    mode = np.array([[3, 2], [2, 2], [3, 2], [1, 1]])
    perm, inv = sh.sort_by_schedule(mode)
    assert (mode[perm][inv] == mode).all()
    assert [tuple(m) for m in mode[perm]] == sorted(tuple(m) for m in mode)


WORKER = r"""
import os, sys
sys.path.insert(0, %r)
import torch, torch.distributed as dist
from hunter_bipedal_control_b200 import sharding as sh
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% sys.argv[1], rank=int(sys.argv[2]), world_size=2)
rank, total = dist.get_rank(), 7
lo, hi = sh.partition(total, 2, rank)
local = torch.arange(lo, hi, dtype=torch.float64)[:, None] * torch.ones(1, 10, dtype=torch.float64) + 0.5
out = sh.gather_to_rank0(local, total, 2, rank, dist)
if rank == 0:
    assert out.shape == (7, 10) and torch.equal(out[:, 0], torch.arange(7, dtype=torch.float64) + 0.5), out
    print("GATHER_OK")
dist.barrier()
dist.destroy_process_group()
"""


def test_gloo_world_size_2_gather(tmp_path):
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    procs = [subprocess.Popen([sys.executable, str(script), str(port), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "GATHER_OK" in outs[0]


def test_host_only_entry_points_reject_misuse():
    """The host-only calls of the ABI (no GPU needed) report misuse through their return code."""
    import ctypes as C
    import hunter_bipedal_control_b200 as hb
    lib = hb.load_library()
    assert lib.hb_plan_references(1, None, None, None) == -1
    assert lib.hb_gait_select(1, None, None, None, None, None, None) == -1
    assert lib.hb_kf_reset(1, None) == -1 and lib.hb_default_kf_params(None) == -1 and lib.hb_default_pd_gains(None) == -1
    assert lib.hb_plan_references(0, (hb.HbPlanInput * 1)(), (C.c_double * 12)(), (hb.HbReference * 1)()) == 0       # empty batch
    sel = hb.GaitSelector(1)
    sel.state[0].head = 77                                                                                           # corrupted ring-buffer index
    with pytest.raises(RuntimeError):
        sel.update([0.1, 0, 0, 0], np.zeros((1, 22)))
    st = hb.kf_states(3)
    assert st[2].P[0] == 100.0 and st[2].P[1] == 0.0 and st[2].P[19] == 100.0 and st[1].x_hat[5] == 0.0
    g = hb.default_pd_gains(); k = hb.default_kf_params()
    assert (g.kp_big_stance, g.kd_feet) == (40.0, 0.01) and (k.foot_radius, k.foot_sensor_noise_velocity) == (0.02, 0.1)
    assert b"capacity" in lib.hb_strerror(-5) or b"planner" in lib.hb_strerror(-5)


def test_task_info_parser_reads_the_wbc_estimator_and_solver_blocks():
    """hb_parse_task_info on a fixture in the layout of the reference's task.info (values changed on purpose): nested blocks, `(i,j) value`
    matrix entries, `;` comments, booleans; absent keys keep the shipped defaults."""
    import hunter_bipedal_control_b200 as hb
    ti = hb.parse_task_info(os.path.join(ROOT, "tests", "golden", "task_wbc_variant.info"))
    w = ti.wbc
    assert list(w.torque_limits) == [25.0, 55.0, 50.0, 58.0, 20.0]
    assert (w.friction_coefficient, w.swing_kp, w.swing_kd) == (0.55, 140.0, 15.0)
    assert (w.base_height_kp, w.base_height_kd, w.base_angular_kp, w.base_angular_kd) == (25.0, 3.5, 18.0, 2.5)
    assert (w.weight_swing_leg, w.weight_base_accel, w.weight_contact_force) == (80.0, 1.5, 0.02)
    assert list(ti.kalman) == [0.021, 0.03, 0.02, 0.5, 0.5, 0.1, 0.02]          # three keys present, four defaults (task.info:336-345)
    assert (ti.contact_force_cutoff_frequency, ti.contact_threshold) == (200.0, 70.0)
    assert (ti.sqp_dt, ti.sqp_iteration, ti.mpc_time_horizon, ti.mpc_cold_start) == (0.0125, 1, 0.75, 0)
    assert ti.found == 1 | 2 | 4 | 8 | 16
    lib = hb.load_library()
    import ctypes as C
    assert lib.hb_parse_task_info(b"/nonexistent/task.info", C.byref(hb.HbTaskInfo())) != 0
    d = hb.HbWbcSettings(); assert lib.hb_default_wbc_settings(C.byref(d)) == 0
    assert list(d.torque_limits) == [28.0, 60.0, 60.0, 60.0, 28.0] and (d.swing_kp, d.swing_kd, d.weight_swing_leg, d.weight_contact_force) == (160.0, 18.0, 100.0, 0.0)


def test_task_info_parser_on_the_reference_file_when_present():
    """The original project's shipped task.info (stored verbatim under tests/golden/hunter/): the values equal the compiled-in defaults."""
    import hunter_bipedal_control_b200 as hb
    ti = hb.parse_task_info(os.path.join(HUNTER_CONFIG, "task.info"))
    import ctypes as C
    d = hb.HbWbcSettings(); hb.load_library().hb_default_wbc_settings(C.byref(d))
    assert np.array_equal(ti.wbc.as_array(), d.as_array())
    assert ti.found == 31 and (ti.sqp_dt, ti.mpc_time_horizon, ti.contact_force_cutoff_frequency) == (0.015, 0.8, 250.0)
    assert list(ti.kalman) == [0.02, 0.02, 0.02, 0.5, 0.5, 0.1, 0.01]


def test_native_shard_helpers_match_python_mirror():
    """hb_shard_partition / hb_shard_sort_by_schedule (C ABI, host only) against sharding.partition / sort_by_schedule."""
    from hunter_bipedal_control_b200 import sharding
    for total in (0, 1, 7, 10, 1024, 65536):
        for w in (1, 2, 3, 8):
            blocks = [sharding.native_partition(total, w, r) for r in range(w)]
            assert blocks == [sharding.partition(total, w, r) for r in range(w)]
            assert blocks[0][0] == 0 and blocks[-1][1] == total and all(a[1] == b[0] for a, b in zip(blocks, blocks[1:]))
    rng = np.random.default_rng(0)
    mode = rng.integers(0, 4, (300, 6)).astype(np.int32)
    p, i = sharding.native_sort_by_schedule(mode)
    p2, i2 = sharding.sort_by_schedule(mode)
    assert np.array_equal(p, p2) and np.array_equal(i, i2)
    srt = mode[p]
    assert all(tuple(srt[k]) <= tuple(srt[k + 1]) for k in range(len(srt) - 1))


def test_model_constants_header_regenerates_from_the_reference_files_when_present(tmp_path):
    """include/hunter_model_constants.h (inertias, joint tree and limits from hunter.urdf; MPC / WBC weights and gains from task.info; default
    joint state and gait templates from reference.info) is generated, not written by hand: regenerating it from the original project's files
    (stored verbatim under tests/golden/hunter/, laid out here as in the original tree) gives the committed bytes."""
    ref = tmp_path / "reference"
    for name, rel in (("hunter.urdf", "legged_examples/legged_hunter/legged_hunter_description/urdf"), ("task.info", "legged_controllers/config/hunter"),
                      ("reference.info", "legged_controllers/config/hunter")):
        (ref / rel).mkdir(parents=True, exist_ok=True)
        shutil.copyfile(os.path.join(HUNTER_CONFIG, name), ref / rel / name)
    out = tmp_path / "hunter_model_constants.h"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_model.py"), ref, str(out)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    assert out.read_bytes() == open(os.path.join(ROOT, "include", "hunter_model_constants.h"), "rb").read()
