"""Fast A/B of library variants on one GPU: the scene is generated ONCE, every variant runs in its own process (BADBA_LIB)
on the pickled scene and reports step / stage / pose-kernel times plus a result fingerprint (residual counts, cost, pose
difference to the first variant) so that a faster but wrong variant is visible at once.

    python tools/ab_fast.py [--workload cfg3] [--steps 5] tools/ab/a.so tools/ab/b.so ...
"""
import json
import os
import pickle
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(scene_path, steps, ref_poses_path):
    import numpy as np
    import torch
    from badslam_b200.direct_ba import DirectBA
    from badslam_b200.scene import pose_error
    with open(scene_path, "rb") as f:
        scene = pickle.load(f)
    K = scene.cfg.num_keyframes
    ba = DirectBA.from_scene(scene)
    surf = ba.surfels()
    backup = surf[:8].clone()
    poses0, act0 = scene.poses_init.copy(), np.zeros(K, np.int32)
    ba.SetLastBAIterationCount(ba.ba_iteration_count())

    def step():
        surf[:8].copy_(backup, non_blocking=True)
        ba.SetKeyframeStates(poses0, act0)
        return ba.BundleAdjustment(None, False, False, False, True, True, 1, 1, increase_ba_iteration_count=False)

    for _ in range(3):
        res = step()
    torch.cuda.synchronize()
    ba.SetProfiling(1)
    ba.GetProfile(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage = np.zeros(3)
    e0.record()
    for _ in range(steps):
        res = step()
        stage += [res.ms_surfel_activation, res.ms_geometry_optimization, res.ms_pose_optimization]
    e1.record()
    torch.cuda.synchronize()
    prof = ba.GetProfile(reset=True)
    poses = ba.GetKeyframeStates()[0]
    out = {"ms_per_step": e0.elapsed_time(e1) / steps, "stage_ms": [round(float(v) / steps, 3) for v in stage],
           "pose_kernel_avg_ms": prof["pose_ms"] / max(prof["pose_launches"], 1), "pose_launches_per_step": prof["pose_launches"] / steps,
           "residuals": int(res.depth_residual_count + res.descriptor_residual_count), "cost": float(res.cost),
           "gn_iterations": int(res.pose_iterations_total)}
    if os.path.exists(ref_poses_path):
        ref = np.load(ref_poses_path)
        errs = [pose_error(poses[k], ref[k]) for k in range(K)]
        out["pose_diff_to_first"] = [float(max(e[0] for e in errs)), float(max(e[1] for e in errs))]
    else:
        np.save(ref_poses_path, poses)
    print("AB_RESULT " + json.dumps(out), flush=True)


def main():
    args = sys.argv[1:]
    if args and args[0] == "--child":
        return child(args[1], int(args[2]), args[3])
    workload, steps = "cfg3", 5
    libs = []
    while args:
        if args[0] == "--workload":
            workload = args[1]; args = args[2:]
        elif args[0] == "--steps":
            steps = int(args[1]); args = args[2:]
        else:
            libs.append(args[0]); args = args[1:]
    from badslam_b200.scene import config_by_name, make_scene
    t0 = time.time()
    scene = make_scene(config_by_name(workload))
    scene_path = f"/tmp/ab_scene_{workload}.pkl"
    with open(scene_path, "wb") as f:
        pickle.dump(scene, f, protocol=4)
    print(f"scene {workload} generated and pickled in {time.time() - t0:.1f} s", flush=True)
    ref_poses = f"/tmp/ab_poses_{workload}.npy"
    if os.path.exists(ref_poses):
        os.remove(ref_poses)
    for lib in ["in-tree"] + libs:
        env = dict(os.environ)
        if lib != "in-tree":
            env["BADBA_LIB"] = os.path.join(ROOT, lib)
        t0 = time.time()
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", scene_path, str(steps), ref_poses], env=env,
                           capture_output=True, text=True)
        line = [l for l in p.stdout.splitlines() if l.startswith("AB_RESULT ")]
        if not line:
            print(f"{lib}: FAILED rc={p.returncode} {p.stderr[-600:]}", flush=True)
            continue
        print(f"{os.path.basename(lib)} ({time.time() - t0:.0f} s): {line[-1][10:]}", flush=True)


if __name__ == "__main__":
    main()
