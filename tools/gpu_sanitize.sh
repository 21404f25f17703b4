#!/bin/bash
# compute-sanitizer (memcheck + racecheck) over a small rollout of every batched level, and an
# ncu summary of K1.  Logs -> gpurun_out/.
mkdir -p gpurun_out
cat > /tmp/san.py <<'PY'
import sys, numpy as np, torch
sys.path.insert(0, '.')
from miniworld_b200.batched import BatchedMiniWorld
from miniworld_b200.envs import LEVELS
LEVEL_KW = [("MiniWorld-FourRooms-v0", dict(want_depth=True)), ("MiniWorld-Hallway-v0", dict(domain_rand=True)),
            ("MiniWorld-MazeS3-v0", {}), ("MiniWorld-PickupObjects-v0", dict(obs_width=160, obs_height=120)),
            ("MiniWorld-OneRoom-v0", dict(msaa_samples=4)), ("MiniWorld-PutNext-v0", dict(domain_rand=True)),
            ("MiniWorld-CollectHealth-v0", {}), ("MiniWorld-Sign-v0", {}), ("MiniWorld-YMaze-v0", {}),
            ("MiniWorld-Sidewalk-v0", dict(obs_format="cwh")), ("MiniWorld-ThreeRooms-v0", dict(obs_format="grey"))]
# every level twice: with the stores K2 makes towards local memory, then with the whole-frame / band stage it uses
# towards a peer GPU (forced on through set_obs_peer)
for staged in (False, True):
    for level, kw in LEVEL_KW:
        env = BatchedMiniWorld(level, 48, **kw)
        if staged:
            env.engine.set_obs_peer(True)
        env.reset(seed=7)
        acts = torch.as_tensor(np.random.default_rng(1).choice([0, 1, 2, 2, 4], size=(12, 48)).astype(np.int32) % env.action_space.n, device="cuda")
        for t in range(12):
            obs, r, te, tr, _ = env.step(acts[t])
        top = env.render_top_view()
        vis = env.visible_ents()
        blob = env.snapshot()
        env.restore(blob)
        torch.cuda.synchronize()
        if isinstance(obs, dict):                 # Sign's dict observation
            obs = obs["obs"]
        print("staged" if staged else "local", level, float(obs.float().mean()), float(top.float().mean()), int(vis.sum()),
              env.engine.overflow_count())
        env.close()
e = LEVELS["MiniWorld-ThreeRooms-v0"](domain_rand=True)
e.reset(seed=1)
for t in range(6):
    e.step(t % 3)
print("threerooms", e.render_obs().mean(), e.render_top_view().mean(), len(e.get_visible_ents()))
PY
for tool in memcheck racecheck; do
  timeout 900 compute-sanitizer --tool $tool --print-limit 20 python /tmp/san.py > gpurun_out/sanitizer_$tool.log 2>&1; echo "$tool rc=$?"
  grep -E "ERROR SUMMARY|RACECHECK SUMMARY|Invalid|hazard" gpurun_out/sanitizer_$tool.log | head -8
done
if [ -n "$MWB_SANITIZE_EXTRAS" ]; then
timeout 600 ncu --set full --clock-control none -k regex:step_kernel -s 6 -c 1 -f -o gpurun_out/prof_k1 python bench.py --steps 3 --warmup 3 --no-cpu > gpurun_out/ncu_k1.log 2>&1; echo "ncu k1 rc=$?"
timeout 600 python tools/bench_configs.py > gpurun_out/configs.jsonl 2> gpurun_out/configs.err; cut -c1-330 gpurun_out/configs.jsonl
fi
