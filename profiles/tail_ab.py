"""A/B of the training step's tail schedule inside one tree: alternates SN_TAIL_SCHEDULE=0 and =1 runs of
`bench.py --no-extras --no-cpu-baseline`, then checks that both arms' --dump-outputs are identical file for file.
Usage: python profiles/tail_ab.py OUT_DIR [runs per arm] [extra arms as NAME=ENV=VALUE,...]"""
import json, os, statistics, subprocess, sys, tempfile
import numpy as np

out = sys.argv[1]
runs = int(sys.argv[2]) if len(sys.argv) > 2 else 5
arms = {"tail0": {"SN_TAIL_SCHEDULE": "0"}, "tail1": {"SN_TAIL_SCHEDULE": "1"}}
for spec in (sys.argv[3].split(",") if len(sys.argv) > 3 and sys.argv[3] else []):
    name, kv = spec.split(":", 1)
    arms[name] = dict(SN_TAIL_SCHEDULE="1", **dict(x.split("=", 1) for x in kv.split(";")))
os.makedirs(out, exist_ok=True)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
res = {a: [] for a in arms}
with open(os.path.join(out, "tail_ab_runs.jsonl"), "w") as f:
    for i in range(runs):
        for a, env in arms.items():
            p = subprocess.run([sys.executable, "bench.py", "--no-extras", "--no-cpu-baseline"], capture_output=True,
                               text=True, env=dict(os.environ, **env))
            line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
            d = json.loads(line)
            res[a].append(d["ms_per_step"])
            f.write(json.dumps({"arm": a, "env": env, "run": i, "ms_per_step": d["ms_per_step"],
                                "clocks": d.get("clocks"), "gpu": gpu}) + "\n")
            f.flush()
summary = {"gpu": gpu, "runs_per_arm": runs}
for a, v in res.items():
    summary[a] = {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v}
dumps = {}
with tempfile.TemporaryDirectory() as td:
    for a in ("tail0", "tail1"):
        d = os.path.join(td, a)
        subprocess.run([sys.executable, "bench.py", "--no-extras", "--no-cpu-baseline", "--steps", "5",
                        "--dump-outputs", d], capture_output=True, text=True, check=True,
                       env=dict(os.environ, **arms[a]))
        dumps[a] = {n: np.load(os.path.join(d, n)) for n in sorted(os.listdir(d)) if n.endswith(".npy")}
    same = sorted(dumps["tail0"]) == sorted(dumps["tail1"]) and all(
        np.array_equal(dumps["tail0"][n], dumps["tail1"][n]) for n in dumps["tail0"])
summary["dump_outputs_identical"] = bool(same)
summary["dump_outputs_files"] = len(dumps["tail0"])
print(json.dumps(summary))
with open(os.path.join(out, "tail_ab_summary.json"), "w") as f:
    json.dump(summary, f, indent=1)
