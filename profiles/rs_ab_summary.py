"""Summary of profiles/rs_ab.sh: headline value, k_rs_score kernel time and the C1 / C3 / C4 values of every
run of both sides, and whether the two sides' --dump-outputs files are byte-identical.

    python profiles/rs_ab_summary.py OUT_DIR TAG RUNS
"""
import glob
import json
import os
import sys

out, tag, runs = sys.argv[1], sys.argv[2], int(sys.argv[3])


def row(path):
    d = json.loads(open(path).read().strip().splitlines()[-1])
    k = {r["kernel"]: r["us_per_launch"] for r in d["kernels"]}
    c = d.get("configs") or {}
    return {"value": d["value"], "us_per_scan": round(d["ms_per_step"] * 1e3 / d["config"]["frames_per_step_per_gpu"], 2),
            "p50_latency_ms": d["p50_latency_ms"], "k_rs_score_us": k.get("k_rs_score"),
            "sm_mhz": d["clocks"].get("sm_mhz"),
            **{f"{n}_value": c[n]["value"] for n in ("C1", "C3", "C4") if n in c},
            "C1_k_rs_score_us": next((r["us_per_launch"] for r in c.get("C1", {}).get("kernels", [])
                                      if r["kernel"] == "k_rs_score"), None)}


res = {"gpu": open(os.path.join(out, f"{tag}_gpu.txt")).read().strip(), "order": "parent, new, parent, new, ..."}
for side in ("parent", "new"):
    res[side] = [row(os.path.join(out, f"{tag}_{side}_{i}.json")) for i in range(1, runs + 1)]
for side in ("parent", "new"):
    v = [r["value"] for r in res[side]]
    res[f"{side}_value_mean"] = round(sum(v) / len(v), 1)
res["gain_pct"] = round(100 * (res["new_value_mean"] / res["parent_value_mean"] - 1), 2)
res["every_new_beats_every_parent"] = min(r["value"] for r in res["new"]) > max(r["value"] for r in res["parent"])
files = sorted(os.path.basename(f) for f in glob.glob(os.path.join(out, f"{tag}_dump_parent", "*.npy")))
same = [f for f in files
        if open(os.path.join(out, f"{tag}_dump_parent", f), "rb").read() == open(os.path.join(out, f"{tag}_dump_new", f), "rb").read()]
res["dump_outputs"] = {"files": len(files), "byte_identical": len(same), "differ": sorted(set(files) - set(same))}
print(json.dumps(res, indent=1))
