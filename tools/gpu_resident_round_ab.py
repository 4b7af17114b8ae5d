"""Resident-path round breakdown and an A/B of two builds at C5 (n = 1000, p = 500 000, screening to 5000 columns,
10-fold CV, s = 1..20).

  python tools/gpu_resident_round_ab.py --round ROOT
      one C5 call of the build in ROOT with the BESS_B200_TRACE time line on; prints one JSON line: per round of each
      chain group the sweep (sweeper 0), the hop to the owners (B1), the slowest owner phase and the hop back (B2)
  python tools/gpu_resident_round_ab.py --parent-tar TAR --out OUT.jsonl [--runs 3]
      TAR holds a tree `parent/` with its library built.  Alternates `bench.py --steps 50 --warmup 3 --no-c2` between
      the parent and this tree, compares their `--dump-outputs` byte for byte, records the round breakdown of both and the
      card (name, power limit, max SM clock), one JSON line per item.
"""
import argparse
import filecmp
import json
import os
import subprocess
import sys
import tarfile
import tempfile

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def round_breakdown(root):
    sys.path.insert(0, root)
    import numpy as np
    import torch
    fd, tr = tempfile.mkstemp(suffix=".txt")
    os.close(fd)
    os.environ["BESS_B200_TRACE"] = tr
    from bess_b200 import cbess
    n, p, k = 1000, 500000, 10
    gen = torch.Generator(device="cuda").manual_seed(5)
    X = torch.randn(n, p, dtype=torch.float64, device="cuda", generator=gen)
    rng = np.random.default_rng(5)
    nz = np.sort(rng.choice(p, k, replace=False))
    beta = rng.uniform(1, 5, k)
    y = (X[:, torch.as_tensor(nz, device="cuda")] @ torch.as_tensor(beta, device="cuda")).cpu().numpy() + rng.normal(0, 3, n)
    w = np.ones(n)
    seq = np.arange(1, 21)
    for _ in range(4):  # the last call's time line is kept
        out = cbess.fit(None, y, 1, w, True, 1, 1, 20, 2, 1, True, 1, True, 10, seq, 1, 20, True, 5000,
                        x_device_ptr=X.data_ptr(), n=n, p=p, want_trace=False)
    rows = np.loadtxt(tr, dtype=np.int64)
    os.unlink(tr)
    t0 = rows[:, 2][rows[:, 2] > 0].min()
    own, swp = {}, {}
    for c, q, a, b in rows:
        (swp if c == 32 else own.setdefault(int(c), {}))[int(q)] = ((a - t0) / 1e3, (b - t0) / 1e3)
    ng = 2
    rounds = []
    for it in range(1, 128):
        for g in range(ng):
            cs = [c for c in sorted(own) if c % ng == g and it in own[c]]
            st = ng * (it - 1) + g  # the sweeper step whose sacrifices this owner phase consumes
            if not cs or st not in swp or st + ng not in swp:
                continue
            durs = {c: own[c][it][1] - own[c][it][0] for c in cs}
            slow = max(durs, key=durs.get)
            first_start = min(own[c][it][0] for c in cs)
            last_end = max(own[c][it][1] for c in cs)
            busy_until = max(last_end, swp[st + ng - 1][1])  # the sweepers may still be on the other group's sweep
            rounds.append({"group": g, "round": it, "sweep_us": float(swp[st][1] - swp[st][0]),
                           "b1_hop_us": first_start - swp[st][1], "slowest_owner_us": durs[slow], "slowest_chain_pos": slow,
                           "owner_spread_us": last_end - first_start - durs[slow],
                           "b2_hop_us": swp[st + ng][0] - busy_until,
                           "sweeper_busy_elsewhere": bool(swp[st + ng - 1][1] > last_end),
                           "round_us": swp[st + ng][0] - swp[st][0]})
    med = {key: float(np.median([r[key] for r in rounds])) for key in
           ("sweep_us", "b1_hop_us", "slowest_owner_us", "owner_spread_us", "b2_hop_us", "round_us")}
    slow_count = {}
    for r in rounds:
        slow_count[r["slowest_chain_pos"]] = slow_count.get(r["slowest_chain_pos"], 0) + 1
    st = out["stats"]
    return {"rounds": len(rounds), "median": med,
            "launch_span_us": float(max(v[1] for d in own.values() for v in d.values())),
            "slowest_owner_by_chain_position": slow_count,
            "owner0_us_by_phase": None if "resident" not in st else list(map(float, st["resident"])),
            "per_round": rounds}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q


def bench(root, extra):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "50", "--warmup", "3", "--no-c2", *extra],
                       cwd=root, capture_output=True, text=True)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f"bench.py failed in {root}:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
    return json.loads(lines[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--round", metavar="ROOT")
    ap.add_argument("--parent-tar")
    ap.add_argument("--out")
    ap.add_argument("--runs", type=int, default=3)
    a = ap.parse_args()
    if a.round:
        print(json.dumps(round_breakdown(a.round)))
        return
    tmp = tempfile.mkdtemp()
    with tarfile.open(a.parent_tar) as t:
        t.extractall(tmp)
    arms = {"parent": os.path.join(tmp, "parent"), "new": HERE}
    def emit(rec):
        print(json.dumps(rec)[:2000], flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(json.dumps(rec) + "\n")

    emit({"item": "card", "card": card()})

    for name, root in arms.items():
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--round", root], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(r.stdout[-3000:] + r.stderr[-3000:])
        emit({"item": "round_breakdown", "arm": name, **json.loads(r.stdout.splitlines()[-1])})
    for run in range(1, a.runs + 1):
        for name, root in arms.items():
            o = bench(root, [])
            emit({"item": "bench", "arm": name, "run": run, "ms_per_step": o.get("ms_per_step"), "value": o.get("value"),
                  "kernel_ms_per_step": o.get("kernel_ms_per_step"), "resident_path": o.get("resident_path"),
                  "clocks": o.get("clocks")})
    dumps = {}
    for name, root in arms.items():
        dumps[name] = tempfile.mkdtemp()
        bench(root, ["--dump-outputs", dumps[name]])
    files = sorted(os.listdir(dumps["parent"]))
    same = files == sorted(os.listdir(dumps["new"])) and all(
        filecmp.cmp(os.path.join(dumps["parent"], f), os.path.join(dumps["new"], f), shallow=False) for f in files)
    emit({"item": "dump_outputs", "files": files, "byte_identical": same})
    emit({"item": "card_after", "card": card()})


if __name__ == "__main__":
    main()
