"""bjj_keyset_create and the existing key-set benchmarks on another tree (the parent commit, built) and on this one, in
alternating processes on one GPU: does the growable table allocation of bjj_keyset_create cost anything?

    python babyjubjub-rs_b200/tools/ab_keyset_update.py --other TREE --out DIR [--rounds 2] [--create-rounds 6]
                                                        [--creates 5] [--keys 65536] [--into FILE]

1. Create: per process, K seeded keys, then `creates` x (bjj_keyset_create of the K keys, host clock around the
   synchronous call; bjj_keyset_destroy, timed too).  Processes alternate other / this `create-rounds` times, so each
   tree's first create in a process follows the other tree's process exit.
2. tools/bench_verify_keyset.py and tools/bench_verify_keyset_lookup.py with --keys K, each tree's own copy, alternating
   other / this `rounds` times; their verify rates and create times are collected.
Writes DIR/keyset_update_ab.json; with --into, also merges it into that keyset_update.json (bench_keyset_update.py's).
"""
import argparse
import ctypes
import glob
import json
import os
import subprocess
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)


def time_creates(root, keys, creates):
    """in this process, with the package of tree `root`: `creates` timed create / destroy pairs of `keys` keys"""
    sys.path.insert(0, root)
    import numpy as np
    import babyjubjub_rs_b200 as bjj
    eng = bjj.Engine(0)
    lib, ctx = eng.lib, eng.ctx
    priv = np.random.default_rng(5).integers(0, 256, size=(keys, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)

    def p(a):
        return a.ctypes.data_as(ctypes.c_void_p)
    out = {"create_s": [], "destroy_s": []}
    for _ in range(creates):
        h = ctypes.c_void_p()
        t0 = time.perf_counter()
        rc = lib.bjj_keyset_create(ctx, keys, p(ax), p(ay), None, ctypes.byref(h))
        out["create_s"].append(round(time.perf_counter() - t0, 4))
        if rc != 0:
            raise RuntimeError("bjj_keyset_create failed: %d" % rc)
        t0 = time.perf_counter()
        lib.bjj_keyset_destroy(ctx, h)
        out["destroy_s"].append(round(time.perf_counter() - t0, 4))
    return out


def run(cmd, cwd):
    p = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("%s failed in %s:\n%s" % (" ".join(cmd), cwd, p.stdout[-2000:] + p.stderr[-2000:]))
    return p.stdout


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--other", help="root of the other tree, built")
    ap.add_argument("--out", help="directory for keyset_update_ab.json")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--create-rounds", type=int, default=6)
    ap.add_argument("--creates", type=int, default=5)
    ap.add_argument("--keys", type=int, default=65536)
    ap.add_argument("--into", help="a keyset_update.json to merge the results into")
    ap.add_argument("--time-creates", metavar="TREE", help=argparse.SUPPRESS)   # the child process of part 1
    args = ap.parse_args()
    if args.time_creates:
        print(json.dumps(time_creates(args.time_creates, args.keys, args.creates)))
        return
    if not args.other or not args.out:
        raise SystemExit("--other and --out are required")
    from bench_verify_base import card_info
    trees = {"other": os.path.abspath(args.other), "this": ROOT}
    report = {"tool": "babyjubjub-rs_b200/tools/ab_keyset_update.py", "card": card_info(0), "keys": args.keys,
              "create": [], "existing_benchmarks": []}
    for _ in range(args.create_rounds):
        for name, tree in trees.items():
            res = json.loads(run([sys.executable, os.path.abspath(__file__), "--time-creates", tree, "--keys", str(args.keys),
                                  "--creates", str(args.creates)], tree).strip().splitlines()[-1])
            report["create"].append({"tree": name, **res})
            print(json.dumps(report["create"][-1]), flush=True)
    for rnd in range(args.rounds):
        for name, tree in trees.items():
            row = {"tree": name, "round": rnd + 1}
            with tempfile.TemporaryDirectory() as tmp:
                run([sys.executable, "babyjubjub-rs_b200/tools/bench_verify_keyset.py", "--out", tmp + "/vk", "--keys",
                     str(args.keys)], tree)
                run([sys.executable, "babyjubjub-rs_b200/tools/bench_verify_keyset_lookup.py", "--out", tmp + "/vkl",
                     "--keys", str(args.keys)], tree)
                vk = json.load(open(glob.glob(tmp + "/vk/*.json")[0]))["key_sets"][-1]
                vkl = json.load(open(glob.glob(tmp + "/vkl/*.json")[0]))["key_sets"][-1]
            row.update({
                "verify_keyset_batch_dev_M_per_s": vk["device_resident"]["verify_keyset_batch_dev"]["M_per_s_mean"],
                "verify_keyset_batch_M_per_s": vk["end_to_end_pinned"]["verify_keyset_batch"]["M_per_s_mean"],
                "verify_keyset_tool_create_s": vk["keyset_create_s"],
                "lookup_verify_dev_M_per_s": vkl["device_resident"]["verify_keyset_lookup_compressed_batch_dev"]["M_per_s_mean"],
                "lookup_verify_M_per_s": vkl["end_to_end_pinned"]["verify_keyset_lookup_compressed_batch"]["M_per_s_mean"],
                "lookup_tool_create_s": vkl["keyset_create_s"]})
            report["existing_benchmarks"].append(row)
            print(json.dumps(row), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "keyset_update_ab.json"), "w") as f:
        json.dump(report, f, indent=1)
    if args.into:
        merged = json.load(open(args.into))
        merged["ab_against_parent"] = report
        with open(args.into, "w") as f:
            json.dump(merged, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
