"""Record the configuration the contraction kernel selects for every ops.gemm launch of the production plans.

    python tools/gemm_launch_configs.py [--out tests/golden/gemm_launch_configs.json]

Runs each plan of tests/gemm_plan_walk.py (UNet at 48x156 for B = 1..8 and at 96x312 for B = 2, the LayerNorm-fold and
learnable-descriptor plans at B = 8, the seg-AE decoder and the RGB VAE encoder at B = 8) once, without numerics, and
writes one line per plan: the selection of every launch in launch order, coded by gemm_plan_walk.config_code (epilogue
instantiation the profiler saw, block_n, CTA pair, split-K factor). tests/test_gemm_plan_launches_gpu.py compares the
live selection against this file on a 148-SM B200, so a change of the cost model shows in its own diff which plans'
launches moved, and the test's failure names each moved launch with its descriptor."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import gemm_plan_walk as W  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "gemm_launch_configs.json"))
    args = ap.parse_args()
    props = torch.cuda.get_device_properties(0)
    if props.multi_processor_count != 148:
        print(f"warning: {props.name} has {props.multi_processor_count} SMs; the pinned file is for a 148-SM B200")
    out = {}
    for plan, builder in W.plan_walks():
        out[plan] = " ".join(W.config_code(r) for r in W.config_walk(builder))
        print(f"{plan}: {len(out[plan].split())} launches")
    with open(args.out, "w") as f:
        f.write("{\n" + ",\n".join(f"  {json.dumps(p)}: {json.dumps(codes)}" for p, codes in out.items()) + "\n}\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
