"""Views per second with a keep mask against no mask, at the same eliminated count.

    python tools/keep_throughput.py [--views 128] [--steps 5] [--rounds 3] [--frac 0.5] [--o_v degree] [--o_n asc]

Arxiv-shaped BA graph (n = 169,343, m = 7). The masked arm protects a seeded `frac` of the vertices and removes every
unprotected one (t = number of unprotected vertices); the unmasked arm removes the same t. Each step is one
schur_views call (elimination + emission to packed rows, device resident) ending in a device synchronise; the two
arms alternate `rounds` times and each round times `steps` steps after one warm-up step. Prints one JSON line with the
card's name and power limit beside the numbers, and the last step's rows, rounds, largest star, fills and
k_eliminate time per arm.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _card():
    import torch
    info = {"gpu": torch.cuda.get_device_name()}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception as ex:  # pragma: no cover
        info["power_limit_w"] = f"unavailable: {type(ex).__name__}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=128)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frac", type=float, default=0.5)
    ap.add_argument("--o_v", default="degree")
    ap.add_argument("--o_n", default="asc")
    a = ap.parse_args()
    import numpy as np
    import torch
    import rlap_b200
    from rlap_b200 import graphs
    if not torch.cuda.is_available():
        raise RuntimeError("keep_throughput.py needs a CUDA device")
    n = 169343
    ei = torch.from_numpy(graphs.barabasi_albert(n, 7, seed=0)).cuda()
    g = rlap_b200.prepare(ei, None, n)
    keep = torch.from_numpy(np.random.default_rng(0).random(n) < a.frac).cuda()
    t = int((~keep).sum())
    arms = {"no_mask": None, "mask": keep}
    step = [0]

    def one(k):
        step[0] += 1
        out, vp, st = rlap_b200.schur_views(g, t, a.o_v, a.o_n, num_views=a.views, seed=1000 + step[0], dtype=None,
                                            keep=k, return_stats=True)
        torch.cuda.synchronize()
        return {"rows": int(vp[-1]), "rounds": st["rounds"], "max_star": st["max_star"], "fills": st["fills"],
                "elim_ms": st["elim_us"] / 1000.0}

    res = {name: [] for name in arms}
    last = {}
    for _ in range(a.rounds):
        for name, k in arms.items():
            one(k)
            t0 = time.perf_counter()
            for _ in range(a.steps):
                last[name] = one(k)
            res[name].append(a.views * a.steps / (time.perf_counter() - t0))
    out = {"shape": "arxiv BA n=169343 m=7", "o_v": a.o_v, "o_n": a.o_n, "views": a.views, "eliminated": t,
           "protected_frac": a.frac, **_card()}
    for name in arms:
        out[name + "_views_per_s"] = [round(x, 1) for x in res[name]]
        out[name + "_last_step"] = last[name]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
