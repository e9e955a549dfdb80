"""What one delivery of the headline workload produces, counted from the CPU oracle's event traces (no GPU).

  python tools/delivery_mix.py [--seeds 4096] [--seed-base 1]

The headline kernel (fuzz_lane_kernel) runs 32 prefixes per warp in lock-step.  How much of its work each delivery
hands to the warp depends on how many messages a delivery produces and how unevenly they fall over the 32 lanes.
This script measures that mix for the bench workload (raft5, double-vote bug, depth 50, invariant every 5), so the
premise of the cooperative fan-out (DESIGN §10.1) can be re-checked when the model or the workload changes:

  - deliveries and trace events per prefix;
  - actor sends per delivery (receive()'s own sends) and flush items per delivery (timer / external sends recorded
    after it), as means and histograms;
  - the delivered message types;
  - per warp step (delivery i of 32 consecutive seeds): distinct delivered types, the largest per-lane item count
    (the trips of a per-lane loop) against the items spread over the lanes present (32-lane rounds).
"""
import argparse
import collections
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RAFT5_TYPES = {1: "BOOT", 2: "CLIENT_CMD", 3: "ELECTION_TICK", 4: "REQUEST_VOTE", 5: "VOTE_REPLY",
               6: "HEARTBEAT_TICK", 7: "APPEND_ENTRIES", 8: "APPEND_REPLY"}


def deliveries(ev):
    """[(delivered type, actor sends, flush items)] of one trace, in order: the sends recorded after a delivery and
    before the next one are its receive()'s sends (sender = the receiver) and then the flush before the next pick."""
    from demi_b200 import _native as N
    out = []
    for e in ev:
        if e["kind"] == N.EV_MSG_EVENT:
            out.append([int(e["type"]), 0, 0, int(e["dst"])])
        elif e["kind"] == N.EV_MSG_SEND and out:
            if e["src"] == out[-1][3]:
                out[-1][1] += 1
            else:
                out[-1][2] += 1
    return [(t, s, f) for t, s, f, _ in out]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=4096)
    ap.add_argument("--seed-base", type=int, default=1)
    args = ap.parse_args()
    import demi_b200 as D
    from demi_b200 import _native as N
    from oracle import binding as O
    ext = D.pack_externals(D.raft5_program())
    per_seed, n_events = [], 0
    for s in range(args.seeds):
        ev, _, res = O.fuzz_trace(N.MODEL_RAFT5, ext, args.seed_base + s, 50, 5, model_flags=1)
        n_events += len(ev)
        per_seed.append(deliveries(ev))
    flat = [d for seq in per_seed for d in seq]
    sends = np.array([d[1] for d in flat])
    flush = np.array([d[2] for d in flat])
    types = collections.Counter(RAFT5_TYPES.get(d[0], str(d[0])) for d in flat)

    steps = {"distinct_types": [], "lanes": [], "items": [], "max_lane_items": [], "rounds": []}
    for g in range(0, args.seeds - 31, 32):
        group = per_seed[g:g + 32]
        for i in range(max(len(q) for q in group)):
            here = [q[i] for q in group if i < len(q)]
            items = [d[1] + d[2] for d in here]
            steps["distinct_types"].append(len({d[0] for d in here}))
            steps["lanes"].append(len(here))
            steps["items"].append(sum(items))
            steps["max_lane_items"].append(max(items))
            steps["rounds"].append(-(-sum(items) // len(here)))

    def hist(a):                                  # share of deliveries with each count
        return {int(k): round(float(c) / len(a), 4) for k, c in zip(*np.unique(a, return_counts=True))}

    report = {
        "workload": "raft5 double-vote bug, max_messages 50, invariant every 5, seeds %d..%d"
                    % (args.seed_base, args.seed_base + args.seeds - 1),
        "deliveries_per_prefix": len(flat) / args.seeds,
        "events_per_prefix": n_events / args.seeds,
        "actor_sends_per_delivery": float(sends.mean()), "actor_sends_hist": hist(sends),
        "flush_items_per_delivery": float(flush.mean()), "flush_items_hist": hist(flush),
        "delivered_types": {k: round(v / len(flat), 4) for k, v in types.most_common()},
        "warp_step": {k: float(np.mean(v)) for k, v in steps.items()},
    }
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
