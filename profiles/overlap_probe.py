"""Does running the C2 step's kernels on two streams help?  The fixed-width launches are HBM-bound (89 % of peak, few
instructions), the string launches issue-bound (72-80 %): side by side the copy kernels could use the bandwidth the string
kernels leave.  Times the 60 M-row C2 step (device API, inputs resident in HBM) sequentially on one stream and with the
fixed-width launches on a second stream, in the orders a caller could choose.
usage: python profiles/overlap_probe.py [--rows N]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=60_000_000)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    db = bench.build_c2_device(args.rows, 20260103, dev)
    step = bench.DeviceStep(db)
    main_s = torch.cuda.current_stream(dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def sequential():
        step.run()

    def two_streams(strings_first, split_strings=False):
        ev = torch.cuda.Event()
        ev.record(main_s)
        s1.wait_event(ev)
        s2.wait_event(ev)
        def fixed():
            db.run_fixed(step.plan, stream=s1.cuda_stream)
        def strings():
            for so in step.strings:
                db.run_string(so, stream=s2.cuda_stream)
        if strings_first:
            strings(); fixed()
        else:
            fixed(); strings()
        e1, e2 = torch.cuda.Event(), torch.cuda.Event()
        e1.record(s1); e2.record(s2)
        main_s.wait_event(e1); main_s.wait_event(e2)

    def timed(fn, k):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(main_s)
        for _ in range(k):
            fn()
        b.record(main_s)
        torch.cuda.synchronize(dev)
        step.check()
        return a.elapsed_time(b) / k

    out = {"rows": args.rows}
    out["sequential_ms"] = timed(sequential, args.steps)
    out["two_streams_fixed_first_ms"] = timed(lambda: two_streams(False), args.steps)
    out["two_streams_strings_first_ms"] = timed(lambda: two_streams(True), args.steps)
    out["sequential_again_ms"] = timed(sequential, args.steps)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
