"""CPU stand-in for a replicate: records which worker ran which item and returns the item's boot (used by
test_host.py)."""
import os
import time


def run(rank, args, item):
    if item.get("fail"):
        raise RuntimeError("boom")
    time.sleep(0.01 * item.get("cost", 1))
    with open(os.path.join(args.out, f"item_{item['boot']}.txt"), "w") as fh:
        fh.write(f"{rank} {int(item['site_order'].sum())}\n")
    return item["boot"]
