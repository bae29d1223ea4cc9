#!/usr/bin/env python
"""Writes profiles/r2_sass_mnemonics.md: mnemonic histogram of the shipped library's SASS (cuobjdump, no GPU needed).
    python tools/sass_mnemonics.py
"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "invpref_kdd_2022_b200", "libinvpref_b200.so")
PICK = [
    ("fused user pass (lazy, EXACT D=64 K=4)", r"upass_rows_staged_kernelILi4ELi1ELi4ELi0ELb1ELi64E"),
    ("item pass ring rows (Adam, stash, EXACT D=64 K=4)", r"bwd_rows_ring_kernelILi4ELi1ELi0ELb1ELi4ELi64E"),
    ("EM re-assignment (EXACT D=64 K=4)", r"cluster_kernelILi4ELi1ELi4ELi64E"),
    ("streaming top-k: evaluator and recommend", r"topk_stream_kernel"),
    ("fused implicit evaluator below 2048 items", r"eval_topk_kernel"),
    ("radix sort: rank + scatter one 8-bit digit", r"rs_scatter_kernel"),
    ("radix sort: tile histogram", r"rs_hist_kernel"),
    ("prefix sum: per-tile scan (head flags, inclusive)", r"sc_scan_kernelILi1ELb1E"),
    ("multi-GPU owner reduce + Adam + push (8 ranks)", r"owner_adam_push_kernelILi4ELi8E"),
    ("multi-GPU all-reduce + barrier over peer memory: post", r"peer_post_kernel"),
    ("multi-GPU all-reduce + barrier over peer memory: wait + reduce", r"peer_reduce_kernel"),
    ("dense Adam sweep", r"sweep_kernelILi4ELi1E"),
    ("tail", r"tail_kernel"),
]
WATCH = ["LDGSTS", "LDGDEPBAR", "DEPBAR", "LDG", "STG", "LDS", "STS", "SHFL", "VOTE", "MATCH", "MUFU", "ATOMS", "ATOMG",
         "RED", "MEMBAR", "NANOSLEEP", "UBLKCP", "UTMALDG", "SYNCS", "UTCHMMA", "HMMA"]


def main():
    txt = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    archs = sorted(set(re.findall(r"arch = (sm_\w+)", txt)))
    funcs, cur = collections.OrderedDict(), None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = collections.Counter()
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)", line)
        if m and cur:
            funcs[cur][m.group(1)] += 1
    total = collections.Counter()
    for c in funcs.values():
        total.update(c)
    out = ["# Round 2 — SASS of the shipped library (`cuobjdump -sass invpref_kdd_2022_b200/libinvpref_b200.so`, "
           "`tools/sass_mnemonics.py`)", "",
           f"Architectures in the fat binary: {archs}; {len(funcs)} kernels.", "",
           "Whole library, selected mnemonics: " + ", ".join(f"`{k}` {total.get(k, 0)}" for k in WATCH), "",
           "No `UBLKCP` / `UTMALDG` / `SYNCS` (bulk copies, TMA, mbarrier) and no `UTC*MMA` / `HMMA` (tensor cores): the path "
           "has no contraction wider than K <= 8 outputs (done with half-warp shuffles), and its row staging is per-lane "
           "`cp.async` (`LDGSTS`) with `cp.async.wait_group` (`LDGDEPBAR` / `DEPBAR`).  The bulk-copy form was built and "
           "measured on the re-assignment kernel (`r2_bulk_copy_ab.md`: 24 % slower, the variant build does contain "
           "`UBLKCP` / `SYNCS`); the per-lane form stays.  The two row kernels are occupancy-bound, not DRAM-bound "
           "(DESIGN.md section 3, finding 2).  `MEMBAR` / `NANOSLEEP` belong to the peer-memory all-reduce "
           "(`fence.sys`, bounded acquire spin); `VOTE` to the radix sort's ballot peer masks.", "",
           "| kernel | instructions | top mnemonics |", "|---|---|---|"]
    for label, rx in PICK:
        name = next((f for f in funcs if re.search(rx, f)), None)
        if name is None:
            continue
        c = funcs[name]
        top = ", ".join(f"{k} {v}" for k, v in c.most_common(9))
        extra = ", ".join(f"{k} {c.get(k, 0)}" for k in ("LDGSTS", "SHFL", "VOTE", "MUFU", "MEMBAR"))
        out.append(f"| {label} (`{name[name.find(rx[:12]) if rx[:12] in name else 0:][:48]}`) | {sum(c.values())} | {top}; {extra} |")
    open(os.path.join(ROOT, "profiles", "r2_sass_mnemonics.md"), "w").write("\n".join(out) + "\n")
    print("\n".join(out[:12]))


if __name__ == "__main__":
    main()
