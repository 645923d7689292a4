"""Static SASS census of the hot loops of libbeacon_b200 (no GPU needed; runs at build time).

For every kernel the bench reports a roofline for, the loop structure is recovered from the backward
branches of `cuobjdump -sass`, and per loop body the instructions that occupy the two units these
kernels are bound by are counted:
  * fp64 pipe: DFMA / DMUL / DADD / DSETP / DMNMX — one warp instruction holds a sub-partition's 16
    fp64 lanes for 2 cycles, i.e. the SM issues at most 2 fp64 warp-instructions per cycle;
  * shared-memory pipe: LDS / STS / SHFL in 128-byte wavefronts (32 lanes x 4 B = 1, x 8 B = 2,
    x 16 B = 4; a 64-bit shuffle is two SHFL), conflict free, unpredicated instructions only
    (predicated ghost-cell copies of the few boundary tiles are listed separately) — the SM moves at
    most one wavefront per cycle.
`bench.py` multiplies these per-loop counts by the trip counts of the run (sub-steps, Jacobi sweeps
counted by the kernel itself, active warps) and divides by the measured time and the sampled SM
clock: that is `roofline.frac`.  The model is checked against ncu's executed-instruction counters in
DESIGN.md §5.

Usage: python tools/sass_census.py [out.json]      (reads beacon_b200/lib/obj/*.o)
"""
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "beacon_b200", "lib", "obj")
FP64 = ("DFMA", "DMUL", "DADD", "DSETP", "DMNMX")


def functions(obj):
    """{demangled-ish function line: [(addr, text)]} of one object file."""
    txt = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in txt.splitlines():
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            out[cur] = []
            continue
        m = re.match(r"\s+/\*([0-9a-f]+)\*/\s+(.*?);", line)
        if m and cur is not None:
            out[cur].append((int(m.group(1), 16), m.group(2).strip()))
    return out


def classify(text):
    """(opcode, predicated, fp64, smem wavefronts, is barrier)"""
    m = re.match(r"(@!?U?P\w+\s+)?([A-Z0-9_]+)((?:\.[A-Z0-9_]+)*)", text)
    if not m:
        return "?", False, 0, 0, False
    pred, op, mods = bool(m.group(1)), m.group(2), m.group(3) or ""
    wf = 0
    if op in ("LDS", "STS"):
        wf = 4 if ".128" in mods else (2 if ".64" in mods else 1)
    elif op == "SHFL":
        wf = 1
    return op, pred, int(op in FP64), wf, op == "BAR"


def loops_of(ins):
    addr = {a: i for i, (a, _) in enumerate(ins)}
    res = []
    for i, (a, s) in enumerate(ins):
        m = re.search(r"\bBRA(?:\.U)?(?:\.[A-Z]+)*\s+.*?(0x[0-9a-f]+)", s)
        if m:
            t = int(m.group(1), 16)
            if t <= a and t in addr:
                res.append((addr[t], i))
    return sorted(set(res))


def count(ins, lo, hi, exclude=()):
    c = collections.Counter()
    for i in range(lo, hi + 1):
        if any(a <= i <= b for a, b in exclude):
            continue
        op, pred, f64, wf, bar = classify(ins[i][1])
        c["instr"] += 1
        c["fp64"] += f64
        c["bar"] += bar
        if wf:
            c["smem_wavefronts_pred" if pred else "smem_wavefronts"] += wf
            c["smem_instr"] += 1
        if op == "MUFU":
            c["mufu"] += 1
        if op in ("LDL", "STL"):
            c["local"] += 1
    return dict(c)


def find(funcs, *needles):
    hits = [k for k in funcs if all(n in k for n in needles)]
    if len(hits) != 1:
        raise RuntimeError(f"kernel {needles}: {len(hits)} matches")
    return hits[0], funcs[hits[0]]


def census():
    out = {"how": "tools/sass_census.py: static per-loop instruction counts of the shipped SASS (per thread = per warp instruction)"}
    # ---- shkadov: the sub-step loop of the single-body kernel is unrolled by two (2 barriers per trip) ------
    f = functions(os.path.join(OBJ, "shkadov.o"))
    for tag, needles in (("shkadov_6_256_2", ("shkadov_kernel", "IdLi6ELi256ELi2E")), ("shkadov_6_512_1", ("shkadov_kernel", "IdLi6ELi512ELi1E")),
                         ("shkadov_10_192_2", ("shkadov_kernel", "IdLi10ELi192ELi2E")),
                         ("shkadov_6_5_256_2", ("shkadov_balanced_kernel", "IdLi6ELi5ELi256ELi2ELi128ELi4E")),
                         ("shkadov_6_5_96_256_2", ("shkadov_balanced_kernel", "IdLi6ELi5ELi256ELi2ELi96ELi1E"))):
        name, ins = find(f, *needles)
        cand = []
        for lo, hi in loops_of(ins):
            c = count(ins, lo, hi)
            if c.get("fp64", 0) >= 100 and c.get("bar", 0) in (1, 2):
                c["per_substep"] = {k: v / c["bar"] for k, v in c.items() if k != "bar"}
                c["range"] = [hex(ins[lo][0]), hex(ins[hi][0])]
                cand.append(c)
        # unrolled-by-two single body (F_SMALL: off <= 1) when present, else the leanest one-barrier body (F_NONE)
        two = [c for c in cand if c["bar"] == 2]
        one = sorted((c for c in cand if c["bar"] == 1), key=lambda c: c["fp64"])
        out[tag] = {"kernel": name, "substep_unrolled2": two[0] if two else None, "substep_bodies": one}
        if len(two) > 1:   # balanced layout: one unrolled body per chunk width, the wider (more fp64) first
            out[tag]["substep_unrolled2_per_width"] = sorted(two, key=lambda c: -c["fp64"])
    # ---- rayleigh / mixing: sweep loop (2 sweeps, 2 barriers per trip) inside the sub-step loop -----------------
    f = functions(os.path.join(OBJ, "mac2d.o"))
    for tag, needles in (("rayleigh_reg", ("mac_reg_kernel", "IdLi50ELi50ELi2ELi5ELi256ELb0E")),
                         ("mixing_big", ("mac_big_kernel", "IdLi100ELi100ELi4ELi5ELi512ELi1ELb0E"))):
        name, ins = find(f, *needles)
        ls = loops_of(ins)
        stats = [(lo, hi, count(ins, lo, hi)) for lo, hi in ls]
        def bfly(lo, hi):
            return sum(1 for i in range(lo, hi + 1) if ins[i][1].split()[0 if not ins[i][1].startswith("@") else 1].startswith("SHFL.BFLY"))
        # the sweep loop: two CTA barriers per trip, the butterfly shuffles of the residual reduction, no inner barrier loop
        sweeps = [s for s in stats if s[2].get("bar", 0) == 2 and s[2].get("fp64", 0) >= 60 and bfly(s[0], s[1]) >= 8 and
                  not any(o[0] >= s[0] and o[1] <= s[1] and (o[0], o[1]) != (s[0], s[1]) and o[2].get("bar", 0) for o in stats)]
        sw = max(sweeps, key=lambda s: s[2]["fp64"])
        outer = min((s for s in stats if s[0] <= sw[0] and s[1] >= sw[1] and (s[0], s[1]) != (sw[0], sw[1])), key=lambda s: s[1] - s[0])
        other = count(ins, outer[0], outer[1], exclude=[(sw[0], sw[1])])
        entry = {"kernel": name,
                 "sweep_pair": dict(sw[2], range=[hex(ins[sw[0]][0]), hex(ins[sw[1]][0])]),
                 "per_sweep": {k: v / 2 for k, v in sw[2].items()},
                 "substep_other": dict(other, range=[hex(ins[outer[0]][0]), hex(ins[outer[1]][0])],
                                       note="sub-step loop body outside the sweep loop: BCs, predictor, first two (peeled) sweeps, corrector, "
                                            "transport coefficients; all warps")}
        # the noinline transport wavefront is placed behind the kernel body (reached by CALL.REL): a barrier-free
        # loop with shuffles outside the sub-step loop's address range
        def shfl(lo, hi):
            return sum(1 for i in range(lo, hi + 1) if classify(ins[i][1])[0] == "SHFL")
        wl = max((s for s in stats if s[0] > outer[1] and not s[2].get("bar", 0) and shfl(s[0], s[1]) >= 6 and s[2].get("fp64", 0) >= 12),
                 key=lambda s: s[2]["instr"])
        entry["wavefront_loop"] = dict(wl[2], range=[hex(ins[wl[0]][0]), hex(ins[wl[1]][0])], note="transport wavefront, ONE warp, 6 columns per trip")
        out[tag] = entry
    return out


if __name__ == "__main__":
    res = census()
    dst = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "beacon_b200", "lib", "sass_census.json")
    json.dump(res, open(dst, "w"), indent=1)
    for k, v in res.items():
        if isinstance(v, dict):
            if "per_sweep" in v:
                print(k, "per sweep:", v["per_sweep"], "| other per sub-step:", {a: b for a, b in v["substep_other"].items() if a in ("fp64", "smem_wavefronts", "instr")},
                      "| wavefront trip:", {a: b for a, b in v["wavefront_loop"].items() if a in ("fp64", "smem_wavefronts", "instr")})
            else:
                u2 = v["substep_unrolled2"]
                print(k, "unrolled2 per sub-step:", u2 and u2["per_substep"], "| one-barrier bodies fp64:", [c["fp64"] for c in v["substep_bodies"]])
                for c in v.get("substep_unrolled2_per_width", []):
                    print("   unrolled2 body", c["range"], "instr", c["instr"], "fp64", c["fp64"])
    print("wrote", dst)
