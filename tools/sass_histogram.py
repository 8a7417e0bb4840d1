"""Per-kernel SASS opcode histograms of libg2048.so (cuobjdump -sass; no GPU needed) -> profiles/r03_sass_opcodes.txt
(profiles/r02_sass_opcodes.txt: the same listing of the round-2 build).
What the listing is evidence for: sm_100a-only cubins; the bulk-copy engine (UBLKCP = cp.async.bulk) in the streaming
kernels; the Threefry instruction mix (SHF.L.W / LOP3 on the ALU pipe, the adds as IMAD on the FMA pipe) and the shared-memory
table loads (LDS.U16 / LDS.U8) in the play kernels; no tensor-core or tensor-memory instructions -- the path has no
contraction (HMMA / UTCMMA / LDTM would be out of place).

It also counts the STEP BODY of the plain play kernels (play3_kernel<partitionable, policy, no recording>): the
instructions from the first sub-key load (LDG.E.64.CONSTANT) to the main loop's back branch, i.e. what one env-step
executes, split by the pipe that takes them (ALU_PIPE below; IMAD* goes to the FMA pipe, LDS / LDG to the LSU pipe).

    python tools/sass_histogram.py [--lib path/to/libg2048.so] [--out profiles/r03_sass_opcodes.txt]"""
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
LIB = ROOT / "2048-ppo-agent_b200" / "libg2048.so"
OUT = ROOT / "profiles" / "r03_sass_opcodes.txt"
# opcodes (first dotted component) issued to the ALU pipe on sm_100a: the integer/logic pipe that takes one warp
# instruction every two cycles per scheduler (VIADD, PRMT and LEA.HI: tools/probes/probe_int.cu, profiles/README.md)
ALU_PIPE = ("LOP3", "SHF", "IADD3", "SEL", "VIADD", "PRMT", "LEA", "ISETP", "IMNMX", "VIMNMX", "FSEL", "FSETP", "PLOP3",
            "P2R", "R2P", "FLO", "BREV", "IABS", "LOP", "IADD", "MOV")
STEP_KERNELS = ("play3_kernel<1, 0, false>", "play3_kernel<1, 1, false>")
KEEP = ("play3_kernel", "play2_kernel", "play_record_compact", "policy_step_obs", "policy_step_kernel", "rollout_steps_kernel",
        "expand_obs_tma_kernel", "pack_samples", "gae_scan_kernel", "gae_scan_fix", "gae_flat4_kernel", "gae_flat3_kernel",
        "gae_time_major_kernel", "gae_time_major_ring_kernel", "gather_samples_tile_kernel", "compact_records_kernel",
        "scan_chunk", "normalize_kernel", "embed_boards_kernel", "embed_grad_partial", "chain_kernel", "replay_envs")


def step_body(listing):
    """Opcode counter of the main loop's step body of one play3_kernel listing (see the module docstring)."""
    ins = re.findall(r"/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)([^;]*);", listing)
    start = next(i for i, (_, op, _) in enumerate(ins) if op.startswith("LDG.E.64.CONSTANT"))
    start_addr = int(ins[start][0], 16)
    for end in range(start, len(ins)):
        addr, op, rest = ins[end]
        m = re.match(r"\s*(0x[0-9a-f]+)\s*$", rest)
        if op == "BRA" and m and int(m.group(1), 16) < start_addr:
            break
    return collections.Counter(op for _, op, _ in ins[start:end + 1])


def pipe_of(op):
    head = op.split(".")[0]
    if head.startswith("IMAD"):
        return "fma"
    if head in ("LDS", "LDG", "STS", "STG", "ATOMS", "ATOMG", "RED", "LDC", "SHFL"):
        return "lsu"
    return "alu" if head in ALU_PIPE else "other"


def main():
    global LIB, OUT
    if "--lib" in sys.argv:
        LIB = Path(sys.argv[sys.argv.index("--lib") + 1]).resolve()
    if "--out" in sys.argv:
        OUT = Path(sys.argv[sys.argv.index("--out") + 1]).resolve()
    sass = subprocess.run(["cuobjdump", "-sass", str(LIB)], capture_output=True, text=True, check=True).stdout
    listings, name = {}, None
    archs = sorted(set(re.findall(r"arch = (sm_\w+)", sass)))
    kernels, name = collections.OrderedDict(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
            kernels[name] = collections.Counter()
            listings[name] = []
            continue
        if name:
            listings[name].append(line)
        m = re.match(r"\s*/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m and name:
            kernels[name][m.group(1)] += 1
    out = [f"# SASS opcode histograms of {LIB.name} (tools/sass_histogram.py); cubin architectures: {', '.join(archs)}",
           f"# kernels in the library: {len(kernels)}", ""]
    everything = collections.Counter()
    for c in kernels.values():
        everything.update(c)
    special = {k: v for k, v in everything.items() if re.match(r"(UBLKCP|UTMA|UTC|LDTM|STTM|HMMA|HGMMA|SYNCS|ATOM|RED|BAR|LDS|STS|LDG|STG|SHF|LOP3|IMAD|IADD3|PRMT|SHFL)", k)}
    out.append("## whole library, selected opcode families")
    for k, v in sorted(special.items(), key=lambda kv: -kv[1]):
        out.append(f"{v:8d}  {k}")
    out.append("")
    out.append("tensor-core / tensor-memory opcodes (HMMA, HGMMA, UTC*MMA, LDTM, STTM): "
               + str(sum(v for k, v in everything.items() if re.match(r"(HMMA|HGMMA|UTC\w*MMA|LDTM|STTM)", k))) + " (none: the path has no contraction)")
    out.append("")
    for name, c in kernels.items():
        if not any(k in name for k in KEEP):
            continue
        total = sum(c.values())
        out.append(f"## {name[:150]}")
        out.append(f"   {total} instructions; " + ", ".join(f"{k} {v}" for k, v in c.most_common(14)))
        out.append("")
    for want in STEP_KERNELS:
        name = next((k for k in kernels if want in k), None)
        if name is None:
            continue
        body = step_body("\n".join(listings[name]))
        by_pipe = collections.Counter()
        for op, v in body.items():
            by_pipe[pipe_of(op)] += v
        out.append(f"## step body of {want} (first sub-key load .. loop back branch)")
        out.append(f"   {sum(body.values())} instructions; by pipe: " + ", ".join(f"{k} {v}" for k, v in by_pipe.most_common()))
        out.append("   " + ", ".join(f"{k} {v}" for k, v in body.most_common()))
        out.append("")
    OUT.write_text("\n".join(out) + "\n")
    print("wrote", OUT, len(kernels), "kernels")


if __name__ == "__main__":
    main()
