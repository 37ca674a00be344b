"""SASS excerpts of the hot kernels for profiles/ (cuobjdump -sass of the in-tree library; runs without a GPU).
    python scripts/sass_excerpts.py > profiles/r2_sass_excerpts.txt"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sass = subprocess.run(["cuobjdump", "-sass", os.path.join(ROOT, "starrocks_b200", "libsr_gpu.so")], capture_output=True, text=True).stdout
lines = sass.split("\n")
starts = [(i, l) for i, l in enumerate(lines) if "Function :" in l]


def body(sub):
    for k, (i, l) in enumerate(starts):
        if sub in l:
            return l.strip(), lines[i:(starts[k + 1][0] if k + 1 < len(starts) else len(lines))]
    return None, []


def ops(b):
    c = collections.Counter()
    for l in b:
        m = re.search(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", l)
        if m:
            c[m.group(1).split(".")[0]] += 1
    return c


def section(title, sub, pats, maxhits=24):
    name, b = body(sub)
    if not b:
        print(f"== {title}: NOT FOUND\n")
        return
    c = ops(b)
    print(f"== {title}\n   {name}\n   instructions: {sum(c.values())}; " + ", ".join(f"{k} {v}" for k, v in c.most_common(18)))
    hits = 0
    for l in b:
        if any(re.search(p, l) for p in pats) and "/*" in l:
            print("   " + re.sub(r"\s+/\* 0x[0-9a-f]+ \*/", "", l).strip())
            hits += 1
            if hits >= maxhits:
                break
    print()


print("SASS excerpts of the hot kernels (cuobjdump -sass starrocks_b200/libsr_gpu.so, sm_100a, CUDA 12.9), round 2.\n"
      "For every kernel: the opcode census of the whole function, then the lines that show the memory path it uses.\n")
section("k_frag_stream_tests<false> (streaming pass, LDG form): 128-bit streaming loads of the two key columns (LDG.E.NA.128), bitmap word fetches from "
        "shared memory (LDS) and global memory (predicated LDG.E.CONSTANT), clamp onto the guard bit (VIMNMX / VIADDMNMX), selection-vector stores",
        "k_frag_stream_testsILb0", [r"LDG\.E\.NA\.128", r"@P\d\s+LDG\.E\.CONSTANT", r"VIMNMX|VIADDMNMX", r"STG\.E\.64", r"VOTE|POPC"])
section("k_frag_gather_join (selection-vector pass of one join): sector gathers of the key column through the selection vector", "k_frag_gather_join",
        [r"LDG", r"STG", r"VOTE|POPC", r"ATOMG"], 16)
section("k_frag_gather_agg<SMEM_AGG=true> (final pass): dependent gathers, shared-memory accumulators (ATOMS / REDS on 32-bit halves)", "k_frag_gather_aggILb1ELb0",
        [r"ATOMS|REDS|RED\.", r"LDG\.E\.CONSTANT", r"LDG\.E\.NA"])
section("k_frag_gather_agg_expand (final pass with one-to-many joins): chain walk through next[] (LDG.E.CONSTANT), global reductions", "k_frag_gather_agg_expand",
        [r"LDG\.E\.CONSTANT", r"RED\.|ATOMG"], 16)
section("k_aggp_scatter<2, CHUNK_SIMPLE> (level-1 scatter of the partitioned aggregate): streaming loads, shared-memory rank atomics (ATOMS), 128-bit record "
        "stores, L2 prefetch of the next tile (CCTL)", "k_aggp_scatterILi2ELi2", [r"ATOMS", r"ATOMG", r"STG\.E\.128", r"CCTL|PREFETCH", r"LDG\.E\.NA"])
section("k_aggp_apply (one CTA per bucket of 8 slices in shared memory): 128-bit record loads, key claim (ATOMS.CAS.64), 32-bit add pairs for the 64-bit states",
        "k_aggp_applyEPK", [r"ATOMS", r"LDG\.E\.128", r"STG"])
section("k_probe_count (join probe, pass 1): 128-bit key loads, bitmap words, first[] words", "k_probe_countE", [r"LDG\.E\.NA\.128", r"LDG\.E\.CONSTANT", r"STG\.E\.128"], 16)
section("k_for_decode<int32> (frame-of-reference pages): word loads of the packed bits, PRMT byte swaps, funnel shifts (SHF), warp scan (SHFL.UP) for ascending "
        "frames, 128-bit stores", "k_for_decodeIi", [r"PRMT", r"SHFL\.UP", r"STG\.E\.128", r"LDG"], 16)
