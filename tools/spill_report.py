"""Per-device-function register / spill report of the decode kernel (CPU only, ~1 min).

    python tools/spill_report.py            # compiles jukebox_b200/csrc/decode_engine.cu to a temporary directory and analyses it
    python tools/spill_report.py file.o     # analyse an existing object

Why it exists: the persistent kernel runs 9 warps per CTA, which caps it at 168 registers, and ptxas'
inter-procedural allocation of the __noinline__ phases is fragile - an unrelated edit in the attention
code has twice moved stage_acts (16 x 16-byte loads in flight per thread) into a regime where it spills
part of its load batch; the STL then waits for the load and serialises everything behind it (+1.6 us per
GEMM phase, +400 us per token).  stage_acts must report STL 0 / LDL 0 before a kernel change is measured.
"""
import os
import re,sys,subprocess,tempfile
if len(sys.argv) > 1:
    o = sys.argv[1]
else:
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tmp = tempfile.TemporaryDirectory()     # private per run: a fixed shared path may belong to another user
    o = os.path.join(tmp.name, "jk_decode_engine_spill.o")
    subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
                    "-c", os.path.join(root, "jukebox_b200", "csrc", "decode_engine.cu"), "-o", o], check=True)
sass=subprocess.run(f"cuobjdump -sass {o}", shell=True, capture_output=True, text=True).stdout.splitlines()
st=[i for i,l in enumerate(sass) if 'Function : ' in l and 'jk_decode_step' in l][0]
ins=[]
for l in sass[st:]:
    m=re.match(r'\s*/\*([0-9a-f]{4,6})\*/\s+(.*?);', l)
    if m: ins.append((int(m.group(1),16), m.group(2)))
sym=subprocess.run(f"cuobjdump -elf {o} | grep -E '0x[0-9a-f]+ +0x[0-9a-f]+ +0x[0-9a-f]+ .*(stage_acts|attn_pv|attn_scores|attn_item|gemm_phase|logits_phase|attn_prefetch|producer_loop)' | grep -v Value", shell=True, capture_output=True, text=True).stdout
funcs=[]
for l in sym.splitlines():
    f=l.split()
    name=[k for k in ("stage_acts","attn_pv","attn_scores","attn_item","gemm_phase","logits_phase","attn_prefetch","producer_loop") if k in l][0]
    funcs.append((int(f[1],16), int(f[2],16), name))
funcs=sorted(set(funcs))
for off,size,name in funcs:
    body=[t for a,t in ins if off<=a<off+size]
    regs=[int(x) for t in body for x in re.findall(r'\bR(\d+)\b', t)]
    print(f"{name:14s} n_ins {len(body):5d} maxR {max(regs) if regs else -1:4d} STL {len([t for t in body if t.startswith('STL')]):3d} LDL {len([t for t in body if 'LDL' in t]):3d}")
kern=[t for a,t in ins if a<funcs[0][0]]
regs=[int(x) for t in kern for x in re.findall(r'\bR(\d+)\b', t)]
print(f"{'kernel':14s} n_ins {len(kern):5d} maxR {max(regs):4d} STL {len([t for t in kern if t.startswith('STL')]):3d} LDL {len([t for t in kern if 'LDL' in t]):3d}")
