"""Dev tool (no GPU): static SASS size of one kernel by source region, from nvdisasm -g of the built library.
usage: code_size.py <lib.so> <substring of the mangled kernel name>"""
import collections, os, re, subprocess, sys, tempfile
lib, key = sys.argv[1], sys.argv[2]
with tempfile.TemporaryDirectory() as td:
    subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=td, capture_output=True)
    cub = [f for f in os.listdir(td) if f.startswith("rt_kernels")][0]
    txt = subprocess.run(["nvdisasm", "-g", os.path.join(td, cub)], capture_output=True, text=True).stdout.split("\n")
start = [i for i, l in enumerate(txt) if l.startswith(".text.") and key in l][0]
cur, inl, cnt = None, None, collections.Counter()
n = 0
for ln in txt[start + 1:]:
    if ln.startswith(".text.") or ln.startswith("\t.section") and n > 100:
        break
    m = re.search(r'//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?', ln)
    if m:
        cur = (os.path.basename(m.group(1)), int(m.group(2)))
        continue
    if re.match(r"\s+/\*[0-9a-f]{4,5}\*/", ln) and cur:
        cnt[cur] += 1
        n += 1
print("total instructions", n, f"= {n * 16 / 1024:.1f} KB")
src = {}
def line_text(f, l):
    if f not in src:
        p = os.path.join("ray-tracer-s8_b200/csrc", f)
        src[f] = open(p).read().split("\n") if os.path.exists(p) else []
    return src[f][l - 1].strip()[:90] if 0 < l <= len(src[f]) else ""
for (f, l), c in cnt.most_common(int(sys.argv[3]) if len(sys.argv) > 3 else 45):
    print(f"{c:5d} {f}:{l:<5d} {line_text(f, l)}")
