"""Per-kernel SASS of two builds of liblsbsort.so, compared ignoring symbol names and addresses: does every kernel of the
first build have an identical instruction stream in the second?

    cuobjdump -sass A/liblsbsort.so > a.sass; cuobjdump -sass B/liblsbsort.so > b.sass
    python tools/sass_compare.py a.sass b.sass"""
import re, subprocess, sys
def parse(path):
    funcs, cur = {}, None
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1); funcs[cur] = []; continue
        if cur is None: continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?);", line)
        if m:
            ins = re.sub(r"`\([^)]*\)", "SYM", m.group(1))
            funcs[cur].append(ins.strip())
    return funcs
old, new = parse(sys.argv[1]), parse(sys.argv[2])
dem = lambda names: dict(zip(names, subprocess.run(["cu++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")))
do, dn = dem(list(old)), dem(list(new))
newsig = {}
for k, v in new.items(): newsig.setdefault(tuple(v), []).append(dn[k])
bad = 0
for k, v in old.items():
    hit = newsig.get(tuple(v))
    print(("SAME " if hit else "DIFF ") + f"{len(v):6d}  {do[k][:110]}" + (f"  == {hit[0][:90]}" if hit else ""))
    bad += not hit
print(f"{len(old) - bad}/{len(old)} parent kernels have an identical instruction stream in the branch build")
