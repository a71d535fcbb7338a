"""Compare the SASS of two builds of one object file kernel by kernel, ignoring addresses and encodings.

    cuobjdump -sass OLD.o > old.sass; cuobjdump -sass NEW.o > new.sass
    python scripts/sass_compare.py old.sass new.sass

A kernel of OLD that NEW has as a template with one more trailing argument equal to 3 (the fp16-split kernels' term
count, csrc/gemm_tc.cu), or as a template <3> where OLD had a plain kernel, is matched to that instantiation."""
import re, subprocess, sys
def funcs(path):
    out, cur, name = {}, None, None
    for line in open(path):
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1); cur = out.setdefault(name, []); continue
        if cur is None: continue
        # instruction text without the address comment and the encoding
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?);", line)
        if m: cur.append(m.group(1).strip())
    return out
def dem(n):
    return subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip()
old, new = funcs(sys.argv[1]), funcs(sys.argv[2])
newd = {dem(k): k for k in new}
same = diff = 0
for k, body in old.items():
    d = dem(k)
    cand = None
    if d in newd: cand = newd[d]
    else:
        # the same kernel with a trailing term count 3 appended / turned into a template
        base = re.sub(r"^void ", "", re.sub(r"\(.*$", "", d))
        for nd, nk in newd.items():
            nb = re.sub(r"\(.*$", "", nd)
            nb = re.sub(r"^void ", "", nb)
            if re.sub(r", 3>$", ">", nb) == base or re.sub(r"<3>$", "", nb) == base or \
                    re.sub(r"<([0-9, ]+), 3>$", r"<\1>", nb) == base:
                cand = nk
    if cand is None:
        print("MISSING", d); diff += 1; continue
    b2 = new[cand]
    ok = body == b2
    same += ok; diff += not ok
    print("IDENTICAL" if ok else "DIFFERENT", f"{len(body):6d} {len(b2):6d}", d, "->", dem(cand))
print(f"{same} identical, {diff} different/missing of {len(old)}")
