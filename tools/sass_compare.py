"""Compare the SASS of two builds of the library kernel by kernel.

    python tools/sass_compare.py OLD.so NEW.so

Functions are matched by demangled name.  The generic selective-scan kernels, their finalize kernels and ssm_step_kernel
gained a trailing d_state template argument N; NEW's N = 16 instantiations are matched to OLD's kernels without it and
its N = 32 / 64 instantiations are left out.  Instruction text (addresses included) must be identical."""
import re, subprocess, sys
def funcs(lib):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
    res, cur, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if cur: res[cur] = body
            cur, body = m.group(1), []
        elif cur is not None and re.search(r"/\*[0-9a-f]{4,}\*/", line):
            body.append(re.sub(r"\s+", " ", line.split(";")[0]).strip())
    if cur: res[cur] = body
    dem = subprocess.run(["c++filt"], input="\n".join(res), capture_output=True, text=True).stdout.splitlines()
    return {d: res[k] for k, d in zip(res, dem)}
old, new = funcs(sys.argv[1]), funcs(sys.argv[2])
old = {k.replace("void ", ""): v for k, v in old.items()}
new = {k.replace("void ", ""): v for k, v in new.items()}
def key_new(name):
    # drop the added N template argument of the N = 16 instantiations
    return re.sub(r", 16>", ">", name).replace("<16>", "").replace("void ", "")
same = diff = 0
newmap = {}
for k, v in new.items():
    generic = re.search(r"(selscan_(fwd|bwd)(_summary)?_kernel|selscan_bwd_finalize_\w+|ssm_step_kernel)<", k)
    if generic:
        if re.search(r"(, |<)(32|64)>", k): continue
        k = key_new(k)
    newmap[k] = v
for k, v in sorted(old.items()):
    if k not in newmap:
        print("MISSING in new:", k); diff += 1; continue
    if newmap[k] == v: same += 1
    else:
        diff += 1; print("DIFFERENT:", k, len(v), len(newmap[k]))
extra = set(newmap) - set(old)
for k in sorted(extra): print("EXTRA in new:", k)
print(f"{same} identical, {diff} different/missing, {len(extra)} extra, of {len(old)} parent kernels")
