"""Compare cuobjdump -sass of two libaadp.so builds kernel by kernel.  Kernels are matched by demangled name; in the new
build the profile variant is the last template argument (0 = the parent's kernel) and ProfDev an extra parameter."""
import re, subprocess, sys
def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    return dict(zip(names, out))
def norm(d):
    d = re.sub(r"\(anonymous namespace\)", "", d)
    if ", aadp::ProfDev)" not in d: return d
    d = d.replace(", aadp::ProfDev)", ")")
    d = re.sub(r"^void (aadp::mask_kernel)<0>", r"\1", d)
    d = re.sub(r"<0>\(", "(", d)          # mask_kernel<0> -> mask_kernel
    d = re.sub(r", 0>\(", ">(", d)        # ..., PRO=0>
    return d
def kernels(path, new):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    ks, cur, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if cur: ks[cur] = body
            cur, body = m.group(1), []
        elif cur is not None:
            t = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip()
            t = re.sub(r"\s*/\* 0x[0-9a-f]+ \*/", "", t)
            if t: body.append(t)
    if cur: ks[cur] = body
    dm = demangle(list(ks))
    res = {}
    for k, v in ks.items():
        d = re.sub(r"\(anonymous namespace\)", "", dm[k])
        if new and ("aadp::" in d) and re.search(r"aadp::(fill_kernel|wave_kernel|packed_kernel|mask_kernel|ucw_enum_kernel)<", d):
            d = d.replace(", aadp::ProfDev)", ")")
            if re.search(r"(, 1>|<1>)\(", d) and not d.startswith("void aadp::ucw_enum_kernel<1>("):
                res.setdefault("__profile_variants__", []).append(d)
                continue
            d = re.sub(r"^void (aadp::mask_kernel)<0>", r"\1", d)
            d = re.sub(r", 0>\(", ">(", d)
        res[d] = v
    return res
a, b = kernels(sys.argv[1], False), kernels(sys.argv[2], True)
pv = b.pop("__profile_variants__", [])
same = [k for k in a if k in b and a[k] == b[k]]
diff = [k for k in a if k in b and a[k] != b[k]]
gone = [k for k in a if k not in b]
extra = [k for k in b if k not in a]
print("parent kernels %d: identical SASS %d, different %d, unmatched %d; profile variants (PRO=1) %d; other new %d"
      % (len(a), len(same), len(diff), len(gone), len(pv), len(extra)))
for k in diff: print("DIFF", k)
for k in gone: print("UNMATCHED", k)
for k in extra: print("NEW", k)
if len(sys.argv) > 3:
    for k in pv: print("PROFILE", k)
