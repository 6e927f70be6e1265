"""SASS identity of two builds of libwab_b200.so: `python tools/sass_identity.py OLD.so NEW.so` lists the kernels added
and removed and every kernel present in both whose `cuobjdump -sass` differs. The anonymous-namespace hash in the
mangled names (it changes with the translation unit's contents) is normalised first."""
import re, subprocess, sys
def funcs(path):
    txt = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    txt = re.sub(r"_GLOBAL__N__[0-9a-f]{8}_", "_GLOBAL__N__HASH_", txt)
    out = {}
    for f in re.split(r"\n\s*Function : ", txt)[1:]:
        name, body = f.split("\n", 1)
        out[name.strip()] = body
    return out
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
print("parent kernels", len(a), "new kernels", len(b))
print("added:", sorted(set(b) - set(a)))
print("removed:", sorted(set(a) - set(b)))
diff = [n for n in a if n in b and a[n] != b[n]]
print("identical:", sum(1 for n in a if n in b and a[n] == b[n]), "differing:", diff)
