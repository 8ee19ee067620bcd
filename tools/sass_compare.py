"""Compare the SASS of every kernel of two builds of libqanneal.so, instruction by instruction (addresses dropped;
anonymous-namespace hashes normalised).  Kernels are matched by name; a kernel present in only one build is listed as such.

    python tools/sass_compare.py OLD.so NEW.so    (exit 1 if any kernel differs or is missing from one build)
"""
import re, subprocess, sys

def funcs(lib):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    res, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if name: res[name] = body
            name, body = m.group(1), []
            continue
        if name and re.match(r"\s+/\*[0-9a-f]{4,}\*/", line):
            ins = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line.split(";")[0]).strip()
            body.append(ins)
    if name: res[name] = body
    return res

def key(name):
    name = re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_(\w+?)_cu_[0-9a-f]+", r"\1", name)
    return name

old, new = funcs(sys.argv[1]), funcs(sys.argv[2])
old = {key(k): v for k, v in old.items()}
new = {key(k): v for k, v in new.items()}
bad = 0
for k in sorted(set(old) | set(new)):
    if k not in old or k not in new:
        print(f"{'only in NEW' if k in new else 'only in OLD'}  {k}"); bad += 1; continue
    same = old[k] == new[k]
    bad += not same
    print(f"{'identical' if same else 'DIFFERENT'}  {len(old[k]):6d} / {len(new[k]):6d} instructions  {k}")
sys.exit(1 if bad else 0)
