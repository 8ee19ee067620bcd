"""Compare the SASS of every kernel of two builds of libqanneal.so, instruction by instruction (addresses dropped).  Kernels
are matched by their demangled names, the anonymous namespace written as its translation unit; a kernel present in only
one build is listed as such.  --rename OLD=NEW (repeatable) matches a kernel whose template arguments were renamed: the
first rule whose OLD occurs in a name of the OLD build replaces it there by NEW.

    python tools/sass_compare.py [--rename OLD=NEW ...] OLD.so NEW.so
    (exit 1 if any kernel differs or is missing from one build)

    e.g. --rename 'k_anneal_ref<(int)1>=k_anneal_ref<(qa::GroupKind)2>'
"""
import argparse, re, subprocess, sys

CUDA_BIN = "/usr/local/cuda/bin"


def funcs(lib):
    out = subprocess.run([f"{CUDA_BIN}/cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
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


def keys(names):
    """demangled names; an anonymous namespace becomes the name of its translation unit (its hash differs per build)"""
    dem = subprocess.run([f"{CUDA_BIN}/cu++filt"], input="\n".join(names) + "\n", capture_output=True, text=True,
                         check=True).stdout.splitlines()
    res = []
    for name, d in zip(names, dem):
        m = re.search(r"_GLOBAL__N__[0-9a-f]+_\d+_(\w+?)_cu_[0-9a-f]+", name)
        res.append(d.replace("<unnamed>", f"{m.group(1)}.cu") if m else d)
    return res


def renamed(k, rules):
    for a, b in rules:
        if a in k:
            return k.replace(a, b)
    return k


ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
ap.add_argument("--rename", action="append", default=[], metavar="OLD=NEW")
ap.add_argument("old")
ap.add_argument("new")
args = ap.parse_args()
rules = [tuple(r.split("=", 1)) for r in args.rename]
old, new = funcs(args.old), funcs(args.new)
old = {renamed(k, rules): v for k, v in zip(keys(list(old)), old.values())}
new = dict(zip(keys(list(new)), new.values()))
bad = 0
for k in sorted(set(old) | set(new)):
    if k not in old or k not in new:
        print(f"{'only in NEW' if k in new else 'only in OLD'}  {k}"); bad += 1; continue
    same = old[k] == new[k]
    bad += not same
    print(f"{'identical' if same else 'DIFFERENT'}  {len(old[k]):6d} / {len(new[k]):6d} instructions  {k}")
sys.exit(1 if bad else 0)
