"""Compare the SASS of the annealing and energy kernels of two builds of libqanneal.so, instruction by instruction
(addresses dropped; anonymous-namespace hashes normalised).  Used to show that the interval-group instantiations leave the
existing ones untouched; the lockstep / warp-per-read template flag became an int and k_energy a template, so those are
matched by their new names.

    python tools/sass_compare.py OLD.so NEW.so    (exit 1 if any listed kernel differs)
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
pairs = [
    ("k_anneal_replayILi1ELi32E", "k_anneal_replayILi1ELi32E"), ("k_anneal_replayILi2ELi32E", "k_anneal_replayILi2ELi32E"),
    ("k_anneal_replayILi1ELi64E", "k_anneal_replayILi1ELi64E"), ("k_anneal_replayILi2ELi64E", "k_anneal_replayILi2ELi64E"),
    ("k_anneal_replayILi0ELi32E", "k_anneal_replayILi0ELi32E"), ("k_anneal_replayILi0ELi64E", "k_anneal_replayILi0ELi64E"),
    ("k_anneal_lockstepILi0ELb1E", "k_anneal_lockstepILi0ELi1E"), ("k_anneal_lockstepILi0ELb0E", "k_anneal_lockstepILi0ELi0E"),
    ("k_anneal_refILb1E", "k_anneal_refILi1E"), ("k_anneal_refILb0E", "k_anneal_refILi0E"),
    ("k_energyEPK", "k_energyILb0EEEvPK"),
]
bad = 0
for a, b in pairs:
    ka = [k for k in old if a in k]
    kb = [k for k in new if b in k]
    if len(ka) != 1 or len(kb) != 1:
        print("?", a, ka, b, kb); bad += 1; continue
    same = old[ka[0]] == new[kb[0]]
    bad += not same
    print(f"{'identical' if same else 'DIFFERENT'}  {len(old[ka[0]]):6d} / {len(new[kb[0]]):6d} instructions  {ka[0]}  ->  {kb[0]}")
sys.exit(1 if bad else 0)
