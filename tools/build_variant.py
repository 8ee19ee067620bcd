"""Development aid: build a variant of libqanneal.so with extra nvcc flags into build/variants/<name>.so
(run it with QA_LIB_PATH=$PWD/build/variants/<name>.so).   python tools/build_variant.py dn_lop3 -DDN_LOP3"""
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import __graft_entry__ as g  # noqa: E402

name, flags = sys.argv[1], sys.argv[2:]
out = ROOT / "build" / "variants" / f"{name}.so"
out.parent.mkdir(parents=True, exist_ok=True)
g.build(force=True, extra_flags=flags, out=out)
print(out)
