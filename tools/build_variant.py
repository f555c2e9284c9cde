"""Builds libnerfies_b200 variants with extra -D flags for A/B timing on the GPU box.

  python tools/build_variant.py epidbg -DNFB_EPI_DEBUG
  NFB_LIB_PATH=nerfies_b200/_variants/libnfb_epidbg.so python bench.py ...
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g

name, defs = sys.argv[1], sys.argv[2:]
out = os.path.join(g.REPO, 'nerfies_b200', '_variants', 'libnfb_%s.so' % name)
g._compile(out, ['-DNFB_WITH_TC'] + defs, force=True)
print(out)
