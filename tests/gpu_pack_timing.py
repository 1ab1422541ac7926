import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from __graft_entry__ import load_pkg
k=load_pkg()
p=k.Problem.synth(2,10000,500,42,0)
rs=k.ResidentSolve(p); rs.set_count_visited(False); rs.load()
for flush in (True, False, False):
    rs.run(flush_l2=flush); rs.download()
    print("flush",flush, rs.timings()["pack_us"])
