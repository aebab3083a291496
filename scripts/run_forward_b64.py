import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import __graft_entry__ as ge; ge.build()
import lipsync_b200 as lb
m = lb.LipSyncModel(); m.load_state_dict(lb.make_synthetic_state_dict(0)); m.to('cuda').eval(); m.compute_precision='bf16'
v, a = lb.synthetic_windows(1, 4)
v = v.repeat(16,1,1,1,1).cuda(); a = a.repeat(16,1,1,1).cuda()
for _ in range(3): m(v, a)
torch.cuda.synchronize()
