import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np
from armada_b200 import synth, abi
from armada_b200.scheduler import DeviceRound
import oracle_lib
seed=7
r = synth.random_round(seed, away=(seed % 4 == 1), round_limit=(seed % 6 == 3), queue_limits=(seed % 6 == 4),
        protected_fraction=0.5 if seed % 3 == 2 else 0.0, lookback=40 if seed % 5 == 1 else 0,
        n_nodes=40 + 13 * (seed % 7), n_jobs=300 + 50 * (seed % 5), n_running=80 + 20 * (seed % 4))
inp=r.to_input()
want=oracle_lib.round_schedule(inp)
got=DeviceRound(0).schedule(inp)
for nm in ("loop_iterations","probes","placements","evicted_pass1","evicted_pass2","fair_preemption_scans"):
    print(nm, getattr(got.stats,nm), getattr(want.stats,nm))
bad=np.nonzero((got.job_state!=want.job_state)|(got.job_node!=want.job_node)|(got.job_method!=want.job_method)|(got.job_scheduled_at_priority!=want.job_scheduled_at_priority))[0]
jc=np.asarray(r.job_class).astype(int); 
for j in bad:
    print('job',j,'cls',jc[j],'pc',r.class_pc[jc[j]],'req',r.class_request[jc[j]]//np.array([2**30,1000,1000]),'q',r.job_queue[j],'gang',r.job_gang[j],'node0',r.job_node[j],'sap0',r.job_scheduled_at_priority[j],
      '| dev st',got.job_state[j],'node',got.job_node[j],'sa',got.job_scheduled_at_priority[j],'pa',got.job_preempted_at_priority[j],'m',got.job_method[j],
      '| ora st',want.job_state[j],'node',want.job_node[j],'sa',want.job_scheduled_at_priority[j],'pa',want.job_preempted_at_priority[j],'m',want.job_method[j])
# first divergence in attempt order
ds, os_ = got.job_seq.astype(np.int64), want.job_seq.astype(np.int64)
print('seq equal:', (ds==os_).all())
mx=int(max(ds.max(), os_.max()))
dev_by={}; ora_by={}
for j in range(len(ds)):
    if ds[j]: dev_by.setdefault(int(ds[j]),[]).append(j)
    if os_[j]: ora_by.setdefault(int(os_[j]),[]).append(j)
for sq in range(1,mx+1):
    a=dev_by.get(sq,[]); b=ora_by.get(sq,[])
    same = a==b and all(got.job_node[j]==want.job_node[j] and got.job_method[j]==want.job_method[j] and got.job_state[j]==want.job_state[j] for j in a)
    if not same:
        print('first divergence at seq',sq,'dev jobs',a,'ora jobs',b)
        for j in sorted(set(a+b)):
            print('  job',j,'cls',jc[j],'q',r.job_queue[j],'gang',r.job_gang[j],'node0',r.job_node[j],'| dev',got.job_state[j],got.job_node[j],got.job_method[j],got.job_preempted_at_priority[j],'| ora',want.job_state[j],want.job_node[j],want.job_method[j],want.job_preempted_at_priority[j])
        break
