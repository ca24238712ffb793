"""Where one CTA of the persistent bf16x3 update kernel spends its time: clock64 stamps of CTA (0, 0)
(thread 0 = a loss warp of half tile a, thread 256 = a loss warp of half tile b; each half runs its own E0-E5 and
waits on its own C* barriers).  One rank: stamp 26 only appears when clip_grad_norm_ clips (Adam redone + a third
barrier), and stamp 27 follows the read of the clip coefficient."""
import os, sys, tempfile
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import omnisafe_b200, bench
from omnisafe_b200._lib import lib, ptr
cfg = bench._custom_cfgs(1, tempfile.mkdtemp(), 40)
cfg['train_cfgs']['matmul_precision'] = 'bf16x3'
algo = omnisafe_b200.Agent('PPOLag', 'SyntheticBox-v0', custom_cfgs=cfg).agent
for _ in range(2): algo.train_epoch()
dbg = torch.zeros(2048, dtype=torch.int64, device='cuda')
torch.cuda.synchronize()
lib().osb_x3_debug_buffer(ptr(dbg))
algo._update()
torch.cuda.synchronize()
lib().osb_x3_debug_buffer(0)
NAMES = {0: 'E0 start', 1: 'C6(prev) ok', 2: 'X stored+sync', 3: 'C1 ok', 4: 'E1 done', 5: 'C2 ok', 6: 'E2 done', 7: 'C3 ok', 8: 'dOUT stored', 9: 'E3 done',
         10: 'C4A ok', 11: 'E4 computed', 12: 'C4B ok', 13: 'E4 stored', 14: 'C5A ok', 15: 'E5 computed', 16: 'C5B ok', 17: 'E5 stored', 20: 'tiles done',
         21: 'C6 ok', 22: 'extracted', 23: 'barrier1', 24: 'reduced', 25: 'barrier2', 26: 'clip redo+bar3', 27: 'clip coef read', 28: 'restaged'}
for which, off in (('thread 0 (half a)', 0), ('thread 256 (half b)', 1024)):
    d = dbg[off:off + 1024].cpu().tolist()
    n = d[0]
    print(f'== {which}: {n} stamps (last update iteration kept the buffer)')
    prev = None
    # print the first minibatch only (until second id 28) ... stamps restart every launch: take the tail launch
    rows = [(d[1 + 2 * i], d[2 + 2 * i]) for i in range(n)]
    # first minibatch of the (last) launch
    t0 = rows[0][1]
    cnt28 = 0
    for id_, clk in rows:
        dt = 0 if prev is None else clk - prev
        print(f'  {NAMES.get(id_, id_):16s} +{dt:7d} cyc   t={clk - t0:8d}')
        prev = clk
        if id_ == 28:
            cnt28 += 1
            if cnt28 == 2: break
