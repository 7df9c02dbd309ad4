import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from fastpcc_b200 import synth
from fastpcc_b200.lossl_coord_int import Config, Model
cfg = dict(channels=256, max_stride_wo_recurrent=2048, max_stride=8192, fea_stride=16)
sd = synth.make_lossl_int_state_dict(seed=7, **cfg)
m = Model(Config(**cfg), device='cuda').load_numpy_state_dict(sd).cuda()
B = int(sys.argv[1])
frames = [torch.from_numpy(synth.with_batch(synth.lidar_frame(1000 + i))).cuda() for i in range(B)]
for it in range(4):
    torch.cuda.synchronize(); t = time.perf_counter()
    d = m.compress_batch(frames); torch.cuda.synchronize(); t1 = time.perf_counter()
    r = m.decompress_batch(d); torch.cuda.synchronize(); t2 = time.perf_counter()
    print(f'iter {it}: compress {1e3*(t1-t):.1f} decompress {1e3*(t2-t1):.1f}', flush=True)
