import os.path as osp, sys; sys.path.insert(0, osp.dirname(osp.dirname(osp.abspath(__file__))))
import torch, time
import svdformer_pointsea_b200 as ps
g=torch.Generator().manual_seed(0)
for B,N,m in ((8,131072,2048),(4,131072,2048),(9,16384,512),(32,16384,2048),(40,16384,512),(16,65536,512)):
    x=(torch.rand(B,N,3,generator=g)-0.5).cuda()
    for _ in range(2): ps.furthest_point_sample(x,m)
    torch.cuda.synchronize(); e0=torch.cuda.Event(enable_timing=True); e1=torch.cuda.Event(enable_timing=True)
    e0.record(); ps.furthest_point_sample(x,m); e1.record(); e1.synchronize()
    print(B,N,m, round(e0.elapsed_time(e1)*1e3/(m-1),3),'us/iter')
