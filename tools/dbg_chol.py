import sys, torch, ctypes
sys.path.insert(0, '.')
from gpzoo_b200 import functional as F, _cabi
F.set_sync_checks(False)
torch.manual_seed(0)
L, M = 10, 1024
Q = torch.randn(L, M, M, device='cuda')
K = Q @ Q.transpose(1, 2) / M + torch.eye(M, device='cuda')
dbg = torch.zeros(10, dtype=torch.int64, device='cuda')      # 4 phases of the first cluster launch + 6 of its first leaf
_cabi.lib().gpz_chol_debug_(ctypes.c_void_p(dbg.data_ptr()))
for _ in range(3):
    Lc, Linv = F.CholeskyInverse.apply(K)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(); Lc, Linv = F.CholeskyInverse.apply(K); e1.record(); torch.cuda.synchronize()
print("total ms (incl clone/memsets)", e0.elapsed_time(e1))
d = dbg.cpu().tolist()[:4]; tot = sum(d)
print("cycles leaf/panel/trail/inv:", d, [round(x / tot, 3) for x in d], "-> us @1.9GHz:", [round(x / 1900, 1) for x in d])
