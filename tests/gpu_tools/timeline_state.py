"""Developer tool: per-phase clock64() timeline of the adjoint-state walk (tc_state_bwd_kernel, CTA of (batch 0, head 0));
needs the -DMLSTM_TIMELINE build of mlstm_tc_bwd.cu:  python -c "from xlstm_yolo_b200 import build; build.build_timeline(('mlstm_tc_bwd.cu',))" """
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from xlstm_yolo_b200 import _lib
_lib.LIB_PATH = _lib.LIB_PATH.replace("libmlstm_b200.so", "libmlstm_b200_tl.so")
from xlstm_yolo_b200 import ops
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from test_gpu_parity import make
B, NH, S, DH = (int(x) for x in (sys.argv[1:5] if len(sys.argv) >= 5 else (8, 4, 1600, 128)))
q, k, v, i, f, dh = (x.cuda() for x in make(B, NH, S, DH, torch.bfloat16, "rand"))
pl = ops.MLSTMPlan(q, k, v, i, f, dh)
for _ in range(2):
    pl.forward(); pl.backward(0); pl.backward(1)
torch.cuda.synchronize()
rows = B * NH * S
rpart_off = rows * 4                                       # BwdLayout: dn | rpart | kpart
tl = pl.ws.view(torch.uint8)[rpart_off:rpart_off + 8 * 32 * 8].view(torch.int64).cpu().view(8, 32)
names = ["top", "prep", "sync2", "issueU", "waitMMA", "waitCs", "pass", "syncthr", "store"]
t0 = tl[0, 0].item()
for who, off in (("compute thread 0", 0), ("issuer", 16)):
    print(who)
    for c in range(8):
        row = tl[c, off:off + 9] - t0
        d = [(row[j] - row[j - 1]).item() for j in range(1, 9)]
        print(f"step {c} start {row[0].item():7d}  " + " ".join(f"{n_}:{x:5d}" for n_, x in zip(names[1:], d)))
