"""Where the training step goes on the GPU: torch.profiler kernel table of two eager steps (development tool)."""
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ccvpe_b200 import losses, models
from ccvpe_b200.ddp import GradientAllReducer
from ccvpe_b200.synthetic import fill_deterministic, synthetic_ground_truth, synthetic_pair

dev = torch.device("cuda")
torch.backends.cudnn.benchmark = True
model = models.CVM_VIGOR("cuda", True)
fill_deterministic(model.state_dict(), seed=0)
model = model.to(dev).set_precision("bf16").train()
red = GradientAllReducer(model)
opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4, fused=True)
B = 8
batch = [t.to(dev) for t in synthetic_pair(B, (320, 640), seed=1)] + [t.to(dev) for t in synthetic_ground_truth(B, seed=1)]
batch[0] = batch[0].contiguous(memory_format=torch.channels_last)
batch[1] = batch[1].contiguous(memory_format=torch.channels_last)

def step():
    red.zero_grad()
    loss = losses.training_loss(model(batch[0], batch[1]), *batch[2:])
    loss.backward()
    red.finish()
    opt.step()

for _ in range(3):
    step()
torch.cuda.synchronize()
from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
    for _ in range(2):
        step()
    torch.cuda.synchronize()
print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=45, max_name_column_width=70))
