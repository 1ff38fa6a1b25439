import os, time, torch, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flash_cosine_sim_attention_b200 import flash_cosine_sim_attention
dev='cuda'
for shape in [(4,8,4096,64),(1,8,512,64)]:
    q,k,v,do=(torch.randn(shape,device=dev,dtype=torch.bfloat16) for _ in range(4))
    q.requires_grad_();k.requires_grad_();v.requires_grad_()
    def step():
        o=flash_cosine_sim_attention(q,k,v,causal=True)
        return torch.autograd.grad(o,(q,k,v),do)
    for _ in range(10): step()
    torch.cuda.synchronize()
    n=200
    t0=time.perf_counter()
    for _ in range(n): step()
    t1=time.perf_counter()
    torch.cuda.synchronize()
    t2=time.perf_counter()
    print(shape, "enqueue us/step", (t1-t0)/n*1e6, "total us/step", (t2-t0)/n*1e6)

# the same small step captured in a CUDA graph: one launch of the whole fwd+bwd (5 kernels with programmatic
# dependent launch edges) per replay - what a launch-bound caller would do (DESIGN.md par. 6, test_cuda_graph_capture_...)
shape = (1, 8, 512, 64)
sq, sk, sv, sdo = (torch.randn(shape, device=dev, dtype=torch.bfloat16) for _ in range(4))
sq.requires_grad_(); sk.requires_grad_(); sv.requires_grad_()
def gstep():
    o = flash_cosine_sim_attention(sq, sk, sv, causal=True)
    return torch.autograd.grad(o, (sq, sk, sv), sdo)
side = torch.cuda.Stream()
side.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(side):
    for _ in range(3): gstep()
torch.cuda.current_stream().wait_stream(side)
graph = torch.cuda.CUDAGraph()
with torch.cuda.graph(graph, stream=side):
    outs = gstep()
for _ in range(10): graph.replay()
torch.cuda.synchronize()
n = 500
t0 = time.perf_counter()
for _ in range(n): graph.replay()
torch.cuda.synchronize()
t1 = time.perf_counter()
print(shape, "CUDA-graph replay: total us/step", (t1 - t0) / n * 1e6)
