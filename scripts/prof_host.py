import cProfile, pstats, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import CFG, make_graphs
graphs = make_graphs(list(range(25)), 143107, 1_500_000)
import torch
from meta_gcn_b200 import dist as mdist, functional as F
from meta_gcn_b200.data import GraphBatch
from meta_gcn_b200.gcn_meta.models import GCNModel
dev = torch.device("cuda")
torch.cuda.set_stream(torch.cuda.Stream(dev))
host = GraphBatch.from_data_list(graphs).with_int32_indices()
torch.manual_seed(0)
model = GCNModel(**CFG).to(dev)
reducer = mdist.FlatGradientReducer(model.parameters())
b = host.to(dev); b.x = b.x.contiguous()
def fwdbwd():
    reducer.zero()
    out = model(b.x[:, 0].view(-1, 1), b.edge_index, deg_K=b.x[:, 1])
    loss = F.cross_entropy(out, b.y.long(), "sum")
    loss.backward()
    return loss
for _ in range(3): fwdbwd()
torch.cuda.synchronize()
pr = cProfile.Profile()
pr.enable()
t0 = time.perf_counter()
for _ in range(5): fwdbwd()
t1 = time.perf_counter()
pr.disable()
torch.cuda.synchronize()
print("host ms per fwd+bwd enqueue:", (t1 - t0) / 5 * 1e3)
st = pstats.Stats(pr); st.sort_stats("tottime").print_stats(25)
