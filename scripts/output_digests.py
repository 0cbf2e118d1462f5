"""SHA-256 of every output tensor of one seeded LSTM forward + BPTT (BASELINE config-2 history shape) and of one Model
forward + backward at BASELINE config 2 (dropout 0), computed with the nnr_b200 package of the tree given by --root.

Two builds compute the same thing when their digests are equal:
    python scripts/output_digests.py --root TREE_A > a.json; python scripts/output_digests.py --root TREE_B > b.json"""
import argparse, hashlib, json, math, os, sys

ap = argparse.ArgumentParser()
ap.add_argument('--root', default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument('--hidden', type=int, default=200)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))
import torch
import nnr_b200
from nnr_b200 import ops
from nnr_b200.synthetic import SyntheticMIND, batch_args
from nnr_b200.trainer import negative_log_softmax


def sha(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


dev = torch.device('cuda:0')
Hd, N, L = args.hidden, 3520, 128
out = {'root': os.path.basename(os.path.abspath(args.root)), 'hidden_dim': Hd}
g = torch.Generator().manual_seed(0)
lens = torch.exp(torch.randn(N, generator=g) * 0.8 + math.log(40.0) - 0.32).round().clamp_(1, L).long()
lens[: N // 50] = L
ntok = int(lens.sum())
len_ = lens.to(torch.int32).to(dev)
off = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)]).to(torch.int32).to(dev)
order = torch.sort(lens, descending=True, stable=True)[1].to(torch.int32).to(dev)
gx = (torch.randn(ntok, 8 * Hd, generator=g) * 0.5).to(dev)
w_hh = (torch.randn(2, 4 * Hd, Hd, generator=g) / math.sqrt(Hd)).to(dev)
h, cst, cn = torch.zeros(ntok, 2 * Hd, device=dev), torch.zeros(ntok, 2 * Hd, device=dev), torch.zeros(N, 2 * Hd, device=dev)
dh, dcn = (torch.randn(ntok, 2 * Hd, generator=g) * 0.1).to(dev), (torch.randn(N, 2 * Hd, generator=g) * 0.1).to(dev)
ops.lstm_fwd(gx, w_hh, len_, off, order, N, L, Hd, h, cst, cn)
out.update(lstm_h=sha(h), lstm_c_stash=sha(cst), lstm_c_n=sha(cn), lstm_gates=sha(gx))
ops.lstm_bwd(gx, cst, w_hh, len_, off, order, N, L, Hd, dh, dcn)
out.update(lstm_dgx=sha(gx))

sys.argv = [sys.argv[0]]
import bench
a = bench.parse()
cfg = bench.make_config(a)
cfg.hidden_dim = Hd
cfg.dropout_rate = 0.0
syn = SyntheticMIND(news_num=20000, vocabulary_size=a.vocab, lengths=a.lengths, seed=0)
cfg.pretrained_word_embedding = syn.word_table()
torch.manual_seed(0)
model = nnr_b200.Model(cfg); model.initialize(); model.to(dev).train()
logits = model(*batch_args(syn.batch(a.batch, seed=1), dev))
loss = negative_log_softmax(logits)
loss.backward()
out.update(logits=sha(logits), loss=sha(loss))
for k, p in model.named_parameters():
    if p.grad is not None:
        out['grad.' + k] = sha(p.grad)
print(json.dumps(out))
