import cProfile, pstats, os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import iea_gan_b200 as P
from iea_gan_b200.default_config import shipped_config
from iea_gan_b200.train_step import make_train_step, NormalNoise, EMA
cfg = shipped_config(H_base=1, device="cuda", clip_norm=1e9)
torch.manual_seed(0)
G, D = P.Generator(**cfg).cuda(), P.Discriminator(**cfg).cuda()
G.train(); D.train()
ev = 1; n = 40 * ev
train = make_train_step(G, D, P.G_D(G, D), NormalNoise(n, cfg["dim_z"], "cuda"), dict(cfg, batch_size=n))
x = torch.rand(n, 1, 256, 256, device="cuda") * 2 - 1
y = torch.arange(40, device="cuda").repeat(ev)
for _ in range(5): train(x, y)
torch.cuda.synchronize()
pr = cProfile.Profile(); pr.enable()
for _ in range(5): train(x, y)
torch.cuda.synchronize()
pr.disable()
st = pstats.Stats(pr); st.sort_stats("tottime").print_stats(28)
