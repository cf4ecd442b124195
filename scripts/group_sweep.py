import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import awesome_b200 as A
import bench as B
dev = torch.device("cuda", 0)
un = B.synth_unaries(42).to(dev)
grid = A.GridSpecHost("linspace", 1, B.H, B.W)
for G in (1, 2, 3, 4, 6, 8):
    mg = A.NumberBasedMultiPriorModule(prior_type=A.ConvexNextNet, prior_args=dict(n_hidden=130, in_features=2, n_hidden_layers=2, precision="f16"), min_priors=G).to(dev)
    tg = torch.stack([torch.roll(un, shifts=(11 * k, 23 * k), dims=(0, 1)) for k in range(G)])
    f = mg.make_fitter(grid, tg, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    ms = B._time_fitter(f, 200)
    print(G, round(ms, 4), "ms/step", round(ms / G, 4), "per frame", round(G * B.N_PIX / ms / 1e6, 1), "Mpx/s", flush=True)
    del f, mg
