"""Scratch diagnostics: CUDA path vs oracle on the fixture and a small synthetic sample (run under gpurun)."""
import sys, time, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import polee_b200 as pb
from polee_b200 import synth
from oracle import polee_oracle as O

g = 'tests/golden/'
colptr = np.fromfile(g + 'fixture_colptr.u32', np.uint32); rowval = np.fromfile(g + 'fixture_rowval.u32', np.uint32)
nzval = np.fromfile(g + 'fixture_nzval.f32', np.float32); eff = np.fromfile(g + 'fixture_efflens.f32', np.float32)
pi = np.fromfile(g + 'fixture_prep_node_parent_idxs.i32', np.int32); js = np.fromfile(g + 'fixture_prep_node_js.i32', np.int32)
m, n = 19743, 313
sample = pb.RNASeqSample(m, n, colptr, rowval, nzval, eff)

def rel(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))

def check(sample, pi, js, K, tag):
    m, n = sample.m, sample.n
    print('==', tag, 'm', m, 'n', n, 'nnz', len(sample.rowval), 'K', K)
    M = O.Model(m, n, sample.colptr, sample.rowval, sample.nzval)
    rng = np.random.default_rng(0)
    h = pb.Handle(num_mc_samples=K, gradonly=False, noise_mode=1, num_steps=3)
    h.set_sample(sample); h.set_tree(pi, js)
    # loglik
    xs = rng.dirichlet(np.ones(n), K).astype(np.float32).clip(1e-10)
    lp, gg = h.loglik_grad(xs, gradonly=False)
    for k in range(K):
        lpo, go = M.log_likelihood(xs[k], gradonly=False)
        print('  loglik k', k, 'lp rel', abs(lp[k] - lpo) / abs(lpo), 'g rel', rel(gg[k], go), 'ident', xs[k].astype(np.float64) @ gg[k] / m)
    w = h.frag_prob_recip(xs[0]); M.log_likelihood(xs[0]); print('  w rel', rel(w, 1 / M.frag_probs))
    # tree
    t = O.PTT(pi, js)
    ys = rng.uniform(0.01, 0.99, (K, n - 1))
    x_d, ladj_d = h.ptt_transform(ys, True)
    xg = rng.normal(size=(K, n)) * 1000
    yg_d = h.ptt_transform_gradients(ys, xg, True)
    yg_d2 = h.ptt_transform_gradients(ys, xg, False)
    for k in range(K):
        x_o, ladj_o = t.transform(ys[k], True)
        yg_o = t.transform_gradients(ys[k], xg[k])
        yg_o2 = t.transform_gradients_no_ladj(ys[k], xg[k])
        print('  tree k', k, 'x biteq', np.array_equal(x_d[k], x_o), 'ladj rel', abs(ladj_d[k] - ladj_o) / abs(ladj_o),
              'ygrad biteq', np.array_equal(yg_d[k], yg_o), rel(yg_d[k], yg_o), 'noladj', rel(yg_d2[k], yg_o2.astype(np.float32)))
    # one step of draws
    mu0, om0, al0 = h.get_params()
    al0 = (rng.normal(size=n - 1) * 0.1).astype(np.float32); h.set_params(mu0, om0, al0)
    zs0 = rng.normal(size=(K, n - 1)).astype(np.float32)
    d = h.lsn_draws(zs0)
    mg = np.zeros(n - 1, np.float32); og = np.zeros(n - 1, np.float32); ag = np.zeros(n - 1, np.float32)
    el = 0
    for k in range(K):
        o = O.lsn_draw(m, n, sample.colptr, sample.rowval, sample.nzval, sample.effective_lengths, pi, js, mu0, om0, al0, zs0[k], gradonly=False)
        print('  draw k', k, 'xs', rel(d['xs'][k], o['xs']), 'ys', rel(d['ys'][k], o['ys']), 'xgrad', rel(d['x_grad'][k], o['x_grad']),
              'ygrad max abs', np.abs(d['y_grad'][k] - o['y_grad']).max(), 'scale', np.abs(o['y_grad']).max())
        mg += o['mu_grad']; og += o['omega_grad']; ag += o['alpha_grad']; el += o['elbo']
    print('  grads mu', np.abs(d['mu_grad'] - mg / K).max(), np.abs(mg / K).max(), 'omega', np.abs(d['omega_grad'] - og / K).max(), np.abs(og/K).max(),
          'alpha', np.abs(d['alpha_grad'] - ag / K).max(), np.abs(ag/K).max(), 'elbo', d['elbo'], el / K)
    h.close()

check(sample, pi, js, 6, 'fixture')
check(sample, pi, js, 1, 'fixture K=1')
check(sample, *pb.api.sequential_tree(n), 2, 'fixture sequential tree')
s = synth.make_sample(200000, 8000, seed=3)
ns = synth.to_numpy_sample(s)
sm = pb.RNASeqSample(ns['m'], ns['n'], ns['colptr'], ns['rowval'], ns['nzval'], ns['efflens'])
check(sm, *synth.balanced_tree(8000, s['gene_sizes'].numpy()), 8, 'synthetic 200k x 8k')

# full fit with injected noise vs oracle
steps, K = 60, 6
rng = np.random.default_rng(1)
noise = rng.normal(size=(steps, K, n - 1)).astype(np.float32)
t0 = time.time(); ro = O.fit_lsn_ptt(m, n, colptr, rowval, nzval, eff, pi, js, num_steps=steps, num_mc_samples=K, noise=noise, gradonly=False, elbo_fix=True); t_or = time.time() - t0
t0 = time.time(); rd = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), sample, tree_topology=(pi, js), num_steps=steps, num_mc_samples=K, noise=noise, gradonly=False, want_elbo=True); t_d = time.time() - t0
for key in ('mu', 'omega', 'alpha'):
    print('fit', key, 'max abs diff', np.abs(rd[key] - ro[key]).max(), 'scale', np.abs(ro[key]).max())
print('elbo first/last', rd['elbo'][:2], ro['elbo'][:2], rd['elbo'][-1], ro['elbo'][-1], 'oracle s', t_or, 'device s', t_d)
t0 = time.time(); rd = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), sample, tree_topology=(pi, js)); print('default 500-step fit s', time.time() - t0)
mu_ref = np.fromfile(g + 'fixture_prep_mu.f32', np.float32); print('corr mu vs reference prep.h5', np.corrcoef(rd['mu'], mu_ref)[0, 1])
xo = O.fit_optimize_ptt(m, n, colptr, rowval, nzval, eff, 100)
h = pb.Handle(approx=1, num_steps=100); h.set_sample(sample); x_dev = h.fit_optimize_ptt(); h.close()
print('optimize_ptt rel', rel(x_dev, xo), x_dev.sum(), xo.sum())
# hsb
l, r, f = pb.make_inverse_ptt_params(pi, js)
yl = rng.normal(0, 2, (5, n - 1)).astype(np.float32)
xa = pb.hsb(yl, l, r, f); xb = O.hsb(yl, l, r, f, impl='ref' if O.ref_lib() else 'oracle')
print('hsb biteq', np.array_equal(xa, xb), rel(xa, xb))
ya, la = pb.inv_hsb(xb, l, r, f); yb, lb = O.inv_hsb(xb, l, r, f, impl='ref' if O.ref_lib() else 'oracle')
print('inv_hsb y biteq', np.array_equal(ya, yb), 'ladj biteq', np.array_equal(la, lb), la.ravel(), lb.ravel())
yg = rng.normal(size=yb.shape); lg = rng.normal(size=(5, 1)).astype(np.float32)
ba = pb.inv_hsb_grad(yg, lg, yb, lb, l, r, f); bb = O.inv_hsb_grad(yg, lg, yb, lb, l, r, f, impl='ref' if O.ref_lib() else 'oracle')
print('inv_hsb_grad biteq', np.array_equal(ba, bb), rel(ba, bb))
