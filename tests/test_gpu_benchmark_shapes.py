"""GPU parity at the shapes bench.py actually times (BASELINE.json C2 / C3 / C4), against the CPU oracle.

The small-batch tests in test_gpu_model.py / test_gpu_train.py pick other tiles, split-K factors and slab modes than the
64-member 128x128 launches of the benchmark; these tests run the benchmarked launch shapes themselves:

  C2  score of 64 members, 128x128, Cin = 2 (the EM ensemble's network evaluation), every tensor-core precision
  C3  128x128, Cin = 7 + season labels, predictor-corrector, bf16 (and the fp32-class modes), 8 members x 3 steps
  C4  DSM loss + every parameter gradient at 128x128, train-mode BatchNorm, bf16 and the fp32-class modes, at batch 8 and at
      bench.py's batch of 64 (where five bf16 weight gradients of the decoder take the halo-slab kernel);
      and the bf16 step at batch 64 replayed from its CUDA graphs, bit for bit

bf16 has no reference implementation to be "equal" to (the reference is fp32-only, sbgm/training.py:325-343 has its AMP branch
commented out); its yardstick is the oracle itself run under `torch.autocast(bfloat16)`: the kernels' bf16 error must stay
within 2x of what autocast does to the reference arithmetic on the same inputs.
"""
import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# per-call score gate: 1e-3 in the fp32-class modes (north star); bf16 at the survey's 2e-2
SCORE_TOL = {"bf16x3": 1e-3, "fp16x2": 1e-3, "bf16": 2e-2}


def _cuda(v):
    return None if v is None else v.to(DEV)


def _build(ck, precision, seed=0):
    from oracle.synth import config_for, synth_state_dict
    from sbgm_danra_b200._smoke import build_model
    cfg = config_for(**ck)
    sd = synth_state_dict(cfg, seed)
    return build_model(cfg, sd, precision, DEV), cfg, sd


@pytest.fixture(scope="module")
def c2_oracle():
    """Oracle score of the C2 launch shape: 64 members sharing one conditioning image, each at its own time."""
    from oracle import score_ref
    from oracle.synth import config_for, synth_batch, synth_state_dict
    cfg = config_for(n_lr=1)
    sd = synth_state_dict(cfg, 0)
    b = synth_batch(batch=64, size=128, n_lr=1, shared_cond=True)
    with torch.no_grad():
        want = score_ref.score_forward(sd, cfg, *b.model_args())
    return b, want


@pytest.mark.parametrize("precision", ["bf16x3", "fp16x2", "bf16"])
def test_c2_score_64_members_128x128_matches_oracle(c2_oracle, precision):
    b, want = c2_oracle
    net, _, _ = _build(dict(n_lr=1), precision)
    with torch.no_grad():
        got = net(*[_cuda(v) for v in b.model_args()]).cpu()
    per = [rel_l2(got[i], want[i]) for i in range(got.shape[0])]
    err = rel_l2(got, want)
    print(f"C2 score, 64 x 128x128 [{precision}]: rel-L2 {err:.3e}, worst member {max(per):.3e}")
    assert err < SCORE_TOL[precision] and max(per) < SCORE_TOL[precision]


@pytest.mark.parametrize("precision", ["bf16x3", "fp16x2", "bf16"])
def test_c2_sampler_step_at_benchmark_shape_matches_oracle(c2_oracle, precision):
    """Two Euler-Maruyama steps of the 64-member call bench.py times (graph-captured step, shared conditioning, label-free
    time-projection table) against the oracle's sampler on the same Philox noise."""
    from oracle import samplers_ref, score_ref
    from oracle.synth import config_for, synth_state_dict
    from sbgm_danra_b200 import score_sampling as ss
    from sbgm_danra_b200.score_unet import diffusion_coeff_fn, marginal_prob_std_fn
    b, _ = c2_oracle
    net, cfg, sd = _build(dict(n_lr=1), precision)
    ss.manual_seed(77)
    got = ss.Euler_Maruyama_sampler(net, marginal_prob_std_fn, diffusion_coeff_fn, batch_size=64, num_steps=2, device=DEV,
                                    img_size=128, cond_img=_cuda(b.cond_img)).cpu()
    score = lambda x, t: score_ref.score_forward(sd, cfg, x, t, None, b.cond_img)
    with torch.no_grad():
        want = samplers_ref.euler_maruyama(score, score_ref.marginal_prob_std, score_ref.diffusion_coeff, 64, 2, img_size=128,
                                           noise=samplers_ref.philox_noise(77))
    err = rel_l2(got, want)
    print(f"C2 EM 2 steps, 64 x 128x128 [{precision}]: rel-L2 {err:.3e}")
    assert err < 2 * SCORE_TOL[precision]
    ss.clear_sampler_cache()


@pytest.mark.parametrize("precision", ["bf16", "bf16x3", "fp16x2"])
def test_c3_pc_sampler_128x128_cin7_seasons_matches_oracle(precision):
    """BASELINE C3 as benchmarked: 128x128, two LR fields + land-sea mask + topography (Cin = 7), season labels,
    predictor-corrector (2 evaluations + batch-mean Langevin step per step): 8 members x 3 steps against
    oracle.samplers_ref.predictor_corrector on the same Philox draws."""
    from oracle import samplers_ref, score_ref
    from oracle.synth import synth_batch
    from sbgm_danra_b200 import score_sampling as ss
    from sbgm_danra_b200.score_unet import diffusion_coeff_fn, marginal_prob_std_fn
    ck = dict(n_lr=2, geo=True, seasons=True)
    net, cfg, sd = _build(ck, precision)
    b = synth_batch(batch=8, size=128, shared_cond=True, **ck)
    ss.manual_seed(31)
    got = ss.pc_sampler(net, marginal_prob_std_fn, diffusion_coeff_fn, batch_size=8, num_steps=3, snr=0.16, device=DEV,
                        img_size=128, y=_cuda(b.y), cond_img=_cuda(b.cond_img), lsm_cond=_cuda(b.lsm_cond),
                        topo_cond=_cuda(b.topo_cond)).cpu()
    score = lambda x, t: score_ref.score_forward(sd, cfg, x, t, b.y, b.cond_img, b.lsm_cond, b.topo_cond)
    with torch.no_grad():
        want = samplers_ref.predictor_corrector(score, score_ref.marginal_prob_std, score_ref.diffusion_coeff, 8, 3,
                                                img_size=128, noise=samplers_ref.philox_noise(31))
    err = rel_l2(got, want)
    print(f"C3 PC 3 steps, 8 x 128x128 Cin=7 + seasons [{precision}]: rel-L2 {err:.3e}")
    assert err < 2 * SCORE_TOL[precision]
    ss.clear_sampler_cache()


def _oracle_dsm(cfg, sd, b, seed, bn_train, autocast=False):
    from oracle import philox_ref, score_ref
    sdo = {k: (v.clone().requires_grad_() if v.is_floating_point() and not k.endswith(("running_mean", "running_var", ".W")) else v.clone())
           for k, v in sd.items()}
    n = b.x.shape[0]
    u = torch.from_numpy(philox_ref.uniform(n, seed, philox_ref.DRAW_DSM_T))
    z = torch.from_numpy(philox_ref.normal(b.x.numel(), seed, philox_ref.DRAW_DSM_Z)).reshape(b.x.shape)
    with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
        loss = score_ref.dsm_loss(sdo, cfg, b.x, u * (1.0 - 1e-3) + 1e-3, z, b.y, b.cond_img, b.lsm_cond, b.topo_cond, b.sdf_cond,
                                  bn_train=bn_train)
    loss.backward()
    return loss.detach().float(), {k: v.grad.float() for k, v in sdo.items() if torch.is_tensor(v) and v.requires_grad and v.grad is not None}


def _ours_dsm(cfg, sd, b, seed, precision, train):
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    net = build_model(cfg, sd, precision, DEV)
    net.train(train)
    score_sampling.manual_seed(seed)
    loss = loss_fn(net, _cuda(b.x), marginal_prob_std_fn, y=_cuda(b.y), cond_img=_cuda(b.cond_img), lsm_cond=_cuda(b.lsm_cond),
                   topo_cond=_cuda(b.topo_cond), sdf_cond=_cuda(b.sdf_cond))
    loss.backward()
    return loss.detach().cpu(), {k: p.grad.cpu() for k, p in net.named_parameters() if p.grad is not None}


def _whole(g, ref, keys):
    return rel_l2(torch.cat([g[k].reshape(-1) for k in keys]), torch.cat([ref[k].reshape(-1) for k in keys]))


def _c4_oracle(batch):
    """C4 shape per sample (128x128, Cin = 7 + seasons, SDF weighting, train-mode BatchNorm): fp32 oracle loss and gradients,
    and the same under CPU bf16 autocast (the yardstick of the bf16 mode)."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    ck = dict(n_lr=2, geo=True, seasons=True)
    cfg = config_for(**ck)
    sd = synth_state_dict(cfg)
    b = synth_batch(batch=batch, size=128, **ck)
    loss, grads = _oracle_dsm(cfg, sd, b, 2025, True)
    loss_ac, grads_ac = _oracle_dsm(cfg, sd, b, 2025, True, autocast=True)
    keys = sorted(grads)
    return cfg, sd, b, loss, grads, keys, abs(float(loss_ac - loss)) / abs(float(loss)), _whole(grads_ac, grads, keys)


@pytest.fixture(scope="module")
def c4_oracle():
    return _c4_oracle(8)


@pytest.fixture(scope="module")
def c4_oracle_batch64():
    return _c4_oracle(64)


def _check_c4(oracle, precision):
    cfg, sd, b, loss, grads, keys, ac_loss_err, ac_grad_err = oracle
    got_loss, got = _ours_dsm(cfg, sd, b, 2025, precision, True)
    assert sorted(got) == keys, "the set of parameters that receive a gradient differs from the reference's"
    lerr = abs(float(got_loss - loss)) / abs(float(loss))
    gerr = _whole(got, grads, keys)
    worst = max((rel_l2(got[k], grads[k]), k) for k in keys)
    print(f"C4 DSM {b.x.shape[0]} x 128x128 [{precision}]: loss rel {lerr:.2e}, whole-gradient rel-L2 {gerr:.3e}, worst {worst[1]} "
          f"{worst[0]:.2e}; autocast-bf16 oracle: loss rel {ac_loss_err:.2e}, whole-gradient {ac_grad_err:.3e}")
    if precision == "bf16":
        assert lerr < max(2 * ac_loss_err, 1e-3) and gerr < 2 * ac_grad_err
    else:
        assert lerr < 1e-4 and gerr < 1e-3 and worst[0] < 2e-2      # worst = a 128-element BatchNorm bias (measured 8.5e-3)


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_c4_dsm_loss_and_gradient_128x128_batch8_matches_oracle(c4_oracle, precision):
    _check_c4(c4_oracle, precision)


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_c4_dsm_loss_and_gradient_128x128_batch64_matches_oracle(c4_oracle_batch64, precision):
    """The batch bench.py times: in bf16 the weight gradients of the conv_up of decoder blocks 1-3, of decoder block 3's conv and
    of the final conv_up run the halo-slab kernel."""
    _check_c4(c4_oracle_batch64, precision)


def test_c4_graph_replay_at_batch64_is_bitwise_reproducible():
    """The step bench.py times (bf16, train mode, batch 64): steps 1-2 run the eager engine, steps 3-5 replay the captured forward
    and backward CUDA graphs.  Same inputs, same Philox seed, no optimizer step -> the loss and every gradient equal step 1's bit
    for bit.  In train mode BatchNorm normalises with batch statistics, so the running buffers that move between steps do not
    enter the gradients."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    ck = dict(n_lr=2, geo=True, seasons=True)
    cfg = config_for(**ck)
    net = build_model(cfg, synth_state_dict(cfg), "bf16", DEV).train()
    b = synth_batch(batch=64, size=128, **ck)
    snaps = []
    for step in range(5):
        score_sampling.manual_seed(3)
        net.zero_grad(set_to_none=True)
        loss = loss_fn(net, _cuda(b.x), marginal_prob_std_fn, y=_cuda(b.y), cond_img=_cuda(b.cond_img), lsm_cond=_cuda(b.lsm_cond),
                       topo_cond=_cuda(b.topo_cond), sdf_cond=_cuda(b.sdf_cond))
        loss.backward()
        snaps.append((loss.item(), {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}))
    runner = next(iter(net._train_runners.values()))
    assert runner.g_fwd is not None and runner.g_bwd is not None, "the step was never captured"
    for loss_k, grads_k in snaps[1:]:
        assert loss_k == snaps[0][0]
        assert grads_k.keys() == snaps[0][1].keys()
        for k in grads_k:
            assert torch.equal(grads_k[k], snaps[0][1][k]), k


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_bf16_training_gradients_within_2x_of_autocast_oracle(mode):
    """The case VERDICT r1 flagged (batch 4, 32x32: whole-gradient rel-L2 1.4e-1 in bf16, train-mode BatchNorm over 4..16
    values per channel): the oracle under torch.autocast(bfloat16) is just as far from fp32 (1.7e-1 here), i.e. it is bf16
    at this sample size, not a kernel bug.  Gate: within 2x of autocast's error on the same inputs and draws."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    ck = dict(n_lr=2, geo=True, seasons=True)
    cfg = config_for(**ck)
    sd = synth_state_dict(cfg)
    b = synth_batch(batch=4, size=32, **ck)
    train = mode == "train"
    loss, grads = _oracle_dsm(cfg, sd, b, 2024, train)
    _, grads_ac = _oracle_dsm(cfg, sd, b, 2024, train, autocast=True)
    keys = sorted(grads)
    _, got = _ours_dsm(cfg, sd, b, 2024, "bf16", train)
    ours, ac = _whole(got, grads, keys), _whole(grads_ac, grads, keys)
    print(f"bf16 gradients, batch 4 / 32x32 / {mode}: kernels {ours:.3e} vs autocast-bf16 oracle {ac:.3e} (both against the fp32 oracle)")
    assert ours < 2 * ac
