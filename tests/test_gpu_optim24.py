"""The fused 2:4 optimizer step on the GPU (spfy_optim24_step, SGD24, AdamW24).

Byte checks: after a step, comp.vals equals spfy_recompress24 of the new master and comp_t.vals / op_t.vals equal
spfy_transpose24(_conv) of the new comp, byte for byte; the metadata never changes; master and state are +0 at every
pruned position.  Numerics: master and state against an fp64 evaluation of torch's formula on the same fp32 inputs,
within 2^-20 of the magnitudes of the terms (a few fp32 roundings), and ten steps against torch's own optimizer plus
refresh() within 1e-5 * max|p|."""
import copy
import dataclasses

import pytest
import torch

pytestmark = pytest.mark.gpu

U20 = 2.0 ** -20
# (m, c, k, stride, pad): 1x1 s1, 3x3 s1, 3x3 s2, 1x1 s2, 7x7 s3 with c != m
CONVS = [(64, 64, 1, 1, 0), (64, 64, 3, 1, 1), (128, 64, 3, 2, 1), (128, 64, 1, 2, 0), (128, 64, 7, 3, 3)]
RULES = {
    "sgd": ("sgd", dict(lr=0.05)),
    "sgd_momentum_dampening": ("sgd", dict(lr=0.05, momentum=0.9, dampening=0.25)),
    "sgd_nesterov_wd": ("sgd", dict(lr=0.05, momentum=0.9, nesterov=True, weight_decay=0.01)),
    "adamw": ("adamw", dict(lr=1e-2, betas=(0.8, 0.95), eps=1e-6, weight_decay=0.05)),
}


def make_layers(spfy, cuda, dtype, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    layers = [spfy.Linear24.from_dense(torch.randn(200, 208, generator=g).to(cuda), torch.randn(200, generator=g).to(cuda),
                                       dtype=dtype)]
    for m, c, k, s, p in CONVS:
        layers.append(spfy.Conv2d24.from_dense(torch.randn(m, c, k, k, generator=g).to(cuda),
                                               torch.randn(m, generator=g).to(cuda), stride=s, padding=p, dtype=dtype))
    return layers


def w2d(layer):
    return layer._w2d() if hasattr(layer, "_w2d") else layer.weight


def mask_of(layer):
    return w2d(layer).detach() != 0  # from_dense keeps no zero in a kept position of randn weights


def twin(spfy, layer):
    """an independent copy of a 2:4 layer: master, bias and both compressed operands cloned"""
    comp = dataclasses.replace(layer.comp, vals=layer.comp.vals.clone(), meta=layer.comp.meta.clone())
    b = layer.bias.detach().clone() if layer.bias is not None else None
    if isinstance(layer, spfy.Conv2d24):
        op_t = dataclasses.replace(layer.op_t, vals=layer.op_t.vals.clone(), meta=layer.op_t.meta.clone())
        return spfy.Conv2d24(layer.weight.detach().clone(memory_format=torch.channels_last), b, comp, op_t, layer.dtype,
                             layer.stride, layer.padding)
    comp_t = dataclasses.replace(layer.comp_t, vals=layer.comp_t.vals.clone(), meta=layer.comp_t.meta.clone())
    return spfy.Linear24(layer.weight.detach().clone(), b, comp, comp_t, layer.dtype)


def operand_refs(spfy, layer):
    """(vals, transposed vals) that spfy_recompress24 and spfy_transpose24(_conv) make from the current master"""
    comp = dataclasses.replace(layer.comp, vals=torch.empty_like(layer.comp.vals))
    comp.vals.copy_(layer.comp.vals)  # the padding bytes, which recompress24 rewrites as +0
    spfy.recompress24(w2d(layer).detach(), comp)
    if isinstance(layer, spfy.Conv2d24):
        vt = spfy.transpose24_conv(comp, layer.kh, layer.kw, layer.stride, layer.padding).vals
    else:
        vt = spfy.transpose24(comp).vals
    return comp.vals, vt


def vals_t_of(layer):
    return layer.op_t.vals if hasattr(layer, "op_t") else layer.comp_t.vals


def metas_of(layer):
    return layer.comp.meta.clone(), (layer.op_t.meta if hasattr(layer, "op_t") else layer.comp_t.meta).clone()


def set_grads(layers, seed, poison=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    g_poison = torch.Generator(device="cpu").manual_seed(seed + 1)  # the gradients do not depend on `poison`
    for layer in layers:
        for p in (layer.weight, layer.bias):
            gr = torch.randn(p.shape, generator=g).to(p.device)
            p.grad = gr.contiguous(memory_format=torch.channels_last) if p.dim() == 4 else gr
        if poison:
            pruned = ~mask_of(layer)
            g2 = layer.weight.grad.permute(0, 2, 3, 1).reshape(layer.m, -1) if hasattr(layer, "op_t") else layer.weight.grad
            bad = torch.where(torch.rand(g2.shape, generator=g_poison).to(g2.device) < 0.5, float("nan"), float("inf"))
            g2[pruned] = bad[pruned]


def make_opt(spfy, rule, params):
    kind, kw = RULES[rule]
    return spfy.SGD24(params, **kw) if kind == "sgd" else spfy.AdamW24(params, **kw)


def torch_opt(rule, params):
    kind, kw = RULES[rule]
    return torch.optim.SGD(params, **kw) if kind == "sgd" else torch.optim.AdamW(params, **kw)


def grad2d(layer):
    gr = layer.weight.grad
    return gr.permute(0, 2, 3, 1).reshape(layer.m, -1) if hasattr(layer, "op_t") else gr


def fp64_step(rule, p, g, st, first, t):
    """torch's update in fp64 on fp32 inputs: (p, {state}, {bound})"""
    kind, kw = RULES[rule]
    p, g = p.double(), g.double()
    st = {k: st.get(k, torch.zeros_like(p)) for k in ("momentum_buffer", "exp_avg", "exp_avg_sq")}
    if kind == "sgd":
        lr, mom, damp, wd, nest = kw["lr"], kw.get("momentum", 0.0), kw.get("dampening", 0.0), kw.get("weight_decay", 0.0), \
            kw.get("nesterov", False)
        gg, gmag = g + wd * p, g.abs() + wd * p.abs()
        out, bnd = {}, {}
        if mom:
            b0 = st["momentum_buffer"].double()
            buf = gg if first else b0 * mom + (1 - damp) * gg
            bmag = gmag if first else b0.abs() * mom + (1 - damp) * gmag
            out["momentum_buffer"], bnd["momentum_buffer"] = buf, U20 * bmag
            gg, gmag = (gg + mom * buf, gmag + mom * bmag) if nest else (buf, bmag)
        return p - lr * gg, out, U20 * (p.abs() + lr * gmag), bnd
    lr, (b1, b2), eps, wd = kw["lr"], kw["betas"], kw["eps"], kw["weight_decay"]
    m0, v0 = st["exp_avg"].double(), st["exp_avg_sq"].double()
    p1 = p * (1 - lr * wd)
    m = m0 + (1 - b1) * (g - m0)
    v = v0 * b2 + (1 - b2) * g * g
    ss, bc2 = lr / (1 - b1 ** t), (1 - b2 ** t) ** 0.5
    denom = v.sqrt() / bc2 + eps
    upd = ss * m / denom
    bnd_m = U20 * (b1 * m0.abs() + (1 - b1) * g.abs())
    return p1 - upd, {"exp_avg": m, "exp_avg_sq": v}, U20 * (p.abs() + upd.abs() + ss * bnd_m / denom * 2 ** 20), \
        {"exp_avg": bnd_m, "exp_avg_sq": U20 * v}


def check_bound(got, ref, bound, what):
    err = (got.double() - ref).abs()
    bad = ~(err <= bound)
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} elements outside the bound, worst {float((err / bound).max())}"


def state2d(layer, s):
    return s.permute(0, 2, 3, 1).reshape(layer.m, -1) if s.dim() == 4 else s


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("rule", list(RULES))
def test_step_bytes_and_fp64(spfy, cuda, dtype, rule):
    """three steps (the first and later ones) of every item kind: operands byte-equal to recompress24 / transpose24(_conv)
    of the new master, metadata untouched, +0 at pruned positions, master and state within the fp64 bound; a gradient
    poisoned with NaN / Inf at pruned positions gives the same bytes"""
    layers = make_layers(spfy, cuda, dtype)
    clean = [twin(spfy, layer) for layer in layers]
    metas = [metas_of(layer) for layer in layers]
    masks = [mask_of(layer) for layer in layers]
    opt = make_opt(spfy, rule, [p for layer in layers for p in layer.parameters()])
    opt_clean = make_opt(spfy, rule, [p for layer in clean for p in layer.parameters()])
    for step in range(3):
        set_grads(layers, 100 + step, poison=True)
        set_grads(clean, 100 + step)
        before = [(w2d(layer).detach().clone(), grad2d(c).clone(),
                   {k: state2d(layer, v).clone() for k, v in opt.state[layer.weight].items() if k != "step"})
                  for layer, c in zip(layers, clean)]
        opt.step()
        opt_clean.step()
        for i, (layer, c, mk, (mm, mt)) in enumerate(zip(layers, clean, masks, metas)):
            what = f"{rule} {dtype} layer {i} step {step}"
            vals, vt = operand_refs(spfy, layer)
            assert torch.equal(layer.comp.vals, vals), what + ": comp.vals"
            assert torch.equal(vals_t_of(layer), vt), what + ": transposed vals"
            assert torch.equal(layer.comp.meta, mm) and torch.equal(metas_of(layer)[1], mt), what + ": meta"
            assert torch.equal(layer.weight.detach(), c.weight.detach()), what + ": poisoned gradient changed the master"
            assert torch.equal(layer.comp.vals, c.comp.vals) and torch.equal(vals_t_of(layer), vals_t_of(c)), what
            w = w2d(layer).detach()
            assert bool((w.view(torch.int32)[~mk] == 0).all()), what + ": master not +0 at pruned positions"
            st = opt.state[layer.weight]
            for k, v in st.items():
                if k != "step":
                    assert bool((state2d(layer, v).view(torch.int32)[~mk] == 0).all()), f"{what}: {k} not +0"
                    assert torch.equal(v, opt_clean.state[c.weight][k]), what + k
            p0, g0, s0 = before[i]
            t = float(st["step"]) if "step" in st else 0.0
            ref_p, ref_s, bnd_p, bnd_s = fp64_step(rule, p0[mk], g0[mk], {k: v[mk] for k, v in s0.items()}, step == 0, t)
            check_bound(w[mk], ref_p, bnd_p, what + ": master")
            for k in ref_s:
                check_bound(state2d(layer, st[k])[mk], ref_s[k], bnd_s[k], f"{what}: {k}")
            assert layer.weight._version == layer._synced_version  # forward needs no refresh()


@pytest.mark.parametrize("rule", list(RULES))
def test_ten_steps_track_torch(spfy, cuda, rule):
    """ten steps with identical gradients: SGD24 / AdamW24 against torch's optimizer plus refresh(), <= 1e-5 max|p|"""
    layers = make_layers(spfy, cuda, torch.float16, seed=3)
    ref = [twin(spfy, layer) for layer in layers]
    opt = make_opt(spfy, rule, [p for layer in layers for p in layer.parameters()])
    opt_ref = torch_opt(rule, [p for layer in ref for p in layer.parameters()])
    for step in range(10):
        set_grads(layers, 200 + step)
        set_grads(ref, 200 + step)
        opt.step()
        opt_ref.step()
        for r in ref:
            r.refresh()
    for i, (layer, r) in enumerate(zip(layers, ref)):
        for p, q in zip(layer.parameters(), r.parameters()):
            tol = 1e-5 * float(q.detach().abs().max())
            assert float((p.detach() - q.detach()).abs().max()) <= tol, (rule, i)


def resnet50_layers(spfy, cuda, g):
    """every ResNet-50 convolution past the stem as a Conv2d24, the stem and every BatchNorm as dense fp32 parameters,
    and a Linear24 fc: the 161 parameter tensors of the model"""
    convs, dense = [], [torch.nn.Parameter(torch.randn(64, 3, 7, 7, generator=g).to(cuda))]
    dense += [torch.nn.Parameter(torch.randn(64, generator=g).to(cuda)) for _ in range(2)]
    cin = 64
    for width, blocks, stride in ((64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)):
        for b in range(blocks):
            s = stride if b == 0 else 1
            specs = [(width, cin, 1, 1, 0), (width, width, 3, s, 1), (4 * width, width, 1, 1, 0)]
            if b == 0:
                specs.append((4 * width, cin, 1, s, 0))
            for m, c, k, st, p in specs:
                convs.append(spfy.Conv2d24.from_dense(torch.randn(m, c, k, k, generator=g).to(cuda) * 0.05, None,
                                                      stride=st, padding=p))
                dense += [torch.nn.Parameter(torch.randn(m, generator=g).to(cuda)) for _ in range(2)]
            cin = 4 * width
    fc = spfy.Linear24.from_dense(torch.randn(1000, 2048, generator=g).to(cuda) * 0.02, torch.randn(1000, generator=g).to(cuda))
    return convs + [fc], dense


def test_resnet50_one_launch_equals_per_parameter_steps(spfy, cuda):
    """one SGD24 step over ResNet-50's 161 parameters is one library launch, runs under sync-debug "error", and writes
    the same bytes as one step() per parameter"""
    g = torch.Generator(device="cpu").manual_seed(11)
    layers, dense = resnet50_layers(spfy, cuda, g)
    params = [p for layer in layers for p in layer.parameters()] + dense
    assert len(params) == 161
    twins = [twin(spfy, layer) for layer in layers]
    dense2 = [torch.nn.Parameter(p.detach().clone()) for p in dense]
    params2 = [p for layer in twins for p in layer.parameters()] + dense2
    opt = spfy.SGD24(params, lr=0.1, momentum=0.9, weight_decay=1e-4)
    opts = [spfy.SGD24([p], lr=0.1, momentum=0.9, weight_decay=1e-4) for p in params2]
    for step in range(2):
        for p, q in zip(params, params2):
            q.grad = torch.randn(p.shape, generator=g).to(cuda).contiguous(
                memory_format=torch.channels_last if p.dim() == 4 and p.is_contiguous(memory_format=torch.channels_last)
                else torch.contiguous_format)
            p.grad = q.grad.clone(memory_format=torch.preserve_format)
        torch.cuda.synchronize()
        n0 = spfy.launch_count()
        torch.cuda.set_sync_debug_mode("error")
        try:
            opt.step()
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert spfy.launch_count() - n0 == 1
        for o in opts:
            o.step()
        for p, q, o in zip(params, params2, opts):
            assert torch.equal(p.detach(), q.detach())
            assert torch.equal(opt.state[p]["momentum_buffer"], o.state[q]["momentum_buffer"])
        for layer, t in zip(layers, twins):
            assert torch.equal(layer.comp.vals, t.comp.vals) and torch.equal(vals_t_of(layer), vals_t_of(t))


def snapshot(layers, opt):
    out = []
    for layer in layers:
        out += [layer.weight.detach().clone(), layer.comp.vals.clone(), vals_t_of(layer).clone()]
        out += [v.clone() for v in opt.state[layer.weight].values()]
    return out


def test_grad_scaler_overflow_skips_then_tracks(spfy, cuda):
    """AdamW24 under torch.amp.GradScaler: a first scale of 2^40 overflows and the step writes nothing (master, state,
    operands and the step count byte-identical) and forward still runs; later steps track a twin stepped on the same
    gradients unscaled on the host side"""
    g = torch.Generator(device="cpu").manual_seed(5)
    lin = spfy.Linear24.from_dense(torch.randn(256, 256, generator=g).to(cuda) * 0.05, torch.zeros(256, device=cuda))
    ref = twin(spfy, lin)
    opt = spfy.AdamW24(lin.parameters(), lr=1e-3)
    opt_ref = spfy.AdamW24(ref.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 40, backoff_factor=2.0 ** -24)
    x = torch.randn(64, 256, generator=g).to(cuda).half()
    target = torch.randn(64, 256, generator=g).to(cuda)
    # give the state something to lose first
    for layer, o in ((lin, opt), (ref, opt_ref)):
        ((layer(x).float() - target) ** 2).mean().backward()
        o.step()
        o.zero_grad()
    for step in range(4):
        before_scale = scaler.get_scale()
        loss = ((lin(x).float() - target) ** 2).mean()
        scaler.scale(loss).backward()
        before = snapshot([lin], opt)
        scaler.step(opt)
        scaler.update()
        opt.zero_grad()
        if step == 0:
            assert all(torch.equal(a, b) for a, b in zip(before, snapshot([lin], opt))), "the skipped step wrote"
            lin(x)  # in sync: no refresh() needed
            continue
        scale = before_scale
        (((ref(x).float() - target) ** 2).mean() * scale).backward()
        for p in ref.parameters():
            p.grad.div_(scale)  # a power of two: exact
        opt_ref.step()
        opt_ref.zero_grad()
        tol = 1e-5 * float(ref.weight.detach().abs().max())
        assert float((lin.weight.detach() - ref.weight.detach()).abs().max()) <= tol, step
        assert float(opt.state[lin.weight]["step"]) == float(opt_ref.state[ref.weight]["step"])


def test_state_dict_round_trip(spfy, cuda):
    """a state_dict saved after 3 steps continues bit for bit in a fresh SGD24, and loads into torch.optim.SGD"""
    layers = make_layers(spfy, cuda, torch.float16, seed=9)
    opt = spfy.SGD24([p for layer in layers for p in layer.parameters()], lr=0.05, momentum=0.9)
    for step in range(3):
        set_grads(layers, 300 + step)
        opt.step()
    sd = copy.deepcopy(opt.state_dict())  # state_dict() holds references to the live state
    a = [twin(spfy, layer) for layer in layers]
    b = [twin(spfy, layer) for layer in layers]
    opt_a = spfy.SGD24([p for layer in a for p in layer.parameters()], lr=0.05, momentum=0.9)
    opt_a.load_state_dict(copy.deepcopy(sd))  # load_state_dict keeps the tensors it is given
    opt_t = torch.optim.SGD([p for layer in b for p in layer.parameters()], lr=0.05, momentum=0.9)
    opt_t.load_state_dict(copy.deepcopy(sd))
    for step in range(3, 5):
        for ls in (layers, a, b):
            set_grads(ls, 300 + step)
        opt.step()
        opt_a.step()
        opt_t.step()
        for layer in b:
            layer.refresh()
    for x, y, z in zip(layers, a, b):
        assert torch.equal(x.weight.detach(), y.weight.detach()) and torch.equal(x.comp.vals, y.comp.vals)
        assert torch.equal(vals_t_of(x), vals_t_of(y))
        assert float((x.weight.detach() - z.weight.detach()).abs().max()) <= 1e-5 * float(z.weight.detach().abs().max())


def test_bottleneck_sgd24_tracks_refresh_flow(spfy, cuda):
    """the bottleneck block of test_bottleneck_sgd_tracks_torch trained with SGD24 and no refresh() gives the losses of
    torch SGD + refresh() within 1e-3 relative over five steps"""
    def build():
        g = torch.Generator(device="cpu").manual_seed(7)
        specs = [(64, 64, 1, 1, 0), (64, 64, 3, 2, 1), (256, 64, 1, 1, 0), (256, 64, 1, 2, 0)]
        convs = [spfy.Conv2d24.from_dense((torch.randn(m, ci, k, k, generator=g) * (2.0 / (ci * k * k)) ** 0.5).to(cuda),
                                          torch.zeros(m, device=cuda), stride=s, padding=p) for m, ci, k, s, p in specs]
        bns = [torch.nn.BatchNorm2d(m).to(cuda) for m, *_ in specs]
        x = torch.randn(8, 64, 16, 16, generator=g).to(cuda).half().contiguous(memory_format=torch.channels_last)
        target = torch.randn(8, 256, 8, 8, generator=g).to(cuda)
        params = [q for cv in convs for q in cv.parameters()] + [q for bn in bns for q in bn.parameters()]
        return convs, bns, x, target, params

    def block(xin, conv, bn):
        h = torch.relu(bn[0](conv[0](xin)))
        h = torch.relu(bn[1](conv[1](h)))
        return torch.relu(bn[2](conv[2](h)) + bn[3](conv[3](xin)))

    convs, bns, x, target, params = build()
    convs_r, bns_r, _, _, params_r = build()
    opt = spfy.SGD24(params, lr=0.05, momentum=0.9)
    opt_r = torch.optim.SGD(params_r, lr=0.05, momentum=0.9)
    for step in range(5):
        opt.zero_grad()
        loss = ((block(x, convs, bns).float() - target) ** 2).mean()
        loss.backward()
        opt.step()
        opt_r.zero_grad()
        loss_r = ((block(x, convs_r, bns_r).float() - target) ** 2).mean()
        loss_r.backward()
        opt_r.step()
        for cv in convs_r:
            cv.refresh()
        assert abs(loss.item() - loss_r.item()) <= 1e-3 * abs(loss_r.item()), (step, loss.item(), loss_r.item())


def test_split_launches_many_groups_and_ragged_dense_items(spfy, cuda):
    """a table of more than 192 items and more than 16 groups takes several launches and writes the bytes of one step()
    per parameter: ResNet-50 with every 2:4 layer in a group of its own, plus dense items that reach the vector tail
    (10 elements), the scalar path (a 7-element view 4 bytes off alignment) and an empty parameter"""
    g = torch.Generator(device="cpu").manual_seed(13)
    layers, dense = resnet50_layers(spfy, cuda, g)
    twins = [twin(spfy, layer) for layer in layers]
    dense2 = [torch.nn.Parameter(p.detach().clone()) for p in dense]

    def ragged(seed):
        gg = torch.Generator(device="cpu").manual_seed(seed)
        out = []
        for _ in range(20):
            out.append(torch.nn.Parameter(torch.randn(10, generator=gg).to(cuda)))
            base = torch.randn(8, generator=gg).to(cuda)
            out.append(torch.nn.Parameter(base[1:]))
        return out + [torch.nn.Parameter(torch.empty(0, device=cuda))]

    extra, extra2 = ragged(1), ragged(1)
    assert extra[1].data_ptr() % 16 == 4
    kw = dict(momentum=0.9, dampening=0.25, weight_decay=1e-3)
    groups = [{"params": list(layer.parameters()), "lr": 0.01 * (1 + i % 7)} for i, layer in enumerate(layers)]
    groups.append({"params": dense + extra, "lr": 0.05})
    opt = spfy.SGD24(groups, **kw)
    params = [p for grp in groups for p in grp["params"]]
    lrs = [grp["lr"] for grp in groups for _ in grp["params"]]
    params2 = [p for layer in twins for p in layer.parameters()] + dense2 + extra2
    assert len(params) == len(params2) > 192 and len(groups) > 16
    opts = [spfy.SGD24([q], lr=lr, **kw) for q, lr in zip(params2, lrs)]
    for step in range(2):
        for p, q in zip(params, params2):
            q.grad = torch.randn(p.shape, generator=g).to(cuda).contiguous(
                memory_format=torch.channels_last if p.dim() == 4 and p.is_contiguous(memory_format=torch.channels_last)
                else torch.contiguous_format)
            p.grad = q.grad.clone(memory_format=torch.preserve_format)
        n0 = spfy.launch_count()
        opt.step()
        assert spfy.launch_count() - n0 > 1
        for o in opts:
            o.step()
        for p, q in zip(params, params2):
            assert torch.equal(p.detach(), q.detach()), step
        for layer, t in zip(layers, twins):
            assert torch.equal(layer.comp.vals, t.comp.vals) and torch.equal(vals_t_of(layer), vals_t_of(t))


def test_grad_scaler_skipped_first_sgd_step_stays_first(spfy, cuda):
    """SGD with dampening under GradScaler: after an overflowing (skipped) first step, the first applied step is torch's
    first step, buf = grad, bit for bit the step of a twin that never saw the skipped one"""
    g = torch.Generator(device="cpu").manual_seed(21)
    lin = spfy.Linear24.from_dense(torch.randn(256, 256, generator=g).to(cuda) * 0.05, torch.zeros(256, device=cuda))
    ref = twin(spfy, lin)
    kw = dict(lr=0.05, momentum=0.9, dampening=0.5)
    opt, opt_ref = spfy.SGD24(lin.parameters(), **kw), spfy.SGD24(ref.parameters(), **kw)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 40, backoff_factor=2.0 ** -24)
    x = torch.randn(64, 256, generator=g).to(cuda).half()
    target = torch.randn(64, 256, generator=g).to(cuda)
    for step in range(4):
        scale = scaler.get_scale()
        scaler.scale(((lin(x).float() - target) ** 2).mean()).backward()
        scaler.step(opt)
        scaler.update()
        opt.zero_grad()
        if step == 0:
            assert scaler.get_scale() < scale  # skipped
            continue
        (((ref(x).float() - target) ** 2).mean() * scale).backward()
        for p in ref.parameters():
            p.grad.div_(scale)  # a power of two: exact
        opt_ref.step()
        opt_ref.zero_grad()
        for p, q in zip(lin.parameters(), ref.parameters()):
            assert torch.equal(p.detach(), q.detach()), step
            assert torch.equal(opt.state[p]["momentum_buffer"], opt_ref.state[q]["momentum_buffer"]), step
        assert torch.equal(lin.comp.vals, ref.comp.vals) and torch.equal(lin.comp_t.vals, ref.comp_t.vals)


@pytest.mark.parametrize("kind", ["sgd", "adamw"])
def test_refused_step_leaves_state_as_it_was(spfy, cuda, kind):
    """a step the library refuses (a gradient 4 bytes off alignment) changes no state: AdamW's step count is not
    advanced and SGD's first step stays pending; the next step equals a twin's first step bit for bit"""
    g = torch.Generator(device="cpu").manual_seed(31)
    lin = spfy.Linear24.from_dense(torch.randn(128, 128, generator=g).to(cuda), None)
    ref = twin(spfy, lin)
    make = (lambda ps: spfy.SGD24(ps, lr=0.05, momentum=0.9, dampening=0.5)) if kind == "sgd" else \
        (lambda ps: spfy.AdamW24(ps, lr=1e-2))
    opt, opt_ref = make(lin.parameters()), make(ref.parameters())
    grad = torch.randn(128, 128, generator=g).to(cuda)
    buf = torch.empty(128 * 128 + 1, device=cuda)
    lin.weight.grad = buf[1:].view(128, 128).copy_(grad)  # the parameter's strides, misaligned
    with pytest.raises(spfy.SpfyError):
        opt.step()
    if kind == "adamw":
        assert float(opt.state[lin.weight]["step"]) == 0.0
    lin.weight.grad = grad.clone()
    ref.weight.grad = grad.clone()
    opt.step()
    opt_ref.step()
    assert torch.equal(lin.weight.detach(), ref.weight.detach()) and torch.equal(lin.comp.vals, ref.comp.vals)
    for k, v in opt_ref.state[ref.weight].items():
        assert torch.equal(opt.state[lin.weight][k], v), k
