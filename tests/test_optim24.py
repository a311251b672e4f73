"""The fused 2:4 optimizer step without a device: the C ABI's refusals (no launch), the Python optimizers' refusals,
and the item tables SGD24 / AdamW24 build for mixed models."""
import ctypes

import pytest
import torch

NEW = ["spfy_optim24_step"]


def test_new_symbols_are_declared_exported_and_bound(spfy):
    from test_boundary import declared_symbols
    names = declared_symbols()
    lib = ctypes.CDLL(spfy.capi.LIB_PATH)
    for n in NEW:
        assert n in names and hasattr(lib, n) and n in spfy.capi.SIGNATURES
    assert (spfy.OPTIM_SGD, spfy.OPTIM_ADAMW) == (0, 1)
    for n in ("SGD24", "AdamW24"):
        assert n in spfy.__all__ and issubclass(getattr(spfy, n), torch.optim.Optimizer)


def _fake(addr):
    return ctypes.c_void_p(addr)


def _item(capi, **kw):
    base = dict(param=1 << 20, grad=2 << 20, state1=3 << 20, state2=4 << 20, step=5 << 20, first=None, rows=64, cols=64,
                ld=64, group=0, dtype=capi.F16, meta=6 << 20, vals=7 << 20, vals_t=8 << 20, kh=1, kw=1, stride=1, pad=0)
    base.update(kw)
    return capi.Optim24Item(**base)


def _call(spfy, algo=None, items=None, groups=None, n_groups=None, grad_scale=None, found_inf=None, **hp):
    capi = spfy.capi
    algo = capi.OPTIM_SGD if algo is None else algo
    items = [_item(capi)] if items is None else items
    if groups is None:
        h = dict(lr=0.1, momentum=0.9, dampening=0.0, weight_decay=0.0, beta1=0.9, beta2=0.999, eps=1e-8, nesterov=0)
        h.update(hp)
        groups = [capi.Optim24Hparams(**h)]
    it = (capi.Optim24Item * len(items))(*items)
    gr = (capi.Optim24Hparams * len(groups))(*groups)
    n0 = capi.launch_count()
    with pytest.raises(spfy.SpfyError) as e:
        capi.spfy_optim24_step(algo, it, len(items), gr, len(groups) if n_groups is None else n_groups, grad_scale,
                               found_inf, None)
    assert capi.launch_count() == n0
    return e.value.code


def test_c_refusals_launch_nothing(spfy):
    capi = spfy.capi
    INV, UNS = capi.E_INVALID, capi.E_UNSUPPORTED
    it = lambda **kw: [_item(capi, **kw)]  # noqa: E731
    assert _call(spfy, algo=7) == INV
    assert _call(spfy, items=it(param=None)) == INV
    assert _call(spfy, items=it(grad=None)) == INV
    assert _call(spfy, items=it(state1=None)) == INV                          # SGD momentum without a buffer
    assert _call(spfy, algo=capi.OPTIM_ADAMW, items=it(state2=None)) == INV  # AdamW without exp_avg_sq
    assert _call(spfy, algo=capi.OPTIM_ADAMW, items=it(step=None)) == INV
    assert _call(spfy, items=it(param=(1 << 20) + 4)) == INV                 # 2:4 fp32 rows: 16-byte aligned
    assert _call(spfy, items=it(meta=None, param=(1 << 20) + 2)) == INV      # dense: 4-byte aligned
    assert _call(spfy, items=it(vals=None)) == INV
    assert _call(spfy, items=it(vals_t=(8 << 20) + 8)) == INV
    assert _call(spfy, items=it(ld=60)) == INV                                # ld < cols
    assert _call(spfy, items=it(group=1)) == INV
    assert _call(spfy, lr=-1.0) == INV
    assert _call(spfy, algo=capi.OPTIM_ADAMW, eps=-1.0) == INV
    assert _call(spfy, nesterov=1, momentum=0.0) == INV
    assert _call(spfy, nesterov=1, dampening=0.5) == INV
    assert _call(spfy, found_inf=_fake((9 << 20) + 2)) == INV
    assert _call(spfy, items=it(first=(9 << 20) + 2)) == INV
    assert _call(spfy, items=it(dtype=capi.F32)) == UNS
    assert _call(spfy, items=it(rows=60)) == UNS
    assert _call(spfy, items=it(cols=60, ld=64)) == UNS
    assert _call(spfy, items=it(cols=9 * 12, ld=9 * 12, kh=3, kw=3)) == UNS   # c % 8
    assert _call(spfy, items=it(kh=17, cols=17 * 8, ld=17 * 8)) == UNS
    assert _call(spfy, items=it(stride=9)) == UNS
    assert _call(spfy, items=it(rows=1 << 24)) == UNS
    assert _call(spfy, items=it(meta=None, rows=1, cols=1 << 31)) == UNS
    # a refusal anywhere in the table comes before the launch of the items ahead of it
    assert _call(spfy, items=[_item(capi, meta=None)] * 300 + it(rows=60)) == UNS


def test_empty_items_are_skipped_before_their_pointers_are_checked(spfy):
    capi = spfy.capi
    empty = capi.Optim24Item(rows=0, cols=0, group=5)  # a numel-0 parameter: data_ptr 0, nothing to read
    hp = capi.Optim24Hparams(lr=0.1, momentum=0.9)
    n0 = capi.launch_count()
    capi.spfy_optim24_step(capi.OPTIM_SGD, (capi.Optim24Item * 1)(empty), 1, (capi.Optim24Hparams * 1)(hp), 1, None, None,
                           None)
    assert capi.launch_count() == n0


def test_step_refuses_host_parameters_before_anything_changes(spfy):
    lin, conv, bn = fake_layers(spfy)
    params = list(lin.parameters()) + list(conv.parameters()) + list(bn.parameters())
    for p in params:
        p.grad = torch.ones_like(p)
    for opt in (spfy.SGD24(params, lr=0.1, momentum=0.9), spfy.AdamW24(params, lr=0.1)):
        n0 = spfy.capi.launch_count()
        with pytest.raises(spfy.SpfyError) as e:
            opt.step()
        assert e.value.code == spfy.capi.E_INVALID and "host" in str(e.value)
        assert spfy.capi.launch_count() == n0 and len(opt.state) == 0


def test_python_refusals(spfy):
    p = torch.nn.Parameter(torch.zeros(8))
    for kw in (dict(lr=-0.1), dict(momentum=-0.5), dict(weight_decay=-1.0), dict(nesterov=True),
               dict(nesterov=True, momentum=0.9, dampening=0.1), dict(maximize=True), dict(foreach=True),
               dict(fused=True), dict(differentiable=True)):
        with pytest.raises(ValueError):
            spfy.SGD24([p], **kw)
    for kw in (dict(lr=-0.1), dict(eps=-1e-8), dict(betas=(1.0, 0.9)), dict(amsgrad=True), dict(maximize=True),
               dict(foreach=True), dict(fused=True), dict(differentiable=True)):
        with pytest.raises(ValueError):
            spfy.AdamW24([p], **kw)
    with pytest.raises(TypeError):
        spfy.SGD24([torch.nn.Parameter(torch.zeros(8, dtype=torch.float16))])
    with pytest.raises(ValueError):  # not dense
        spfy.SGD24([torch.nn.Parameter(torch.zeros(8, 8)[:, :4])])
    with pytest.raises(ValueError):  # mixed devices
        spfy.SGD24([p, torch.nn.Parameter(torch.zeros(8, device="meta"))])
    opt = spfy.SGD24([p], lr=0.1)
    with pytest.raises(ValueError):
        opt.add_param_group({"params": [torch.nn.Parameter(torch.zeros(8, device="meta"))]})
    assert len(opt.param_groups) == 1
    with pytest.raises(ValueError):
        opt.add_param_group({"params": [torch.nn.Parameter(torch.zeros(8))], "nesterov": True})
    p.grad = torch.zeros(8).to_sparse()
    with pytest.raises(TypeError):
        opt._table()  # what step() builds, after its device check


def fake_layers(spfy):
    """a Linear24 and a Conv2d24 on host tensors (their constructors touch no device), plus a BatchNorm"""
    comp = spfy.Compressed24(torch.zeros(16384, dtype=torch.uint8), torch.zeros(2048, dtype=torch.uint8), 64, 128,
                             torch.float16, spfy.LAYOUT_SM100)
    comp_t = spfy.Compressed24(torch.zeros(16384, dtype=torch.uint8), torch.zeros(2048, dtype=torch.uint8), 128, 64,
                               torch.bfloat16, spfy.LAYOUT_SM100)
    lin = spfy.Linear24(torch.zeros(64, 128), torch.zeros(64), comp, comp_t, torch.float16)
    ccomp = spfy.Compressed24(torch.zeros(16384 * 5, dtype=torch.uint8), torch.zeros(2048 * 5, dtype=torch.uint8), 128,
                              9 * 64, torch.bfloat16, spfy.LAYOUT_SM100)
    op_t = spfy.Transpose24Conv(torch.zeros(16384 * 8, dtype=torch.uint8), torch.zeros(2048 * 8, dtype=torch.uint8), 128,
                                64, 3, 3, 2, 1, torch.bfloat16, [])
    conv = spfy.Conv2d24(torch.zeros(128, 64, 3, 3).contiguous(memory_format=torch.channels_last), None, ccomp, op_t,
                         torch.bfloat16, 2, 1)
    return lin, conv, torch.nn.BatchNorm2d(128)


def test_item_table_of_a_mixed_model(spfy):
    lin, conv, bn = fake_layers(spfy)
    params = list(lin.parameters()) + list(conv.parameters()) + list(bn.parameters())
    opt = spfy.SGD24([{"params": params[:2]}, {"params": params[2:], "lr": 0.5}], lr=0.1, momentum=0.9)
    for p in params:
        p.grad = torch.ones_like(p)
    bn.bias.grad = None  # skipped
    conv.weight.grad = torch.ones(128, 64, 3, 3)  # a gradient in another layout: copied into the parameter's
    items, hps, ps, layers, keep, steps, firsts = opt._table()
    assert len(items) == 4 and [x is y for x, y in zip(ps, [lin.weight, lin.bias, conv.weight, bn.weight])] == [True] * 4
    assert [layer is x for layer, x in zip(layers, (lin, conv))] == [True, True] and steps == []
    assert (hps[0].lr, hps[1].lr, hps[0].momentum) == (0.1, 0.5, 0.9)
    a, b, c, d = items
    assert (a.meta, a.vals, a.vals_t) == (lin.comp.meta.data_ptr(), lin.comp.vals.data_ptr(), lin.comp_t.vals.data_ptr())
    assert (a.rows, a.cols, a.ld, a.dtype, a.kh, a.kw, a.stride, a.pad, a.group) == (64, 128, 128, spfy.F16, 1, 1, 1, 0, 0)
    assert b.meta is None and (b.rows, b.cols) == (1, 64) and b.param == lin.bias.data_ptr()
    assert (c.rows, c.cols, c.ld, c.dtype, c.kh, c.kw, c.stride, c.pad, c.group) == (128, 576, 576, spfy.BF16, 3, 3, 2, 1, 1)
    assert c.vals_t == conv.op_t.vals.data_ptr() and c.param == conv.weight.data_ptr()
    assert len(keep) == 1 and keep[0].stride() == conv.weight.stride() and c.grad == keep[0].data_ptr()
    assert d.meta is None and (d.rows, d.cols, d.group) == (1, 128, 1)
    # momentum buffers: created as zeros in the parameter's layout, torch's first step pending in a device flag
    assert [p is q for (p, _), q in zip(firsts, ps)] == [True] * 4
    for it, p, (_, flag) in zip(items, ps, firsts):
        buf = opt.state[p]["momentum_buffer"]
        assert it.first == flag.data_ptr() and float(flag) == 1.0
        assert it.state1 == buf.data_ptr() and buf.stride() == p.stride() and not bool(buf.any())
    # until a step has been applied, the first step stays pending
    items, *_, firsts2 = opt._table()
    assert [f is g for (_, f), (_, g) in zip(firsts, firsts2)] == [True] * 4
    opt._first.clear()  # what an applied step without found_inf does
    items, *_, firsts = opt._table()
    assert [it.first for it in items] == [None] * 4 and firsts == []
    # AdamW: torch's state names, a float32 step count on the parameter's device
    opt = spfy.AdamW24(params, lr=0.1)
    items, hps, ps, layers, keep, steps, firsts = opt._table()
    assert len(steps) == 4 and firsts == [] and all(s.dtype == torch.float32 and s.dim() == 0 for s in steps)
    for it, p in zip(items, ps):
        st = opt.state[p]
        assert (it.state1, it.state2, it.step) == (st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(),
                                                   st["step"].data_ptr())
    assert hps[0].beta1 == 0.9 and hps[0].beta2 == 0.999 and hps[0].weight_decay == 0.01


def test_state_moves_from_torch_sgd(spfy):
    """torch's SGD state_dict (momentum_buffer None for a parameter it has not stepped) loads into SGD24"""
    p = torch.nn.Parameter(torch.zeros(8))
    t = torch.optim.SGD([p], lr=0.1, momentum=0.9)
    p.grad = torch.ones(8)
    t.step()
    opt = spfy.SGD24([p], lr=0.1, momentum=0.9)
    opt.load_state_dict(t.state_dict())
    items, *_ = opt._table()
    assert items[0].first is None and items[0].state1 == opt.state[p]["momentum_buffer"].data_ptr()
