"""Argument checks of the joint-training wrappers (ops.bpr_fwd_bwd, ops.infonce_fwd / _bwd, ops.scatter_add_rows,
ops.modal_mix_fwd / _bwd, ops.rownorm_bwd, ops.sign_noise_, ops.bpr_infonce_fwd / _bwd): the kernels read int64 ids,
fp32 rows of a fixed width and per-row vectors through raw pointers, so every operand is validated before any device
call and these run without a GPU."""
import pytest
import torch

from diffmm_b200 import _lib, ops

B, D = 6, 8


def _i64(n=B):
    return torch.zeros(n, dtype=torch.int64)


@pytest.mark.parametrize("case", ["users_i32", "pos_i32", "neg_short", "users_2d", "users_strided", "u_f64", "i_narrow",
                                  "i_transposed"])
def test_bpr_checks_its_operands(case):
    u, i, users, pos, neg = torch.zeros((10, D)), torch.zeros((12, D)), _i64(), _i64(), _i64()
    if case == "users_i32":
        users = users.int()
    elif case == "pos_i32":
        pos = pos.int()
    elif case == "neg_short":
        neg = _i64(B - 1)
    elif case == "users_2d":
        users = _i64().view(2, 3)
    elif case == "users_strided":
        users = _i64(2 * B)[::2]
    elif case == "u_f64":
        u = u.double()
    elif case == "i_narrow":
        i = torch.zeros((12, D - 1))
    else:
        i = torch.zeros((D, 12)).t()
    with pytest.raises(ValueError, match=r"^(users|pos|neg|u_emb|i_emb):"):
        ops.bpr_fwd_bwd(u, i, users, pos, neg)


@pytest.mark.parametrize("fn,case", [(f, c) for f in ("fwd", "bwd") for c in ("idx_i32", "idx_2d", "idx_strided", "v1_f64",
                                                                               "v2_narrow")]
                         + [("bwd", c) for c in ("lse_short", "inv1_f64", "inv2_strided")])
def test_infonce_checks_its_operands(fn, case):
    v1, v2, idx = torch.zeros((10, D)), torch.zeros((10, D)), _i64()
    saved = [torch.zeros(B), torch.zeros(B), torch.zeros(B)]
    if case == "idx_i32":
        idx = idx.int()
    elif case == "idx_2d":
        idx = _i64().view(2, 3)
    elif case == "idx_strided":
        idx = _i64(2 * B)[::2]
    elif case == "v1_f64":
        v1 = v1.double()
    elif case == "v2_narrow":
        v2 = torch.zeros((10, D + 4))
    elif case == "lse_short":
        saved[0] = torch.zeros(B - 1)
    elif case == "inv1_f64":
        saved[1] = saved[1].double()
    else:
        saved[2] = torch.zeros(2 * B)[::2]
    with pytest.raises(ValueError, match=r"^(idx|v1|v2|lse|inv1|inv2):"):
        if fn == "fwd":
            ops.infonce_fwd(v1, v2, idx, 0.2)
        else:
            ops.infonce_bwd(v1, v2, idx, 0.2, saved)


@pytest.mark.parametrize("case", ["idx_i32", "idx_long", "idx_strided", "src_f64", "dst_narrow", "dst_transposed"])
def test_scatter_add_rows_checks_its_operands(case):
    src, idx, dst = torch.zeros((B, D)), _i64(), torch.zeros((10, D))
    if case == "idx_i32":
        idx = idx.int()
    elif case == "idx_long":
        idx = _i64(B + 1)
    elif case == "idx_strided":
        idx = _i64(2 * B)[::2]
    elif case == "src_f64":
        src = src.double()
    elif case == "dst_narrow":
        dst = torch.zeros((10, D - 4))
    else:
        dst = torch.zeros((D, 10)).t()
    with pytest.raises(ValueError, match=r"^(idx|src|dst):"):
        ops.scatter_add_rows(src, idx, dst)


@pytest.mark.parametrize("fn,case", [(f, c) for f in ("fwd", "bwd") for c in ("w_short", "w_long", "w_f64", "w_strided", "w_2d",
                                                                               "z_shape", "z_f64", "z_strided", "no_modality",
                                                                               "five_modalities")]
                         + [("bwd", "g_shape")])
def test_modal_mix_checks_its_operands(fn, case):
    y = torch.zeros((5, 8))
    zs, w, g = [torch.zeros((5, 8)), torch.zeros((5, 8))], torch.zeros(2), torch.zeros((5, 8))
    if case == "w_short":
        w = torch.zeros(1)
    elif case == "w_long":
        w = torch.zeros(3)
    elif case == "w_f64":
        w = w.double()
    elif case == "w_strided":
        w = torch.zeros(4)[::2]
    elif case == "w_2d":
        w = torch.zeros((1, 2))
    elif case == "z_shape":
        zs[1] = torch.zeros((5, 4))
    elif case == "z_f64":
        zs[0] = zs[0].double()
    elif case == "z_strided":
        zs[1] = torch.zeros((5, 16))[:, ::2]
    elif case == "no_modality":
        zs, w = [], torch.zeros(0)
    elif case == "five_modalities":
        zs, w = [torch.zeros((5, 8)) for _ in range(5)], torch.zeros(5)
    else:
        g = torch.zeros((8, 5))
    with pytest.raises(ValueError, match=r"^(w|zs|z\[\d\]|g):"):
        if fn == "fwd":
            ops.modal_mix_fwd(y, zs, w, 0.6)
        else:
            ops.modal_mix_bwd(g, y, zs, w, 0.6)


@pytest.mark.parametrize("case", ["g_rows", "g_cols", "g_f64", "inv_short", "inv_f64", "inv_strided", "y_f64"])
def test_rownorm_bwd_checks_g_and_inv(case):
    y, inv, g = torch.zeros((5, 8)), torch.zeros(5), torch.zeros((5, 8))
    if case == "g_rows":
        g = torch.zeros((4, 8))
    elif case == "g_cols":
        g = torch.zeros((5, 9))
    elif case == "g_f64":
        g = g.double()
    elif case == "inv_short":
        inv = torch.zeros(4)
    elif case == "inv_f64":
        inv = inv.double()
    elif case == "inv_strided":
        inv = torch.zeros(10)[::2]
    else:
        y = y.double()
    with pytest.raises(ValueError, match=r"^(y|g|inv):"):
        ops.rownorm_bwd(y, inv, g)


@pytest.mark.parametrize("case", ["rnd_rows", "rnd_cols", "rnd_f64", "rnd_transposed", "e_f64"])
def test_sign_noise_checks_rnd_against_e(case):
    e, rnd = torch.zeros((5, 8)), torch.zeros((5, 8))
    if case == "rnd_rows":
        rnd = torch.zeros((4, 8))
    elif case == "rnd_cols":
        rnd = torch.zeros((5, 7))
    elif case == "rnd_f64":
        rnd = rnd.double()
    elif case == "rnd_transposed":
        rnd = torch.zeros((8, 5)).t()
    else:
        e = e.double()
    with pytest.raises(ValueError, match=r"^(e|rnd):"):
        ops.sign_noise_(e, rnd, 0.1)


def _joint(n=20):
    tables = [torch.zeros((n, 64)), torch.zeros((n, 128))[:, :64]]
    i = _i64()
    problems = [(0, 1, i, 0, 0.2, 1.0), (1, 1, i, 4, 0.5, 0.0)]
    return tables, problems, (0, 4, i, i, i)


@pytest.mark.parametrize("case", ["view_32_of_64", "view_f64", "emb_narrow", "idx_i32", "idx_short", "users_i32",
                                  "neg_short", "no_problem", "thirteen_problems"])
@pytest.mark.parametrize("fn", ["fwd", "bwd"])
def test_bpr_infonce_checks_views_and_indices(fn, case):
    tables, problems, bpr = _joint()
    i = _i64()
    if case == "view_32_of_64":
        tables[1] = torch.zeros((20, 64))[:, :32]        # ld 64 passes the C check; 64 columns would be read
    elif case == "view_f64":
        tables[1] = tables[1].double()
    elif case == "emb_narrow":
        tables.append(torch.zeros((20, 48)))
        bpr = (2, 4, i, i, i)
    elif case == "idx_i32":
        problems[0] = (0, 1, i.int(), 0, 0.2, 1.0)
    elif case == "idx_short":
        problems[1] = (1, 1, _i64(B - 1), 4, 0.5, 0.0)
    elif case == "users_i32":
        bpr = (0, 4, i.int(), i, i)
    elif case == "neg_short":
        bpr = (0, 4, i, i, _i64(B + 1))
    elif case == "no_problem":
        problems = []
    else:
        problems = problems[:1] * 13
    with pytest.raises(ValueError, match=r"^(tables\[\d\]|problems\[\d\] idx|users|neg|problems):"):
        if fn == "fwd":
            ops.bpr_infonce_fwd(tables, problems, bpr, B)
        else:
            saved = (torch.zeros((len(problems), B)), torch.zeros((len(problems), 2, B)))
            ops.bpr_infonce_bwd(tables, problems, bpr, B, saved, torch.ones(()), torch.ones(()), [None] * len(tables))


@pytest.mark.parametrize("case", ["grad_32_of_64", "grad_rows", "grad_f64", "lse_short", "inv_f64", "g_cl_2", "g_bpr_f64"])
def test_bpr_infonce_bwd_checks_gradient_tables_and_saved(case):
    tables, problems, bpr = _joint()
    P = len(problems)
    lse, inv, g_cl, g_bpr = torch.zeros((P, B)), torch.zeros((P, 2, B)), torch.ones(()), torch.ones(())
    grads = [torch.zeros((20, 64)), torch.zeros((20, 80))[:, :64]]
    if case == "grad_32_of_64":
        grads[1] = torch.zeros((20, 64))[:, :32]
    elif case == "grad_rows":
        grads[0] = torch.zeros((19, 64))
    elif case == "grad_f64":
        grads[0] = grads[0].double()
    elif case == "lse_short":
        lse = torch.zeros((P, B - 1))
    elif case == "inv_f64":
        inv = inv.double()
    elif case == "g_cl_2":
        g_cl = torch.ones(2)
    else:
        g_bpr = g_bpr.double()
    with pytest.raises(ValueError, match=r"^(grad_tables\[\d\]|lse|inv|g_cl|g_bpr):"):
        ops.bpr_infonce_bwd(tables, problems, bpr, B, (lse, inv), g_cl, g_bpr, grads)


def test_valid_cpu_operands_pass_the_checks_and_stop_at_the_device():
    """The checks accept what the joint step passes (padded views, 0-d upstream gradients, a table without a gradient);
    the CPU tensors are then refused by the device check, not run."""
    i = _i64()
    v = torch.zeros((10, 72))[:, :D]
    cases = [
        lambda: ops.bpr_fwd_bwd(v, torch.zeros((12, D)), i, i, i),
        lambda: ops.infonce_fwd(v, v, i, 0.2),
        lambda: ops.infonce_bwd(v, v, i, 0.2, (torch.zeros(B), torch.zeros(B), torch.zeros(B))),
        lambda: ops.scatter_add_rows(torch.zeros((B, D)), i, v),
        lambda: ops.modal_mix_fwd(torch.zeros((5, 8)), [torch.zeros((5, 8))], torch.zeros(1), 0.6),
        lambda: ops.modal_mix_bwd(torch.zeros((5, 8)), torch.zeros((5, 8)), [torch.zeros((5, 8))] * 4, torch.zeros(4), 0.6),
        lambda: ops.rownorm_bwd(torch.zeros((5, 8)), torch.zeros(5), torch.zeros((5, 12))[:, :8]),
        lambda: ops.sign_noise_(v, torch.zeros((10, 12))[:, :D], 0.1),
    ]
    tables, problems, bpr = _joint()
    P = len(problems)
    cases += [
        lambda: ops.bpr_infonce_fwd(tables, problems, bpr, B),
        lambda: ops.bpr_infonce_bwd(tables, problems, bpr, B, (torch.zeros((P, B)), torch.zeros((P, 2, B))), torch.ones(()),
                                    torch.ones(()), [torch.zeros((20, 80))[:, :64], None]),
    ]
    for call in cases:
        with pytest.raises(_lib.DiffMMError, match="CUDA"):
            call()
