"""Argument checks of the reverse-chain staging wrappers (ops.time_bias, ops.time_embedding, ops.gemv_f32,
ops.bias_act_pack): the 1-D and 2-D fp32 operands the kernels read through raw pointers are validated before any device
call, so these run without a GPU."""
import pytest
import torch

from diffmm_b200 import ops


def _emb(d=10):
    return torch.zeros((d, d)), torch.zeros(d)


@pytest.mark.parametrize("case", ["w_f64", "w_transposed", "w_not_square", "w_1d", "b_short", "b_f64", "b_2d",
                                  "b_strided", "not_tensor"])
@pytest.mark.parametrize("fn", ["time_bias", "time_embedding"])
def test_time_embedding_weights_are_checked(fn, case):
    w, b = _emb()
    if case == "w_f64":
        w = w.double()
    elif case == "w_transposed":
        w = torch.zeros((10, 10)).t()
    elif case == "w_not_square":
        w = torch.zeros((10, 9))
    elif case == "w_1d":
        w = torch.zeros(100)
    elif case == "b_short":
        b = torch.zeros(9)
    elif case == "b_f64":
        b = b.double()
    elif case == "b_2d":
        b = torch.zeros((1, 10))
    elif case == "b_strided":
        b = torch.zeros(20)[::2]
    else:
        w = w.numpy()
    with pytest.raises(ValueError, match="emb_w|emb_b"):
        if fn == "time_bias":
            ops.time_bias(w, b, torch.zeros((8, 30)), 20, torch.zeros(8), 0, 2)
        else:
            ops.time_embedding(w, b, 4, t_all=3, temb_f32=torch.zeros((4, 10)))


@pytest.mark.parametrize("case", ["weight_f64", "weight_transposed", "col0_past_end", "col0_negative", "bias_short",
                                  "bias_f64", "bias_strided"])
def test_time_bias_checks_weight_and_bias(case):
    w, b = _emb()
    weight, col0, bias = torch.zeros((8, 30)), 20, torch.zeros(8)
    if case == "weight_f64":
        weight = weight.double()
    elif case == "weight_transposed":
        weight = torch.zeros((30, 8)).t()
    elif case == "col0_past_end":
        col0 = 21
    elif case == "col0_negative":
        col0 = -1
    elif case == "bias_short":
        bias = torch.zeros(7)
    elif case == "bias_f64":
        bias = bias.double()
    else:
        bias = torch.zeros(16)[::2]
    with pytest.raises(ValueError, match="weight|bias"):
        ops.time_bias(w, b, weight, col0, bias, 0, 2)


@pytest.mark.parametrize("case", ["x_short", "x_long", "x_f64", "x_strided", "x_2d", "w_f64", "w_transposed",
                                  "k_zero", "k_past_end", "out_short"])
def test_gemv_f32_checks_its_operands(case):
    w, K, x, out = torch.zeros((6, 40)), 33, torch.zeros(33), None
    if case == "x_short":
        x = torch.zeros(32)
    elif case == "x_long":
        x = torch.zeros(34)
    elif case == "x_f64":
        x = x.double()
    elif case == "x_strided":
        x = torch.zeros(66)[::2]
    elif case == "x_2d":
        x = torch.zeros((1, 33))
    elif case == "w_f64":
        w = w.double()
    elif case == "w_transposed":
        w = torch.zeros((40, 6)).t()
    elif case == "k_zero":
        K = 0
    elif case == "k_past_end":
        K, x = 41, torch.zeros(41)
    else:
        out = torch.zeros(5)
    with pytest.raises(ValueError, match="x|w|K|out"):
        ops.gemv_f32(w, K, x, out)


@pytest.mark.parametrize("case", ["bias_short", "bias_f64", "bias_strided", "z_f64", "z_transposed"])
def test_bias_act_pack_checks_z_and_bias(case):
    z, bias = torch.zeros((3, 12)), torch.zeros(12)
    if case == "bias_short":
        bias = torch.zeros(11)
    elif case == "bias_f64":
        bias = bias.double()
    elif case == "bias_strided":
        bias = torch.zeros(24)[::2]
    elif case == "z_f64":
        z = z.double()
    else:
        z = torch.zeros((12, 3)).t()
    h = torch.zeros((3, 12), dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="z|bias"):
        ops.bias_act_pack(z, bias, 1, h)


def test_valid_cpu_operands_pass_the_checks_and_stop_at_the_device():
    """The checks accept what the chain passes; the CPU tensors are then refused by the device check, not run."""
    from diffmm_b200 import _lib
    w, b = _emb()
    with pytest.raises(_lib.DiffMMError, match="CUDA"):
        ops.time_bias(w, b, torch.zeros((8, 30)), 20, torch.zeros(8), 0, 2)
    with pytest.raises(_lib.DiffMMError, match="CUDA"):
        ops.time_bias(w, b, torch.zeros((8, 30)), 20, None, 0, 2)
    with pytest.raises(_lib.DiffMMError, match="CUDA"):
        ops.time_embedding(w, b, 4, t_all=3, temb_f32=torch.zeros((4, 10)))
    with pytest.raises(_lib.DiffMMError, match="CUDA"):
        ops.gemv_f32(torch.zeros((6, 40)), 33, torch.zeros(34)[1:])
    with pytest.raises(_lib.DiffMMError, match="CUDA"):
        ops.bias_act_pack(torch.zeros((3, 12)), torch.zeros(12), 1, torch.zeros((3, 12), dtype=torch.bfloat16))
