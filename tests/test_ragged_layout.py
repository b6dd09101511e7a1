"""The host-side layout of ragged batched problems (bore_b200/ragged.py): offsets, 64-bit sums, the
NaN-padded loss, the permutation stream of the list form, and every shape error.  No device."""
import numpy as np
import pytest

from bore_b200.ragged import RaggedLayout, ragged_inputs, ragged_rows


def test_offsets_are_prefix_sums_in_problem_order():
    lay = RaggedLayout([3, 1, 5, 2], [2, 0, 1, 4])
    assert lay.rows.tolist() == [0, 3, 4, 9, 11]
    assert lay.perms.tolist() == [0, 6, 6, 11, 19]
    assert lay.losses.tolist() == [0, 2, 2, 3, 7]
    assert lay.rows.dtype == lay.perms.dtype == lay.losses.dtype == np.int64
    assert lay.steps(2).tolist() == [4, 0, 3, 4]


def test_sums_are_64_bit():
    # 4,096 problems of 16,384 observations in 50 dimensions: sum N_p * D passes 2**31
    lay = RaggedLayout(np.full(4096, 16384), np.full(4096, 100))
    assert lay.rows[-1] * 50 == 4096 * 16384 * 50 > 2 ** 31
    assert lay.perms[-1] == 4096 * 16384 * 100 > 2 ** 32


def test_loss_is_padded_with_nan():
    lay = RaggedLayout([4, 2, 7], [2, 0, 3])
    flat = np.arange(5, dtype=np.float32) + 1
    out = lay.pad_loss(flat)
    assert out.shape == (3, 3) and out.dtype == np.float32
    assert out[0, :2].tolist() == [1, 2] and np.isnan(out[0, 2])
    assert np.isnan(out[1]).all()
    assert out[2].tolist() == [3, 4, 5]
    assert RaggedLayout([1, 2], [0, 0]).pad_loss(np.zeros(0, np.float32)).shape == (2, 0)


def test_equal_counts_draw_the_uniform_calls_permutations():
    M, N, D, E = 5, 17, 3, 4
    rs = np.random.RandomState(0)
    X = rs.uniform(size=(M, N, D))
    y = rs.uniform(size=(M, N))
    a, b = np.random.RandomState(7), np.random.RandomState(7)
    # the uniform path of BatchedMaximizableSequential.fit
    uniform = np.stack([np.stack([a.permutation(N) for _ in range(E)]) for _ in range(M)])
    lay, Xc, yc, w, perm = ragged_inputs(list(X), list(y), M, D, E, random_state=b)
    assert np.array_equal(perm, uniform.reshape(-1)) and perm.dtype == np.int32
    assert np.array_equal(Xc, X.reshape(M * N, D)) and np.array_equal(yc, y.reshape(-1)) and w is None
    assert a.randint(1 << 30) == b.randint(1 << 30)  # the same state afterwards


def test_ragged_permutations_follow_problem_then_epoch():
    n, e = [3, 5, 2], [2, 1, 0]
    X = [np.zeros((k, 2)) for k in n]
    y = [np.zeros(k) for k in n]
    a, b = np.random.RandomState(3), np.random.RandomState(3)
    lay, _, _, _, perm = ragged_inputs(X, y, 3, 2, e, random_state=b)
    want = np.concatenate([a.permutation(3), a.permutation(3), a.permutation(5)])
    assert np.array_equal(perm, want)
    lay, _, _, _, perm = ragged_inputs(X, y, 3, 2, e, shuffle=False)
    assert perm.tolist() == [0, 1, 2, 0, 1, 2, 0, 1, 2, 3, 4]
    given = [np.array([[2, 1, 0], [0, 2, 1]]), np.array([[4, 3, 2, 1, 0]]), np.zeros((0, 2), int)]
    sw = [np.ones(3), np.full((5, 1), 2.0), np.zeros(2)]
    lay, _, _, w, perm = ragged_inputs(X, y, 3, 2, e, sample_weight=sw, permutations=given)
    assert perm.tolist() == [2, 1, 0, 0, 2, 1, 4, 3, 2, 1, 0]
    assert w.dtype == np.float32 and w.tolist() == [1, 1, 1, 2, 2, 2, 2, 2, 0, 0]


def test_exclude_rows():
    counts, rows = ragged_rows([np.ones((2, 3)), np.zeros((0, 3)), [], np.full((1, 3), 5.0)], 4, 3)
    assert counts.tolist() == [2, 0, 0, 1] and rows.shape == (3, 3) and rows[2, 0] == 5.0


def _data(n=(3, 4), D=2):
    return [np.zeros((k, D)) for k in n], [np.zeros(k) for k in n]


@pytest.mark.parametrize("case", [
    "x_not_list", "x_length", "y_length", "x_dims", "x_width", "x_empty", "y_shape", "epochs_length",
    "epochs_negative", "epochs_fraction", "epochs_scalar_fraction", "weight_length", "weight_shape",
    "perm_length", "perm_shape", "perm_range", "no_random_state"])
def test_shape_and_length_errors_raise_value_error(case):
    X, y = _data()
    kw = dict(random_state=np.random.RandomState(0))
    args = [X, y, 2, 2, 1]
    if case == "x_not_list":
        args[0] = np.zeros((2, 3, 2))
    elif case == "x_length":
        args[0] = X[:1]
    elif case == "y_length":
        args[1] = y + [np.zeros(3)]
    elif case == "x_dims":
        args[0] = [np.zeros(3), X[1]]
    elif case == "x_width":
        args[0] = [np.zeros((3, 5)), X[1]]
    elif case == "x_empty":
        args[0], args[1] = [np.zeros((0, 2)), X[1]], [np.zeros(0), y[1]]
    elif case == "y_shape":
        args[1] = [np.zeros(4), y[1]]
    elif case == "epochs_length":
        args[4] = [1, 2, 3]
    elif case == "epochs_negative":
        args[4] = [1, -1]
    elif case == "epochs_fraction":
        args[4] = [1, 1.5]
    elif case == "epochs_scalar_fraction":
        args[4] = 1.5
    elif case == "weight_length":
        kw["sample_weight"] = [np.ones(3)]
    elif case == "weight_shape":
        kw["sample_weight"] = [np.ones(3), np.ones(5)]
    elif case == "perm_length":
        kw["permutations"] = [np.zeros((1, 3), int)]
    elif case == "perm_shape":
        kw["permutations"] = [np.zeros((1, 3), int), np.zeros((2, 4), int)]
    elif case == "perm_range":
        kw["permutations"] = [np.zeros((1, 3), int), np.full((1, 4), 4)]
    elif case == "no_random_state":
        kw = {}
    with pytest.raises(ValueError):
        ragged_inputs(*args, **kw)


def test_layout_errors():
    with pytest.raises(ValueError):
        RaggedLayout([1, 2], [1])
    with pytest.raises(ValueError):
        RaggedLayout([], [])
    with pytest.raises(ValueError):
        RaggedLayout([1, 0], [1, 1])
    with pytest.raises(ValueError):
        RaggedLayout([1, 2], [1, -2])
    with pytest.raises(ValueError):
        RaggedLayout([1 << 31], [1])
    with pytest.raises(ValueError):
        ragged_rows([np.ones((2, 3))], 2, 3)
    with pytest.raises(ValueError):
        ragged_rows([np.ones((2, 3)), np.ones((2, 4))], 2, 3)
