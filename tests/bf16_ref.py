"""Float64 restatement of the bf16 propagation contract of parallel.bipartite_propagate_mean
(precision="bf16") on the whole, unsharded graph: A = [[0, R], [R^T, 0]], X = [users; items].

    acc = X0;  x = round(X0)
    for l = 1..L:  y = A x;  acc = acc + y;  x = round(y)
    out = acc / (L + 1)

`round` is bfloat16 round-to-nearest-even, applied to whole rows of the table, which is what the
sharded code does: user rows by the SpMM epilogue (y16), item rows after their all-reduce. The
backward of the operator is the same operator on the gradients (A is symmetric)."""
import torch


def round_bf16(x):
    """x rounded to bfloat16 (nearest even), returned in x's dtype."""
    return x.to(torch.bfloat16).to(x.dtype)


def propagate_bf16(A, X0, n_layers, rnd=round_bf16):
    if n_layers == 0:
        return X0.clone()
    acc, x = X0.clone(), rnd(X0)
    for _ in range(n_layers):
        y = A @ x
        acc = acc + y
        x = rnd(y)
    return acc * (1.0 / (n_layers + 1))


class PropagateBf16(torch.autograd.Function):
    """propagate_bf16 with the contract's backward: the same rounded operator on the gradient."""

    @staticmethod
    def forward(ctx, X0, A, n_layers):
        ctx.A, ctx.n_layers = A, n_layers
        return propagate_bf16(A, X0, n_layers)

    @staticmethod
    def backward(ctx, g):
        return propagate_bf16(ctx.A, g.contiguous(), ctx.n_layers), None, None
