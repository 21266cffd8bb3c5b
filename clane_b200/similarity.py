"""Similarity plugins -- drop-in for ``clane.similarity`` (/root/reference/clane/similarity.py).

The registry is this module's namespace: the CLI resolves ``similarity.method`` with
``getattr(similarity, name)`` and constructs it with ``**kwargs`` (__main__.py:39-48).
Plugins are called as ``sim(v1, v2)`` with two ``[E, d]`` (or 1-D) tensors and return ``[E]``.

Built-in plugins carry ``_clane_kernel``; ``Graph.build_P`` dispatches on it to the fused
per-edge score + neighbour-softmax kernels.  A user plugin without the tag is still honoured
(its scores are computed by the plugin on device tensors, the softmax stays in CUDA).
Precision of the fused scorers on fp32 embeddings: ``CosineSimilarity`` is bit-exact with the
reference at every width; ``AsymmertricSimilarity`` reads TF32 at d in {32, 64, 96, 128} and is
fp32-accurate (3xTF32) at every other width.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib


class Similarity:
    def is_trainable(self):
        return isinstance(self, nn.Module)


class CosineSimilarity(Similarity):
    """``<v1_e, v2_e> / (||V1||_F * ||V2||_F)`` -- the reference divides every per-pair dot by
    the two GLOBAL Frobenius norms of the batched inputs (similarity.py:37); it is the true
    cosine only for a single pair.  That behaviour is reproduced, not fixed."""

    _clane_kernel = "cosine"

    def __init__(self, **kwargs) -> None:
        super(CosineSimilarity, self).__init__()

    def __call__(self, v1: torch.Tensor, v2: torch.Tensor) -> torch.Tensor:
        if v1.dim() == 1:
            v1 = v1.unsqueeze(0)
        if v2.dim() == 1:
            v2 = v2.unsqueeze(0)
        if v1.dim() != 2 or v2.dim() != 2 or v1.shape[1] != v2.shape[1] or (
                v1.shape[0] != v2.shape[0] and 1 not in (v1.shape[0], v2.shape[0])):
            raise RuntimeError(f"CosineSimilarity expects two [E, d] batches, got {tuple(v1.shape)} and {tuple(v2.shape)}")
        _lib.require_cuda()
        L = _lib.lib()
        out_device = v1.device
        e = max(int(v1.shape[0]), int(v2.shape[0]))
        s = _lib.stream_handle()
        if v1.shape[0] == v2.shape[0]:
            out, norms2 = self._raw(v1, v2)
        else:
            # [1, d] against [E, d]: the reference's matmul broadcasts the single row (similarity.py:35-37) while each
            # global norm runs over its tensor AS GIVEN -- dots of the expanded batch, the single row's norm counted once
            out, nb = self._raw(v1.expand(e, -1), v2.expand(e, -1))
            one = v1 if v1.shape[0] == 1 else v2
            _, n1 = self._raw(one, one)
            norms2 = torch.stack([n1[0], nb[1]]) if v1.shape[0] == 1 else torch.stack([nb[0], n1[0]])
        _lib.check(L.clane_cosine_finalize(out.data_ptr(), norms2.data_ptr(), e, out.data_ptr(), s),
                   "clane_cosine_finalize")
        res = out[:e].to(out_device)
        torch.cuda.current_stream().synchronize()
        return res

    @staticmethod
    def _raw(v1: torch.Tensor, v2: torch.Tensor):
        """(per-pair dots [E], the two global square sums [2]) on the device, in the reference's summation orders."""
        dev = _lib.require_cuda()
        L = _lib.lib()
        e, d = int(v1.shape[0]), int(v1.shape[1])
        ld = int(L.clane_padded_ld(d))
        # pair i is the edge  i -> e + i  of a bipartite helper graph over the stacked rows
        Z = torch.zeros([2 * e, ld], dtype=torch.float32, device=dev)
        Z[:e, :d] = v1.to(device=dev, dtype=torch.float32)
        Z[e:, :d] = v2.to(device=dev, dtype=torch.float32)
        erow = torch.arange(0, e, dtype=torch.int32, device=dev)
        col = torch.arange(e, 2 * e, dtype=torch.int32, device=dev)
        out = torch.empty(max(e, 1), dtype=torch.float32, device=dev)
        norms2 = torch.empty(2, dtype=torch.float32, device=dev)
        plan = _lib.Plan(2 * e, e, d)          # scores-only plan: reduction scratch, no schedule
        _lib.check(L.clane_scores_cosine(plan.handle, Z.data_ptr(), erow.data_ptr(), col.data_ptr(), 0, e,
                                         out.data_ptr(), norms2.data_ptr(), _lib.stream_handle()), "clane_scores_cosine")
        torch.cuda.current_stream().synchronize()   # the plan's scratch is freed when it goes out of scope
        return out, norms2


class AsymmertricSimilarity(nn.Module, Similarity):
    """Trainable bilinear score ``<Phi_src z_src, Phi_dst z_dst>`` (similarity.py:40-57; the spelling is API).

    ``Phi_src`` / ``Phi_dst`` are bias-free ``nn.Linear(n_dim, n_dim)`` layers with Xavier-normal weights, as upstream
    (checkpoints and optimisers address them by these names).  A direct call scores pairs with torch on whatever device
    the inputs live on.  ``Graph.build_P`` on fp32 embeddings does not gather ``[E, d]`` rows for it: it projects every
    NODE once on the tensor cores (tcgen05 GEMM, TMA-staged), takes the per-edge dots of the projected rows and applies
    the row softmax.  The precision depends on the width:
      * ``n_dim`` in {32, 64, 96, 128}: ``clane_build_p_asym``, tensor-core inputs read as TF32 -- scores agree with the
        fp32 module to ~1e-3 relative (tests/test_gpu_parity.py::test_asymmetric_scorer_fused_build_p);
      * every other ``n_dim``: ``clane_build_p_asym_fp32``, 3xTF32 (each operand split into a TF32 part and its fp32
        remainder) -- every projected value within (4 + 3 n_dim) 2^-23 sum_k |z_k w_k| of the exact product, i.e. fp32
        accuracy (tests/test_asym_fp32.py).
    Only this class's own ``forward`` is fused: a subclass that overrides it is scored by its ``forward`` on gathered
    rows (the generic plugin path), as are fp64 embeddings."""

    _clane_kernel = "asym"

    def __init__(self, n_dim: int, **kwargs) -> None:
        super().__init__()
        for name in ("Phi_src", "Phi_dst"):
            layer = nn.Linear(n_dim, n_dim, bias=False)
            nn.init.xavier_normal_(layer.weight)
            setattr(self, name, layer)

    def stacked_weights(self, device) -> torch.Tensor:
        """``[W_src ; W_dst]`` as one contiguous fp32 ``[2 n_dim, n_dim]`` matrix on ``device`` (the B operand of the GEMM)."""
        return torch.cat([self.Phi_src.weight, self.Phi_dst.weight]).detach().to(device=device, dtype=torch.float32).contiguous()

    def forward(self, z_src: torch.Tensor, z_dst: torch.Tensor) -> torch.Tensor:
        projected_src, projected_dst = self.Phi_src(z_src), self.Phi_dst(z_dst)
        return (projected_src.unsqueeze(-2) @ projected_dst.unsqueeze(-1)).squeeze()
