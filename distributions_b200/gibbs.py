"""Blocked collapsed Gibbs on one GPU for one cross-cat kind, with group births and deaths.

    kind = gibbs.BlockedGibbs(ctx, features, columns, assign, models.PitmanYor(alpha, d), n_empty=1)
    kind.sweep(n_blocks=8, generator=torch.Generator(device="cuda").manual_seed(0))

sweep() splits the rows into blocks with boundaries at multiples of 32 rows, so observed-mask words slice cleanly;
block(r0, r1) takes any row range and shifts the mask words of an unaligned one into place.  Per block:
remove the block's rows from their groups, mark them unassigned, count the group sizes, regroup (drop the emptied
groups, restore `n_empty` fresh empty groups, relabel the assignments and compact every feature), evaluate the prior
at the new G, score and sample the block's rows against it, and add them to the groups drawn.  Every block is scored
against exactly `n_empty` empty groups, so a block can open up to `n_empty` new groups.  The only host round trip per
block is the new G, read back by regroup_batch; everything else stays on the device, on torch's current stream.

What the chain samples.  The rows of one block are drawn independently of each other, each from its conditional given
the rows outside the block.  That is a valid Markov kernel, but for blocks of more than one row its stationary
distribution is not the DP / Pitman-Yor posterior over partitions; blocks of one row (`block(r, r + 1)`) make a
collapsed Gibbs sampler whose stationary distribution is the posterior (tests/test_gpu_gibbs_exact.py checks both
against the exact distributions over every partition of tiny tables).  `blocks()` makes one block of every row when
N <= 32: that block removes every row, regroup leaves only the `n_empty` fresh groups, and each row is drawn uniformly
among them without looking at the data.
"""
import numpy as np
import torch

from . import models


def block_mask_words(words, r0, r1):
    """the observed-mask words of rows [r0, r1) as a call over those rows reads them: bit n % 32 of word n / 32 is row
    r0 + n.  An aligned r0 is a slice of the kind's words; otherwise each word is the kind's words shifted right by
    r0 % 32, (w[i] >> s) | (w[i + 1] << (32 - s)), with the bits past r1 cleared (torch ops on the words' device)."""
    s, w0, n_words = r0 % 32, r0 // 32, -(-(r1 - r0) // 32)
    if s == 0:
        return words[w0:(r1 + 31) // 32]
    w = words[w0:w0 + n_words + 1].to(torch.int64) & 0xFFFFFFFF
    if w.numel() == n_words:
        w = torch.cat([w, w.new_zeros(1)])
    out = ((w[:n_words] >> s) | (w[1:] << (32 - s))) & 0xFFFFFFFF
    tail = (r1 - r0) % 32
    if tail:
        out[-1] &= (1 << tail) - 1
    if words.dtype == torch.int32:
        out = torch.where(out >= 1 << 31, out - (1 << 32), out)
    return out.to(words.dtype)


class BlockedGibbs:
    """features: the capi.Feature objects of one kind, all at G groups, with statistics matching (columns, assign);
    columns: one device tensor per feature (niw: [N][d]); assign: int32 device tensor of N group ids in [0, G);
    prior: models.PitmanYor or models.LowEntropy; observed: None, or per feature None / capi.pack_observed words on the
    device."""

    def __init__(self, ctx, features, columns, assign, prior, n_empty=1, observed=None):
        assert n_empty >= 1, "a mixture keeps at least one empty group"
        assert isinstance(prior, (models.PitmanYor, models.LowEntropy)), "prior: models.PitmanYor or models.LowEntropy"
        assert assign.dtype == torch.int32 and assign.is_cuda and assign.dim() == 1
        assert len(features) == len(columns) and (observed is None or len(observed) == len(features))
        self.ctx, self.features, self.columns, self.assign = ctx, list(features), list(columns), assign
        self.prior_model, self.n_empty, self.observed = prior, int(n_empty), observed
        self.N = assign.numel()
        self.G = features[0].groups if features else int(assign.max().item()) + 1
        self._cap = 0
        self._reserve(self.G + self.n_empty)

    def _reserve(self, n):
        """counts, compacted counts and prior buffers for n groups, grown with headroom"""
        if n <= self._cap:
            return
        self._cap = max(64, 2 * n)
        self.counts = torch.zeros(self._cap, dtype=torch.int32, device=self.assign.device)
        self.counts_out = torch.zeros(self._cap, dtype=torch.int32, device=self.assign.device)
        self.prior = torch.zeros(self._cap, dtype=torch.float32, device=self.assign.device)

    def blocks(self, n_blocks):
        """row ranges [r0, r1) of n_blocks blocks whose boundaries are multiples of 32 (one block of every row when N <= 32)"""
        size = -(-self.N // max(1, int(n_blocks)))
        size = -(-size // 32) * 32
        return [(r0, min(self.N, r0 + size)) for r0 in range(0, self.N, size)]

    def _slice(self, r0, r1):
        cols = [c[r0:r1] for c in self.columns]
        obs = None
        if self.observed is not None:
            obs = [None if m is None else block_mask_words(m, r0, r1) for m in self.observed]
        return cols, obs

    def block(self, r0, r1, generator):
        """one Gibbs block over rows [r0, r1) (any 0 <= r0 < r1 <= N); returns K+ (the live groups the block was scored
        against).  The block's rows are drawn independently of each other, given the rows outside the block."""
        # the library calls run on torch's current stream, in order with the torch ops between them
        ctx, s, n = self.ctx, torch.cuda.current_stream(self.assign.device).cuda_stream, r1 - r0
        cols, obs = self._slice(r0, r1)
        ids = self.assign[r0:r1]
        ctx.remove_rows_batch(self.features, cols, ids, n, stream=s, observed=obs)
        ids.fill_(-1)
        self._reserve(self.G + self.n_empty)
        ctx.count_assignments(self.assign, self.N, self.G, self.counts, stream=s)
        self.G = ctx.regroup_batch(self.features, self.counts, self.G, self.n_empty, self.assign, self.N,
                                   counts_out=self.counts_out, stream=s)
        if isinstance(self.prior_model, models.PitmanYor):
            ctx.prior_pitman_yor_dev(self.prior_model.alpha, self.prior_model.d, self.G, self.counts_out, self.prior, stream=s)
        else:
            ctx.prior_low_entropy_dev(self.prior_model.dataset_size, self.G, self.counts_out, self.prior, stream=s)
        u = torch.rand(n, generator=generator, device=generator.device, dtype=torch.float32).to(self.assign.device)
        ctx.score_sample_batch(self.features, cols, n, self.prior, u, ids, stream=s, observed=obs)
        ctx.add_rows_batch(self.features, cols, ids, n, stream=s, observed=obs)
        return self.G - self.n_empty

    def sweep(self, n_blocks, generator, on_block=None):
        """one pass over all rows in n_blocks blocks; on_block(self, r0, r1, k_live) after each block"""
        for r0, r1 in self.blocks(n_blocks):
            k = self.block(r0, r1, generator)
            if on_block is not None:
                on_block(self, r0, r1, k)
        return self.G

    def group_sizes(self):
        """the current group sizes (host int64 array of G entries)"""
        a = self.assign.cpu().numpy()
        return np.bincount(a[a >= 0], minlength=self.G)


def sweep(ctx, features, columns, assign, prior, n_blocks, n_empty, generator, observed=None):
    """one blocked Gibbs sweep (see BlockedGibbs); returns the new G.  assign is updated in place and the features
    follow; the caller reads the new G from the return value (every feature's `groups` also has it)."""
    return BlockedGibbs(ctx, features, columns, assign, prior, n_empty, observed).sweep(n_blocks, generator)


__all__ = ["BlockedGibbs", "sweep"]
