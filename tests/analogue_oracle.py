"""CPU reference of the analogue loop (test infrastructure): the reference's merge_fragments loop
(equivariant_diffusion.py:515-607) run on whole molecules, built from the oracle port's own pieces (oracle/edm_oracle.py)."""
from typing import Callable, Optional, Tuple

import torch

from oracle.edm_oracle import (NoiseTape, StateDict, Tensor, _times, combined_noise, edm_merge_fragments, gamma_lookup,
                               sample_p_xh_given_z0, sample_p_zs_given_zt)


def edm_analogue(sd: StateDict, gamma: Tensor, node_mask: Tensor, edge_mask: Tensor, fixed_mask: Tensor,
                 context: Tensor, z_known: Tensor, tape: NoiseTape, diffusion_level: int = 50, resample_steps: int = 1,
                 blend_power: int = 3, hook: Optional[Callable] = None) -> Tuple[Tensor, Tensor]:
    """Analogues of the whole molecules in z_known.  With fixed atoms (every sample must have one) it IS
    edm_merge_fragments.  With none, merge_fragments would divide the fixed-atom centre of mass by a zero count
    (align_fragment_com: NaN), so the re-injection is left out: the same loop without _reinject, which draws no
    re-injection noise."""
    per_sample = fixed_mask.reshape(fixed_mask.size(0), -1).sum(1)
    if bool((per_sample > 0).all()):
        return edm_merge_fragments(sd, gamma, node_mask, edge_mask, fixed_mask, context, z_known, tape, diffusion_level,
                                   resample_steps, blend_power, hook)
    if bool((per_sample > 0).any()):
        raise ValueError("edm_analogue: either every sample has fixed atoms or none has")
    resample_steps = max(resample_steps, 1)
    b = node_mask.size(0)
    T = gamma.numel() - 1
    s0 = torch.full([b, 1], diffusion_level, dtype=torch.int64) / T
    g = gamma_lookup(gamma, s0)
    shp = (b, 1, 1)
    z = torch.sqrt(torch.sigmoid(-g)).view(shp) * z_known + torch.sqrt(torch.sigmoid(g)).view(shp) * combined_noise(
        tape, node_mask)
    for s in range(T - 1, -1, -1):
        if s > diffusion_level:
            continue
        s_arr, t_arr = _times(s, T, b)
        for _ in range(resample_steps):
            z = sample_p_zs_given_zt(sd, gamma, s_arr, t_arr, z, node_mask, edge_mask, context, tape, hook)
    return sample_p_xh_given_z0(sd, gamma, z, node_mask, edge_mask, context, tape, hook)
