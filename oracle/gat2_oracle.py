"""Plain-PyTorch CPU restatement of FragNet's GAT2 hot path.  TEST INFRASTRUCTURE ONLY.

Every function restates, op for op, what the reference computes (file:line cited per
function, paths relative to the reference root), written functionally over a flat
``{name: tensor}`` parameter mapping with the reference's ``state_dict`` key names, so the
same weights drive the oracle and the CUDA path.  It deliberately keeps the reference's
cost structure -- gather, concatenate ``[target | edge | source]``, multiply by the head
vector, reduce, scatter-softmax, scatter-add -- so that timing it on host cores is a fair
"port" CPU baseline, and so that rounding follows the reference closely.

Pinning: parity is unpinned by the reference (no tests / golden vectors upstream); this file
is pinned against the unmodified reference code itself in
``tests/test_oracle_vs_reference.py`` (build container only) and through the fixtures
written by ``tests/golden/make_golden.py``.
"""
from __future__ import annotations

from typing import Callable, Dict, Mapping, Optional, Sequence

import torch
import torch.nn.functional as F

from .shims import add_self_loops, scatter_add, scatter_softmax

Params = Mapping[str, torch.Tensor]
NEG_SLOPE = 0.2          # nn.LeakyReLU(0.2), gat2.py:83
# ``drop_fn(site, t)``: replaces ``F.dropout(t, drop_ratio, training)`` at one dropout site of an encoder.  ``site`` is
# ("input", "atoms" | "frags") for the dropout on the raw features, (layer, "atoms" | "frags" | "bond" | "fbond") for
# the ReLU(Dropout(.)) after a layer.  Tests pass one that applies a known keep-mask, to replay the masks of a run.
DropFn = Callable[[tuple, torch.Tensor], torch.Tensor]


def _dropper(drop_fn: Optional[DropFn], drop_ratio: float, training: bool):
    if drop_fn is None:
        return lambda site, t: F.dropout(t, drop_ratio, training)
    return drop_fn


def _linear(P: Params, name: str, x: torch.Tensor) -> torch.Tensor:
    return F.linear(x, P[name + ".weight"], P[name + ".bias"])


def attention_block(h: torch.Tensor, target: torch.Tensor, source: torch.Tensor,
                    edge_vec: torch.Tensor, alpha: torch.Tensor):
    """One GAT2 block over one graph.

    ``h`` [N,H,d] projected node features, ``edge_vec`` [E,De] per-edge vector shared by all
    heads, ``alpha`` [H, d+De+d].  Follows gat2.py:146-169 (bond graph), :196-224 (atom graph),
    :250-272 (fragment-connection graph), :286-316 (fragment graph):
    message = cat[target | edge | source]; logit = LeakyReLU(sum(message * alpha));
    softmax over the edges of each target; aggregate source features; and the per-SOURCE sum
    of attention probabilities (the interpretability weights).
    """
    n_nodes, n_heads = h.size(0), h.size(1)
    h_src = torch.index_select(h, 0, source)
    h_tgt = torch.index_select(h, 0, target)
    e_rep = edge_vec.repeat(n_heads, 1, 1).permute(1, 0, 2)
    message = torch.cat([h_tgt, e_rep, h_src], dim=-1)
    logits = F.leaky_relu(torch.sum(message * alpha, dim=2), NEG_SLOPE)
    probs = scatter_softmax(logits, target, dim=0)
    weighted = probs[..., None] * torch.index_select(h, 0, source)
    summed = scatter_add(weighted, target, dim=0)
    by_source = scatter_add(probs, source, dim=0)
    return summed.view(n_nodes, -1), by_source


def layer_forward(P: Params, prefix: str, num_heads: int,
                  x_atoms, edge_index, edge_attr, frag_index, x_frags, atom_to_frag_ids,
                  x_bond_nodes, edge_index_bonds_graph, edge_attr_bond_graph,
                  x_fbond_nodes, edge_index_fbond_graph, edge_attr_fbond_graph,
                  bond_mask: Optional[int] = None, frag_bond_mask: Optional[int] = None,
                  atom_mask_individual=None):
    """``FragNetLayerA.forward`` (gat2.py:121-330).  Returns the 8-tuple of gat2.py:318-328.

    ``x_frags`` and ``edge_attr`` are accepted and ignored exactly as in the reference
    (``x_frags`` is overwritten at gat2.py:234; ``edge_attr`` is only a dtype donor, :184).
    """
    p = lambda n: P[prefix + n]
    H = num_heads
    # -- bond graph: row 0 of the edge list is the softmax segment (gat2.py:138-169)
    tgt, src = edge_index_bonds_graph[0], edge_index_bonds_graph[1]
    ea = F.linear(edge_attr_bond_graph, p("edge_attr_bond_embed.weight"), p("edge_attr_bond_embed.bias"))
    hb = F.linear(x_bond_nodes, p("projection_b.weight"), p("projection_b.bias"))
    hb = hb.view(x_bond_nodes.size(0), H, -1)
    new_bond, attn_bonds = attention_block(hb, tgt, src, ea, p("a_b"))
    if bond_mask is not None:                                      # gat2.py:173-176
        with torch.no_grad():
            new_bond[bond_mask:bond_mask + 2, :] = 0.0
    # -- atom graph with appended self loops; row 1 is the segment (gat2.py:179-224)
    ei_loops, _ = add_self_loops(edge_index)
    loop_attr = torch.zeros(x_atoms.size(0), new_bond.size(1), dtype=new_bond.dtype)
    e_full = torch.cat((new_bond, loop_attr), dim=0)
    src, tgt = ei_loops[0], ei_loops[1]
    ha = F.linear(x_atoms, p("projection_a.weight"), p("projection_a.bias"))
    ha = ha.view(x_atoms.size(0), H, -1)
    x_atoms_new, attn_atoms = attention_block(ha, tgt, src, e_full, p("a"))
    if atom_mask_individual is not None:                           # gat2.py:227-231
        with torch.no_grad():
            x_atoms_new[atom_mask_individual, :] = 0.0
    # -- atom -> fragment sum pooling (gat2.py:234)
    x_frags_pooled = scatter_add(x_atoms_new, atom_to_frag_ids, dim=0)
    # -- fragment-connection graph; row 0 is the segment (gat2.py:239-272)
    tgt, src = edge_index_fbond_graph[0], edge_index_fbond_graph[1]
    eaf = F.linear(edge_attr_fbond_graph, p("edge_attr_fbond_embed.weight"), p("edge_attr_fbond_embed.bias"))
    hfb = F.linear(x_fbond_nodes, p("projection_fb.weight"), p("projection_fb.bias"))
    hfb = hfb.view(x_fbond_nodes.size(0), H, -1)
    new_fbond, attn_fbonds = attention_block(hfb, tgt, src, eaf, p("f_a_b"))
    if frag_bond_mask is not None:                                 # gat2.py:275-278
        with torch.no_grad():
            new_fbond[2 * frag_bond_mask, :] = 0.0
            new_fbond[2 * frag_bond_mask + 1, :] = 0.0
    # -- fragment graph, no projection, no self loops; row 1 is the segment (gat2.py:283-316)
    src, tgt = frag_index[0], frag_index[1]
    hf = x_frags_pooled.view(x_frags_pooled.size(0), H, -1)
    x_frags_new, attn_frags = attention_block(hf, tgt, src, new_fbond, p("f"))
    return (x_atoms_new, x_frags_new, new_bond, new_fbond,
            attn_atoms, attn_frags, attn_bonds, attn_fbonds)


def fragnet_forward(P: Params, batch: Dict[str, torch.Tensor], num_layer: int, num_heads: int = 4,
                    drop_ratio: float = 0.0, training: bool = False, prefix: str = "pretrain.",
                    masks: Optional[dict] = None, return_attentions: bool = False,
                    drop_fn: Optional[DropFn] = None):
    """``FragNet.forward`` (gat2.py:381-442): input dropout, layer 0 on raw features, then
    ``ReLU(Dropout(.))`` on the four outputs of every layer; layers >= 1 receive the bond
    features as both ``edge_attr`` and bond-graph node features (:421-434).

    With ``return_attentions`` the attention tensors of the LAST layer are appended, which is
    the arrangement of ``vizualize/model.py:72-142``.  ``drop_fn`` replaces ``F.dropout`` at every site (``DropFn``).
    """
    masks = masks or {}
    drop = _dropper(drop_fn, drop_ratio, training)
    post = lambda site, t: F.relu(drop(site, t))
    x_atoms = drop(("input", "atoms"), batch["x_atoms"])
    x_frags = drop(("input", "frags"), batch["x_frags"])
    edge_feat = batch["edge_attr"]
    bond_nodes = batch["node_features_bonds"]
    fbond_nodes = batch["node_features_fbonds"]
    attn = ()
    for li in range(num_layer):
        out = layer_forward(
            P, f"{prefix}layers.{li}.", num_heads,
            x_atoms, batch["edge_index"], edge_feat, batch["frag_index"], x_frags,
            batch["atom_to_frag_ids"], bond_nodes, batch["edge_index_bonds_graph"],
            batch["edge_attr_bonds"], fbond_nodes, batch["edge_index_fbonds"],
            batch["edge_attr_fbonds"], **masks)
        x_atoms, x_frags = post((li, "atoms"), out[0]), post((li, "frags"), out[1])
        edge_feat = post((li, "bond"), out[2])
        fedge_feat = post((li, "fbond"), out[3])
        bond_nodes, fbond_nodes = edge_feat, fedge_feat
        attn = out[4:]
    if return_attentions:
        return (x_atoms, x_frags, edge_feat, fedge_feat) + tuple(attn)
    return x_atoms, x_frags, edge_feat, fedge_feat


_ACTS = {"relu": F.relu, "silu": F.silu, "gelu": F.gelu, "celu": F.celu, "selu": F.selu,
         "relu6": F.relu6, "leakyrelu": F.leaky_relu}


def fthead_forward(P: Params, enc: torch.Tensor, fthead: str = "FTHead3", act: str = "relu",
                   drop_ratio: float = 0.0, training: bool = False, prefix: str = "fthead."):
    """Regression heads.  FTHead3: gat2.py:719-725 (``act(dropout(linear))`` per hidden layer);
    FTHead4: :669-675; FTHead1: :580-588; FTHead2: :745-751 (ReLU, p=0.1)."""
    drop = lambda t, p=drop_ratio: F.dropout(t, p, training)
    if fthead in ("FTHead3", "FTHead5", "FTHead2"):
        n = len([k for k in P if k.startswith(prefix + "predictor.") and k.endswith(".weight")])
        fn = F.relu if fthead == "FTHead2" else _ACTS[act]
        pd = 0.1 if fthead == "FTHead2" else drop_ratio
        for i in range(n - 1):
            enc = fn(drop(_linear(P, f"{prefix}predictor.{i}", enc), pd))
        return _linear(P, f"{prefix}predictor.{n - 1}", enc)
    if fthead == "FTHead4":
        x = _ACTS[act](_linear(P, prefix + "dense", drop(enc)))
        return _linear(P, prefix + "out_proj", drop(x))
    if fthead == "FTHead1":
        x = F.relu(_linear(P, prefix + "lin1", drop(enc)))
        return _linear(P, prefix + "out", drop(x))
    raise ValueError(fthead)


def readout(x_atoms, x_frags, batch):
    """Graph readout: per-molecule sums of atoms and fragments, concatenated
    (gat2.py:820-823, pretrain_heads.py:93-96)."""
    frags_pooled = scatter_add(x_frags, batch["frag_batch"], dim=0)
    atoms_pooled = scatter_add(x_atoms, batch["batch"], dim=0)
    return torch.cat((atoms_pooled, frags_pooled), 1)


def finetune_forward(P: Params, batch, num_layer: int = 4, num_heads: int = 4, drop_ratio: float = 0.0,
                     training: bool = False, fthead: str = "FTHead3", act: str = "relu"):
    """``FragNetFineTune.forward`` (gat2.py:816-826)."""
    x_atoms, x_frags, _, _ = fragnet_forward(P, batch, num_layer, num_heads, drop_ratio, training)
    return fthead_forward(P, readout(x_atoms, x_frags, batch), fthead, act, drop_ratio, training)


# ---- gat2_lite: bond graph + atom graph + pooling only (fragnet/model/gat/gat2_lite.py) ------------------------
def lite_layer_forward(P: Params, prefix: str, num_heads: int, x_atoms, edge_index, edge_attr, x_frags,
                       atom_to_frag_ids, x_bond_nodes, edge_index_bonds_graph, edge_attr_bond_graph):
    """``gat2_lite.FragNetLayerA.forward`` (gat2_lite.py:65-150): the bond block (:78-104), self loops with zero
    edge vectors and the atom block (:107-138), the pooling (:140).  Returns the 8-tuple of :143-148 (the
    fragment-side entries are ``None``)."""
    p = lambda n: P[prefix + n]
    H = num_heads
    tgt, src = edge_index_bonds_graph[0], edge_index_bonds_graph[1]
    ea = F.linear(edge_attr_bond_graph, p("edge_attr_bond_embed.weight"), p("edge_attr_bond_embed.bias"))
    hb = F.linear(x_bond_nodes, p("projection_b.weight"), p("projection_b.bias")).view(x_bond_nodes.size(0), H, -1)
    new_bond, attn_bonds = attention_block(hb, tgt, src, ea, p("a_b"))
    ei_loops, _ = add_self_loops(edge_index)
    e_full = torch.cat((new_bond, torch.zeros(x_atoms.size(0), new_bond.size(1), dtype=new_bond.dtype)), dim=0)
    src, tgt = ei_loops[0], ei_loops[1]
    ha = F.linear(x_atoms, p("projection_a.weight"), p("projection_a.bias")).view(x_atoms.size(0), H, -1)
    x_atoms_new, attn_atoms = attention_block(ha, tgt, src, e_full, p("a"))
    x_frags_new = scatter_add(x_atoms_new, atom_to_frag_ids, dim=0)
    return x_atoms_new, x_frags_new, new_bond, None, attn_atoms, None, attn_bonds, None


def lite_fragnet_forward(P: Params, batch, num_layer: int, num_heads: int = 4, drop_ratio: float = 0.0,
                         training: bool = False, prefix: str = "pretrain.", drop_fn: Optional[DropFn] = None):
    """``gat2_lite.FragNet.forward`` (gat2_lite.py:174-216): ``ReLU(Dropout(.))`` on atoms, pooled fragments and bond
    features after every layer; layers >= 1 take the bond features as edge attributes and bond-graph nodes.
    ``drop_fn``: as in ``fragnet_forward`` (no "fbond" site)."""
    drop = _dropper(drop_fn, drop_ratio, training)
    post = lambda site, t: F.relu(drop(site, t))
    x_atoms, x_frags = drop(("input", "atoms"), batch["x_atoms"]), drop(("input", "frags"), batch["x_frags"])
    edge_feat, bond_nodes = batch["edge_attr"], batch["node_features_bonds"]
    for li in range(num_layer):
        out = lite_layer_forward(P, f"{prefix}layers.{li}.", num_heads, x_atoms, batch["edge_index"], edge_feat, x_frags,
                                 batch["atom_to_frag_ids"], bond_nodes, batch["edge_index_bonds_graph"],
                                 batch["edge_attr_bonds"])
        x_atoms, x_frags, edge_feat = post((li, "atoms"), out[0]), post((li, "frags"), out[1]), post((li, "bond"), out[2])
        bond_nodes = edge_feat
    return x_atoms, x_frags, edge_feat, None


def lite_finetune_forward(P: Params, batch, num_layer: int = 4, num_heads: int = 4, drop_ratio: float = 0.0,
                          training: bool = False, fthead: str = "FTHead3", act: str = "relu"):
    """``gat2_lite.FragNetFineTune.forward`` (gat2_lite.py:498-509)."""
    x_atoms, x_frags, _, _ = lite_fragnet_forward(P, batch, num_layer, num_heads, drop_ratio, training)
    return fthead_forward(P, readout(x_atoms, x_frags, batch), fthead, act, drop_ratio, training)


def edge_layer_forward(P: Params, prefix: str, num_heads: int, x_atoms, edge_index, edge_attr, frag_index, x_frags,
                       atom_to_frag_ids, x_bond_nodes, edge_index_bonds_graph, edge_attr_bond_graph, cnx_attr):
    """``gat2_edge.FragNetLayerA.forward`` (gat2_edge.py:62-175): bond-graph block, atom-graph block with self loops,
    pooling, and the fragment-graph block whose edge vectors are ``cnx_attr_transform(cnx_attr)`` (:152-158).  Returns
    ``(x_atoms_new, x_frags_new, new_bond, attn_atoms, attn_frags, attn_bonds)`` (:172-173)."""
    p = lambda n: P[prefix + n]
    H = num_heads
    tgt, src = edge_index_bonds_graph[0], edge_index_bonds_graph[1]                      # :75
    ea = F.linear(edge_attr_bond_graph, p("edge_attr_bond_embed.weight"), p("edge_attr_bond_embed.bias"))
    hb = F.linear(x_bond_nodes, p("projection_b.weight"), p("projection_b.bias")).view(x_bond_nodes.size(0), H, -1)
    new_bond, attn_bonds = attention_block(hb, tgt, src, ea, p("a_b"))
    ei_loops, _ = add_self_loops(edge_index)                                              # :107-112
    e_full = torch.cat((new_bond, torch.zeros(x_atoms.size(0), new_bond.size(1), dtype=new_bond.dtype)), dim=0)
    src, tgt = ei_loops[0], ei_loops[1]
    ha = F.linear(x_atoms, p("projection_a.weight"), p("projection_a.bias")).view(x_atoms.size(0), H, -1)
    x_atoms_new, attn_atoms = attention_block(ha, tgt, src, e_full, p("a"))
    pooled = scatter_add(x_atoms_new, atom_to_frag_ids, dim=0)                            # :139
    src, tgt = frag_index[0], frag_index[1]                                               # :145
    hf = pooled.view(pooled.size(0), H, -1)
    cnx = F.linear(cnx_attr, p("cnx_attr_transform.weight"), p("cnx_attr_transform.bias"))
    x_frags_new, attn_frags = attention_block(hf, tgt, src, cnx, p("f"))
    return x_atoms_new, x_frags_new, new_bond, attn_atoms, attn_frags, attn_bonds


def edge_fragnet_forward(P: Params, batch, num_layer: int, num_heads: int = 4, drop_ratio: float = 0.0,
                         training: bool = False, prefix: str = "pretrain.", drop_fn: Optional[DropFn] = None):
    """``gat2_edge.FragNet.forward`` (gat2_edge.py:198-239).  ``drop_fn``: as in ``fragnet_forward`` (no "fbond"
    site)."""
    drop = _dropper(drop_fn, drop_ratio, training)
    post = lambda site, t: F.relu(drop(site, t))
    x_atoms, x_frags = drop(("input", "atoms"), batch["x_atoms"]), drop(("input", "frags"), batch["x_frags"])
    edge_feat, bond_nodes = batch["edge_attr"], batch["node_features_bonds"]
    for li in range(num_layer):
        out = edge_layer_forward(P, f"{prefix}layers.{li}.", num_heads, x_atoms, batch["edge_index"], edge_feat,
                                 batch["frag_index"], x_frags, batch["atom_to_frag_ids"], bond_nodes,
                                 batch["edge_index_bonds_graph"], batch["edge_attr_bonds"], batch["cnx_attr"])
        x_atoms, x_frags, edge_feat = post((li, "atoms"), out[0]), post((li, "frags"), out[1]), post((li, "bond"), out[2])
        bond_nodes = edge_feat
    return x_atoms, x_frags, edge_feat


def edge_finetune_forward(P: Params, batch, num_layer: int = 4, num_heads: int = 4, drop_ratio: float = 0.0,
                          training: bool = False, fthead: str = "FTHead3", act: str = "relu"):
    """``gat2_edge.FragNetFineTune.forward`` (gat2_edge.py:550-561)."""
    x_atoms, x_frags, _ = edge_fragnet_forward(P, batch, num_layer, num_heads, drop_ratio, training)
    return fthead_forward(P, readout(x_atoms, x_frags, batch), fthead, act, drop_ratio, training)


def _mlp_stack(P: Params, name: str, x: torch.Tensor, L: int, act_first: bool) -> torch.Tensor:
    if act_first:                       # bond-length head: activation BEFORE each linear (pretrain_heads.py:72-74)
        for l in range(L + 1):
            x = _linear(P, f"{name}.{l}", F.relu(x))
        return x
    for l in range(L):                  # other heads: linear, ReLU; last linear bare (:78-81, :85-88, :97-100)
        x = F.relu(_linear(P, f"{name}.{l}", x))
    return _linear(P, f"{name}.{L}", x)


def pretrain_heads_forward(P: Params, x_atoms, x_frags, edge_feat, batch, L: int = 2, prefix: str = "head."):
    """``PretrainTask.forward`` (pretrain_heads.py:64-102)."""
    ei = batch["edge_index"]
    pair = x_atoms[ei.T]
    z = torch.concat((pair[:, 0, :], pair[:, 1, :], edge_feat), axis=1)
    bond_length = _mlp_stack(P, prefix + "bl_layers", _linear(P, prefix + "bl_reduce_layer", z), L, True)
    bond_angle = _mlp_stack(P, prefix + "ba_layers", x_atoms, L, False)
    dihedral = _mlp_stack(P, prefix + "da_layers", edge_feat, L, False)
    energy = _mlp_stack(P, prefix + "FC_layers", readout(x_atoms, x_frags, batch), L, False)
    return bond_length, bond_angle, dihedral, energy


def pretrain_forward(P: Params, batch, num_layer: int = 4, num_heads: int = 4, drop_ratio: float = 0.0,
                     training: bool = False, drop_fn: Optional[DropFn] = None):
    """``FragNetPreTrain.forward`` (pretrain_heads.py:134-141).  ``drop_fn``: see ``fragnet_forward``."""
    x_atoms, x_frags, e_edge, _ = fragnet_forward(P, batch, num_layer, num_heads, drop_ratio, training,
                                                  drop_fn=drop_fn)
    return pretrain_heads_forward(P, x_atoms, x_frags, e_edge, batch)


def pretrain_loss(preds: Sequence[torch.Tensor], batch) -> torch.Tensor:
    """The loss the reference's pretraining loop actually optimises
    (train/pretrain/pretrain_utils.py:22-26): ``loss_lngth`` is overwritten by the dihedral
    term before use, so the total is 2*MSE(dihedral) + MSE(angle) + MSE(energy)."""
    _, angle, dihedral, energy = preds
    mse = F.mse_loss
    l_dh = mse(dihedral, batch["dh_angl"])
    return l_dh + mse(angle, batch["bnd_angl"]) + l_dh + mse(energy.view(-1), batch["y"])


def params_from_module(module: torch.nn.Module, requires_grad: bool = True) -> Dict[str, torch.Tensor]:
    """Detached CPU fp32 copies of a module's parameters keyed by state_dict name."""
    out = {}
    for k, v in module.state_dict().items():
        t = v.detach().to("cpu", torch.float32).clone()
        out[k] = t.requires_grad_(requires_grad) if t.is_floating_point() else t
    return out
