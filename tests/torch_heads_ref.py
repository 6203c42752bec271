"""Torch restatement of the models' head post-processing (pyramid.py:291-309, 331-332), with neg_max per level -- the gradient
oracle of the head-map training path: torch autograd through `heads` on the CPU is what the library's map gradients are checked
against.  The code is oracle/make_golden.py's ref_heads (which cannot be imported without the reference) with the level's reduction
chosen by neg_max[l] instead of by the level index.  Test / bench infrastructure, not product code."""
import torch


def heads(loc_maps, conf_maps, neg_max, softmax):
    """loc_maps[l] / conf_maps[l]: [B,4,H_l,W_l] tensors -> (loc[B,N,4], conf[B,N,2]).  neg_max[l] != 0: neg = max(ch0..2),
    pos = ch3 (pyramid.py:293-297); else neg = ch0, pos = max(ch1..3) (:299-304)."""
    loc, conf = [], []
    for lx, tmp_conf, nm in zip(loc_maps, conf_maps, neg_max):
        if nm:
            a, b, c, pos_conf = tmp_conf.chunk(4, 1)
            neg_conf = torch.cat([a, b, c], 1)
            max_conf, _ = neg_conf.max(1)
            max_conf = max_conf.view_as(pos_conf)
            conf.append(torch.cat([max_conf, pos_conf], 1).permute(0, 2, 3, 1).contiguous())
        else:
            neg_conf, a, b, c = tmp_conf.chunk(4, 1)
            pos_conf = torch.cat([a, b, c], 1)
            max_conf, _ = pos_conf.max(1)
            max_conf = max_conf.view_as(neg_conf)
            conf.append(torch.cat([neg_conf, max_conf], 1).permute(0, 2, 3, 1).contiguous())
        loc.append(lx.permute(0, 2, 3, 1).contiguous())
    loc = torch.cat([o.view(o.size(0), -1) for o in loc], 1)
    conf = torch.cat([o.view(o.size(0), -1) for o in conf], 1)
    loc = loc.view(loc.size(0), -1, 4)
    conf = conf.view(conf.size(0), -1, 2)
    if softmax:
        conf = torch.nn.Softmax(dim=-1)(conf)
    return loc, conf
