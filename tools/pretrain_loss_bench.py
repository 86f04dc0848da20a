"""Times the masked-region-classification (MVRC) loss of the pre-training task on one B200, fused vs torch.

    python tools/pretrain_loss_bench.py [--iters 300] [--warmup 10] [--steps 60] [--out FILE]

head: the MVRC head + loss alone, forward + backward, at B = 64, R = 100 (the pre-training shape) and R = 36 (config 6),
      C = 1601 classes, H = 768, 15 % of the regions masked (soft targets), the others all-zero.
        torch  the fp32 VisualLinguisticBertMVRCHead on every region + soft_cross_entropy as the reference writes it
               (common/utils/misc.py:124-144: host read of the valid count, boolean-mask gathers, fp32 log-softmax)
        fused  VisualLinguisticBertForPretraining.mvrc_loss with a static max_valid (sync-free)
      The targets (41 MB at R = 100) fit the 126 MB L2 and are not flushed between iterations.
step: the config-6 encoder step (VL-BERT-base 12L/768, 64 text + 36 region tokens, batch 64, dropout 0.1) with the whole
      pre-training objective mlm_loss + MVRC loss, forward + backward:
        eager_torch_mvrc  fused mlm_loss + the torch MVRC loss, launched eagerly (the host sync keeps it out of a graph)
        graphed_fused     fused mlm_loss + fused mvrc_loss, captured once in GraphedStep and replayed
        graphed_mlm_only  the same graph without the MVRC loss (config 6 of bench.py): what the MVRC loss adds to a step
Times are CUDA-event means over the timed iterations after warm-up.  One JSON line on stdout, with the card name and its
power limit.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import bench  # noqa: E402
import mvrc_oracle as mo  # noqa: E402

C, H, MASK = 1601, 768, 0.15


def torch_soft_cross_entropy(logits2d, targets2d):
    """the reference's formulation (common/utils/misc.py:124-144), reduction 'mean'"""
    valid = (targets2d.sum(1) - 1).abs() < 0.1
    if valid.sum().item() == 0:
        return logits2d.new_zeros(())
    return (-F.log_softmax(logits2d[valid], 1) * targets2d[valid]).sum(1).mean(0)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
    except Exception as e:                       # the numbers stay labelled with the card name
        q = "unavailable (%s)" % e
    return {"name": name, "power_limit_and_max_sm_clock": q}


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def config(w, p_drop):
    import vlbert_b200
    return vlbert_b200.default_config(hidden_size=w["hidden"], num_hidden_layers=w["layers"], num_attention_heads=w["heads"],
                                      intermediate_size=w["inter"], visual_size=w["hidden"], hidden_dropout_prob=p_drop,
                                      attention_probs_dropout_prob=p_drop, visual_region_classes=C)


def targets_for(B, R, seed, device):
    return mo.synth_targets(B, R, C, MASK, torch.Generator().manual_seed(seed)).to(device)


def head_bench(R, iters, warmup, dev):
    import vlbert_b200
    B = 64
    w = dict(bench.WORKLOADS[6], layers=1)
    torch.manual_seed(1)
    m = vlbert_b200.VisualLinguisticBertForPretraining(config(w, 0.0), with_rel_head=False, with_mlm_head=False).to(dev)
    g = torch.Generator().manual_seed(2)
    obj = torch.randn(B, R, H, generator=g).to(dev).requires_grad_(True)
    tgt = targets_for(B, R, 3, dev)
    n_valid = int(mo.valid_rows(tgt).sum())
    cap = int(B * R * MASK * 1.5)              # static bound: 1.5x the expected masked count

    def torch_step():
        loss = torch_soft_cross_entropy(m.mvrc_head(obj).view(-1, C), tgt.view(-1, C))
        loss.backward()
        return loss

    def fused_step():
        loss, _, _ = m.mvrc_loss(obj, tgt, max_valid=cap)
        loss.backward()
        return loss

    l_t, l_f = float(torch_step().detach()), float(fused_step().detach())
    ms_t, ms_f = timed(torch_step, iters, warmup), timed(fused_step, iters, warmup)
    return {"B": B, "R": R, "C": C, "H": H, "valid_rows": n_valid, "max_valid": cap, "torch_ms": round(ms_t, 4),
            "fused_ms": round(ms_f, 4), "speedup": round(ms_t / ms_f, 3), "loss_torch": l_t, "loss_fused": l_f,
            "loss_rel_diff": abs(l_f - l_t) / abs(l_t)}


def step_bench(steps, warmup, dev):
    import vlbert_b200
    w = bench.WORKLOADS[6]
    B, R = w["batch"], w["regions"]
    torch.manual_seed(12345)
    m = vlbert_b200.VisualLinguisticBertForPretraining(config(w, bench.P_DROP), with_rel_head=False).to(dev)
    m.visual_ln_text.weight.data.fill_(1.0)
    m.max_length_hint = bench.seq_len(w)
    m.train()
    inputs = bench.make_inputs(w, B, 7, dev) + [targets_for(B, R, 8, dev)]
    n_lab, cap = B * 10, int(B * R * MASK * 1.5)

    def encode(ids, types, tvis, tmask, ovl, omask):
        return vlbert_b200.VisualLinguisticBert.forward(m, ids, types, tvis, tmask, ovl, omask, output_all_encoded_layers=False,
                                                        output_text_and_object_separately=True)

    def loss_torch(mm, ids, types, tvis, tmask, ovl, omask, labels, mvrc):
        text_out, object_out, _ = encode(ids, types, tvis, tmask, ovl, omask)
        l_mlm, _, _ = mm.mlm_loss(text_out, labels, max_labelled=n_lab)
        return l_mlm + torch_soft_cross_entropy(mm.mvrc_head(object_out).view(-1, C), mvrc.view(-1, C))

    def loss_fused(mm, ids, types, tvis, tmask, ovl, omask, labels, mvrc):
        text_out, object_out, _ = encode(ids, types, tvis, tmask, ovl, omask)
        l_mlm, _, _ = mm.mlm_loss(text_out, labels, max_labelled=n_lab)
        l_mvrc, _, _ = mm.mvrc_loss(object_out, mvrc, max_valid=cap)
        return l_mlm + l_mvrc

    def eager():
        m.zero_grad(set_to_none=True)
        loss_torch(m, *inputs).backward()

    def loss_mlm_only(mm, ids, types, tvis, tmask, ovl, omask, labels, mvrc):
        text_out, _, _ = encode(ids, types, tvis, tmask, ovl, omask)
        return mm.mlm_loss(text_out, labels, max_labelled=n_lab)[0]

    ms_eager = timed(eager, steps, warmup)
    graphed = vlbert_b200.GraphedStep(m, loss_fused, inputs, warmup=3)
    ms_graph = timed(lambda: graphed(), steps, warmup)
    del graphed
    graphed_mlm = vlbert_b200.GraphedStep(m, loss_mlm_only, inputs, warmup=3)
    ms_mlm = timed(lambda: graphed_mlm(), steps, warmup)
    return {"config": w["name"], "B": B, "R": R, "mlm_labelled": n_lab, "mvrc_max_valid": cap, "eager_torch_mvrc_ms": round(ms_eager, 3),
            "graphed_fused_ms": round(ms_graph, 3), "speedup": round(ms_eager / ms_graph, 3),
            "samples_per_s_graphed": round(B / ms_graph * 1e3, 1), "graphed_mlm_only_ms": round(ms_mlm, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=300, help="timed iterations of the head measurements")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--steps", type=int, default=60, help="timed encoder steps")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pretrain_loss_bench.py needs a CUDA device")
    dev = "cuda"
    rec = {"tool": "pretrain_loss_bench", "card": card(),
           "head": [head_bench(R, a.iters, a.warmup, dev) for R in (100, 36)],
           "step": step_bench(a.steps, max(3, a.warmup // 2), dev)}
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
