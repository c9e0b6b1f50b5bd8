#!/usr/bin/env python
"""generate.py - synthetic visual-dialog generation with the questioner and teacher models (CLI of the reference's
generate.py: same single-dash flags, same output JSON layout), running on the B200 engine.

    python generate.py -mode cc12m_gen -start_path_q ckpt_q -start_path_a ckpt_a -cc12m_image_feats ... -save_name out.json
    python generate.py -synthetic 128 -batch_size 64 -num_beams 5          # seeded synthetic images + random weights
    python generate.py -synthetic 128 -batch_size 64 -num_beams 5 -q_num_beams 5   # beam-searched questions too (4-gram blocked)
    python generate.py -synthetic 128 -batch_size 64 -answer_candidates 5          # 5 sampled answers per round, lowest perplexity kept
    python generate.py -synthetic 128 -batch_size 64 -num_beams 6 -num_beam_groups 3 -diversity_penalty 0.5 -answer_candidates 6
                                                                                   # diverse beams ranked by perplexity

Multi-GPU: launch with torchrun (one process per GPU); images are sharded by rank and gathered once at the end.
The dataset readers (LMDB / tokenizer) of the reference are host I/O outside the hot path: without them (-synthetic)
the script uses the seeded generators of gst_visdial_b200.synthetic and writes token ids instead of decoded text.
"""
from __future__ import annotations

import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from gst_visdial_b200 import dist as D  # noqa: E402
from gst_visdial_b200 import options  # noqa: E402
from gst_visdial_b200 import synthetic as S  # noqa: E402
from gst_visdial_b200 import weights as W  # noqa: E402
from gst_visdial_b200.dialog import generate_dialogs  # noqa: E402
from gst_visdial_b200.io import output as IOO  # noqa: E402
from gst_visdial_b200.models.visual_dialog_decoder import VisualDialogDecoder  # noqa: E402
from gst_visdial_b200.models.visual_dialog_encoder import VisualDialogEncoder  # noqa: E402
from gst_visdial_b200.models.visual_dialog_model import EncoderDecoderModel  # noqa: E402


def build_model(params, model_name, ckpt_path, seed):
    p = dict(params)
    p['model'] = model_name
    enc, dec = VisualDialogEncoder(p), VisualDialogDecoder(p)
    dec.decoder.bert.embeddings = enc.bert_pretrained.bert.embeddings          # generate.py:65
    model = EncoderDecoderModel(p, enc, dec)
    model = torch.nn.DataParallel(model, [p['gpu_ids'][0]])
    if ckpt_path:
        ckpt = torch.load(ckpt_path, map_location='cpu')
        model.module.load_state_dict(ckpt['model_state_dict'])
        print(f"model successfully loaded from {ckpt_path}")
    else:
        model.module.load_state_dict(W.synthetic_state_dict(enc.config, dec.config, seed=seed))
        print(f"[{model_name}] no checkpoint given: seeded random weights (seed {seed})")
    model.to(p['device']).eval()
    return model


def ids_to_text(row):
    return " ".join(str(int(t)) for t in row if int(t) != 0)


def main(argv=None):
    params = options.read_command_line(argv)
    rank, world, local = D.init_from_env("nccl")
    if world > 1:
        params['gpu_ids'] = [local]
        params['device'] = f"cuda:{local}"
    torch.cuda.set_device(params['device'])
    shards = None
    if params['feature_shards']:
        from gst_visdial_b200.io import features as IOF
        shards = IOF.FeatureShards([d for d in params['feature_shards'].split(',') if d])
        captions = {int(k): v for k, v in json.load(open(params['caption_ids'])).items()} if params['caption_ids'] else {}
        all_ids = sorted(shards.image_ids())
    elif params['synthetic'] <= 0:
        raise SystemExit("give -feature_shards DIR[,DIR] (+ -caption_ids) or -synthetic N; the reference's LMDB / tokenizer readers are "
                         "host I/O outside this package (convert an LMDB once with gst_visdial_b200.io.features)")
    q_model = build_model(params, 'enc_dec_q', params['start_path_q'], seed=7)
    a_model = build_model(params, 'enc_dec_a', params['start_path_a'], seed=0)
    enc_cfg = a_model.module.encoder.config
    total = len(all_ids) if shards is not None else params['synthetic']
    start, end = D.shard_range(total, rank, world)
    a_kwargs = dict(temperature=0.7, top_k=7, top_p=0.0, ngram_blocking_size=0)
    if params['num_beams'] > 1:
        a_kwargs.update(num_beams=params['num_beams'], num_beam_groups=params['num_beam_groups'], diversity_penalty=params['diversity_penalty'])
        if params['beam_sample']:
            a_kwargs.update(do_sample=True)
    q_kwargs = dict(temperature=0.7, top_k=7, top_p=0.0, ngram_blocking_size=4)
    if params['q_num_beams'] > 1:
        q_kwargs.update(num_beams=params['q_num_beams'], num_beam_groups=params['q_num_beam_groups'],
                        diversity_penalty=params['q_diversity_penalty'])
        if params['q_beam_sample']:
            q_kwargs.update(do_sample=True)
    decode = None
    if params['vocab_file']:
        from transformers import BertTokenizer
        tok = BertTokenizer(params['vocab_file'])
        decode = lambda ids: tok.decode(ids, skip_special_tokens=True)      # noqa: E731  (generate.py:18-23)
    bs = params['batch_size']
    spans = [(s, min(bs, end - s)) for s in range(start, end, bs)]

    def batches():
        if shards is None:
            for s, n in spans:
                yield S.synthetic_batch(s, n, vocab_size=enc_cfg.vocab_size, v_feature_size=enc_cfg.v_feature_size, max_seq_len=params['max_seq_len'])
        else:
            id_batches = [all_ids[s:s + n] for s, n in spans]
            for ids, fb in zip(id_batches, IOF.Prefetcher(shards, id_batches, depth=2)):
                fb.update(IOF.caption_batch([captions.get(i, []) for i in ids], max_seq_len=params['max_seq_len']))
                yield fb

    # every finished batch is appended to this rank's JSON-lines file by a writer thread (gst_visdial_b200/io/output.py)
    final = os.path.join(params['save_path'], params['save_name'])
    part = f"{final}.rank{rank}.jsonl"
    # A failing rank must not leave the others hanging in the barrier, and rank 0 must not merge partial files: every rank
    # reports a status flag (one all_reduce) before the merge and all of them raise if any failed.
    failure = None
    try:
        with torch.no_grad(), IOO.JsonlWriter(part) as writer:
            for (span_start, _), batch in zip(spans, batches()):
                # sampling keyed by (-seed, model role, round, GLOBAL image index, step): the tokens of an image do not depend on the
                # batch size or on how many ranks share the job
                res = generate_dialogs(a_model, batch, q_model=q_model, num_rounds=params['num_rounds'], a_kwargs=a_kwargs, q_kwargs=q_kwargs,
                                       with_ppl=True, device=params['device'], seed=params.get('seed', 0), row_offset=span_start,
                                       answer_candidates=params['answer_candidates'])
                meta = {int(i): {"url": "", "caption": (decode or ids_to_text)(IOO.strip_ids(row) if decode else row)}
                        for i, row in zip(batch["image_id"].tolist(), batch["enc_input_ids"].tolist())}
                writer.write(IOO.batch_records(batch["image_id"], res.questions, res.answers, res.answer_ppl, res.abnormal,
                                               decode=decode or ids_to_text, meta=meta))
    except Exception as e:                                                   # noqa: BLE001 - reported to every rank below
        failure = e
    if world > 1:
        flag = torch.tensor([1 if failure is not None else 0], device=params['device'])
        torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MAX)
        if int(flag.item()) and failure is None:
            failure = RuntimeError("another rank failed while generating; no output was merged")
    if failure is not None:
        if world > 1:
            torch.distributed.destroy_process_group()
        raise failure
    if rank == 0:
        merged = f"{final}.jsonl"
        with open(merged, "w") as dst:
            for r in range(world):
                with open(f"{final}.rank{r}.jsonl") as src:
                    for line in src:
                        dst.write(line)
                os.remove(f"{final}.rank{r}.jsonl")
        n = IOO.jsonl_to_reference_json(merged, final)                     # the reference's single-array file (generate.py:258)
        print(f"wrote {n} dialogs to {final} (streamed copy: {merged})")
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
