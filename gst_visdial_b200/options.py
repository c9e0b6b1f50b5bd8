"""Command-line flags of the generation scripts: the reference's single-dash flags (options.py:13-88) that the
generation / scoring path reads, with the same names and defaults, plus a few additions for the B200 path."""
from __future__ import annotations

import argparse
import os

from . import weights as W


def read_command_line(argv=None):
    p = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    # ---- reference flags (options.py) ----
    p.add_argument('-start_path', default='', help='path of starting model checkpt')
    p.add_argument('-start_path_q', default='', help='path of starting questioner model checkpt')
    p.add_argument('-start_path_a', default='', help='path of starting answerer model checkpt')
    p.add_argument('-model_enc_config', default=W.DEFAULT_ENC_CONFIG, help='model definition of the bert model')
    p.add_argument('-model_dec_config', default=W.DEFAULT_DEC_CONFIG, help='model definition of the bert model')
    p.add_argument('-cc12m_image_feats', default='data/cc12m/features/', help='LMDB / shard directory of region features')
    p.add_argument('-cc12m_caption', default='', help='caption json of the chunk')
    p.add_argument('-chunk', default='', help='the number of chunks to use')
    p.add_argument('-threshold', default=50, type=int, help='perplexity-based data selection threshold')
    p.add_argument('-mode', default='cc12m_gen', type=str,
                   choices=['vd_train', 'vd_eval_val', 'vd_eval_test', 'vd_gen_val', 'cc12m_gen', 'cc12m_train'])
    p.add_argument('-model', default='enc_dec_a', type=str, choices=['enc_only_a', 'enc_dec_a', 'enc_dec_q'])
    p.add_argument('-num_workers', default=8, type=int)
    p.add_argument('-batch_size', default=72, type=int)
    p.add_argument('-select_data', action='store_true', help='using perplexity-based data selection')
    p.add_argument('-gpu_ids', nargs="+", type=int, default=[0], help="List of ids of GPUs to use.")
    p.add_argument('-max_seq_len', default=256, type=int, help='maximum sequence length for the dialog sequence')
    p.add_argument('-max_utt_len', default=25, type=int, help='maximum sequence length for each utterance')
    p.add_argument('-save_path', default='checkpoints/', help='Path to save outputs')
    p.add_argument('-save_name', default='', help='file name to save')
    # ---- additions ----
    p.add_argument('-compute_dtype', default='bf16', choices=['bf16', 'fp32'], help='arithmetic of the CUDA engine')
    p.add_argument('-num_beams', default=1, type=int, help='>1: beam search for the answers instead of top-k sampling')
    p.add_argument('-q_num_beams', default=1, type=int,
                   help='>1: beam search for the questions instead of top-k sampling (keeps the 4-gram blocking against the question history)')
    p.add_argument('-num_beam_groups', default=1, type=int,
                   help='>1: diverse beam search for the answers: the -num_beams beams in this many groups (must divide -num_beams)')
    p.add_argument('-diversity_penalty', default=0.0, type=float,
                   help='Hamming diversity penalty between the answer beam groups (with -num_beam_groups > 1)')
    p.add_argument('-q_num_beam_groups', default=1, type=int,
                   help='>1: diverse beam search for the questions: the -q_num_beams beams in this many groups (must divide -q_num_beams)')
    p.add_argument('-q_diversity_penalty', default=0.0, type=float,
                   help='Hamming diversity penalty between the question beam groups (with -q_num_beam_groups > 1)')
    p.add_argument('-beam_sample', action='store_true',
                   help='beam sampling for the answers (HF do_sample with beams): -num_beams > 1 beams drawn with the answer sampler\'s '
                        'temperature 0.7 and top-k 7; with -answer_candidates N, N independent searches per image')
    p.add_argument('-q_beam_sample', action='store_true',
                   help='beam sampling for the questions: -q_num_beams > 1 beams drawn with temperature 0.7 and top-k 7')
    for who, what in (('', 'answers'), ('q_', 'questions')):
        p.add_argument(f'-{who}repetition_penalty', default=1.0, type=float,
                       help=f'HF repetition penalty for the {what}: scores of ids already in the decoder input are divided (or, when '
                            'negative, multiplied) by it; 1 = off')
        p.add_argument(f'-{who}no_repeat_ngram_size', default=0, type=int,
                       help=f'HF no_repeat_ngram_size for the {what}: no n-gram occurs twice in the decoder input; 0 = off')
        p.add_argument(f'-{who}min_length', default=0, type=int,
                       help=f'HF min_length for the {what}: [SEP] is banned while the decoder input ([CLS] included) is shorter; 0 = off')
    p.add_argument('-answer_candidates', default=1, type=int,
                   help='>1: the teacher draws this many answers per round (samples, or the best of its -num_beams beams) and the one with '
                        'the lowest perplexity goes into the dialog')
    p.add_argument('-synthetic', default=0, type=int, help='generate dialogs for N seeded synthetic images (no dataset / checkpoint needed)')
    p.add_argument('-feature_shards', default='', help='comma-separated shard directories (gst_visdial_b200.io.features) instead of the LMDB')
    p.add_argument('-caption_ids', default='', help='json {image_id: [caption token ids]} for the images of the shards (pre-tokenized captions)')
    p.add_argument('-vocab_file', default='', help='optional BERT vocab.txt: decode the generated ids to text in the output')
    p.add_argument('-num_options', default=100, type=int, help='answer options per round (evaluate_gen.py)')
    p.add_argument('-num_rounds', default=10, type=int)
    p.add_argument('-seed', default=0, type=int)
    args = p.parse_args(argv)
    params = vars(args)
    for who, beams, groups, penalty in (('', 'num_beams', 'num_beam_groups', 'diversity_penalty'),
                                        ('q_', 'q_num_beams', 'q_num_beam_groups', 'q_diversity_penalty')):
        if params[groups] < 1 or params[groups] > 1 and (params[beams] <= 1 or params[beams] % params[groups] != 0):
            p.error(f"-{groups} {params[groups]} must be 1 or divide -{beams} {params[beams]} > 1")
        if not (0.0 <= params[penalty] < float('inf')):
            p.error(f"-{penalty} must be finite and >= 0")
    for who in ('', 'q_'):
        rp = params[f'{who}repetition_penalty']
        if not (0.0 < rp < float('inf')):
            p.error(f"-{who}repetition_penalty must be finite and > 0 (1 = off)")
        for name in ('no_repeat_ngram_size', 'min_length'):
            if params[who + name] < 0:
                p.error(f"-{who}{name} must be >= 0 (0 = off)")
    for flag, beams, groups in (('beam_sample', 'num_beams', 'num_beam_groups'), ('q_beam_sample', 'q_num_beams', 'q_num_beam_groups')):
        if params[flag] and (params[beams] <= 1 or params[groups] > 1):
            p.error(f"-{flag} needs -{beams} > 1 and no beam groups")
    if params['beam_sample'] and params['num_beams'] * params['answer_candidates'] > 8:
        p.error("-beam_sample runs -answer_candidates searches of -num_beams beams per image: their product must be at most 8")
    params['device'] = f"cuda:{params['gpu_ids'][0]}"
    params['engine_max_batch'] = params['batch_size']
    params['engine_max_beams'] = max(1, params['num_beams'], params['q_num_beams'], params['answer_candidates'],
                                     params['num_beams'] * params['answer_candidates'] if params['beam_sample'] else 1)
    if params['save_name'] == '':
        params['save_name'] = 'generated_dialogs.json'
    os.makedirs(params['save_path'], exist_ok=True)
    return params
