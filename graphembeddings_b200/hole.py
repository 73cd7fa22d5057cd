"""`holE.py` rewritten on top of libhole_b200 -- same flags, same files in --data_dir, same
outputs in --output_dir, no TensorFlow.

    python -m graphembeddings_b200.hole --data_dir D --output_dir O [flags of holE.py:598-619]
    python -m graphembeddings_b200.hole --data_dir D --output_dir O --infer

Function names follow the reference: init_data (holE.py:44-94), evaluate_batch (205-234),
run_training (249-370), init_inference_data (381-424), eval_link_prediction (427-472),
score_mrr (475-490), infer_triples (530-582).  Differences, all deliberate and listed in
DESIGN.md: triples come from a device-resident per-epoch permutation instead of a TF shuffle
queue; every validation point scores the WHOLE triples-valid.txt on the device (the reference's TODO,
holE.py:350) and writes the reference's scalar / histogram summaries to a TensorBoard events file; corruption is the Philox sampler (--padded_size accepted, unused); `--infer` runs the
all-entity filtered head+tail protocol with the unreachable `infer_threshold` gate off unless
--infer_gate is given; --save_embeddings is rejected (a py2-only debug dump).  --log_loss,
--negative_ratio and --l2_regularization select the logistic branch (holE.py:194-196, 206-220).
"""
import argparse
import errno
import os
import sys
import time
from collections import defaultdict

import numpy as np
import torch

from . import data as D
from . import tf_bundle
from . import tf_events
from .engine import (HOLE_RANK_BF16, HOLE_RANK_BF16X3, HOLE_SIDE_HEAD, HOLE_SIDE_RELATION, HOLE_SIDE_TAIL,
                     HoleEngine, inverse_time_decay)

_SIDES = {"tail": HOLE_SIDE_TAIL, "head": HOLE_SIDE_HEAD, "relation": HOLE_SIDE_RELATION}


def _candidate_range(side_name, relation_count, entity_count):
    """Rows a side ranks: the entity rows for "tail" / "head", the relation rows for "relation"."""
    return (0, relation_count) if side_name == "relation" else (relation_count, entity_count)

FLAGS = None


class HolEData(object):
    """Pre-processing data used during training and inference (holE.py:25-34)."""

    def __init__(self):
        self.type_to_ids = defaultdict(list)
        self.id_to_type = dict()
        self.entity_count = 0
        self.relation_count = 0
        self.triple_count = 0
        self.triples = None
        self.validation_triples = None


class HolEInferenceData(HolEData):
    """holE.py:373-378"""

    def __init__(self):
        self.id_to_metadata = dict()
        self.true_triples = defaultdict(lambda: defaultdict(set))
        self.test_triples = defaultdict(lambda: defaultdict(set))
        super(HolEInferenceData, self).__init__()


class InferenceCandidates(object):
    """holE.py:493-498"""

    def __init__(self, relations, tail_candidates, max_triples, min_confidence):
        self.relations = relations
        self.tail_candidates = tail_candidates
        self.max_triples = max_triples
        self.min_confidence = min_confidence


# --------------------------------------------------------------------------------------
# data
# --------------------------------------------------------------------------------------
def init_data(flags=None):
    """Model pre-processing (holE.py:44-94) without the TF reader graph: triples are loaded
    once as int32 [T,3] = (head, tail, relation)."""
    flags = flags or FLAGS
    entity_file = os.path.join(flags.data_dir, 'entity_metadata.tsv')
    relation_file = os.path.join(flags.data_dir, 'relation_ids.txt')
    train_triple_file = os.path.join(flags.data_dir, 'triples.txt')
    valid_triple_file = os.path.join(flags.data_dir, 'triples-valid.txt')

    data = HolEData()
    data.relation_count = D.count_lines(relation_file)
    md = D.load_entity_metadata(entity_file)
    data.entity_count = md.entity_count
    data.type_to_ids = md.type_to_ids
    data.id_to_type = md.id_to_type
    data.triples = D.load_triples(train_triple_file)
    data.triple_count = data.triples.shape[0]
    data.validation_triples = D.load_triples(valid_triple_file)
    D.check_triple_ids(data.triples, data.entity_count, data.relation_count, train_triple_file)
    D.check_triple_ids(data.validation_triples, data.entity_count, data.relation_count, valid_triple_file)
    if len(data.id_to_type) != data.entity_count or (data.id_to_type and max(data.id_to_type) != data.entity_count - 1):
        raise ValueError(f"{entity_file}: the Index column must cover rows 0..{data.entity_count - 1} exactly once "
                         "(every table row needs a type for the corruption sampler)")
    print('Entities: ', data.entity_count - data.relation_count, 'Relations: ', data.relation_count,
          'Triples: ', data.triple_count)
    print('Types: ', {k: len(v) for k, v in data.type_to_ids.items()} if len(data.type_to_ids) < 40
          else f'{len(data.type_to_ids)} types')
    return data


def init_inference_data(flags=None):
    """holE.py:381-424: candidate pools per type (mentions >= min_mentions or id starting with
    'P'), test triples and the train/valid-true sets for (h, r) pairs present in test."""
    flags = flags or FLAGS
    data = HolEInferenceData()
    md = D.load_entity_metadata(os.path.join(flags.data_dir, 'entity_metadata.tsv'))
    data.entity_count = md.entity_count
    data.id_to_type = md.id_to_type
    for index, meta in md.id_to_metadata.items():
        diffbot_id = meta.split(' ', 1)[0]
        if md.mentions[index] >= flags.min_mentions or diffbot_id.startswith('P'):
            data.type_to_ids[md.id_to_type[index]].append(index)
        data.id_to_metadata[index] = meta
    data.relation_count = D.count_lines(os.path.join(flags.data_dir, 'relation_ids.txt'))
    data.test = D.load_triples(os.path.join(flags.data_dir, 'test_positive_triples.txt'))
    D.check_triple_ids(data.test, data.entity_count, data.relation_count, 'test_positive_triples.txt')
    for h, t, r in data.test.tolist():
        data.test_triples[h][r].add(t)
    known = []
    for name in ('triples.txt', 'triples-valid.txt'):
        path = os.path.join(flags.data_dir, name)
        if os.path.exists(path):
            known.append(D.load_triples(path))
            D.check_triple_ids(known[-1], data.entity_count, data.relation_count, name)
    data.known = np.concatenate(known) if known else np.zeros((0, 3), np.int32)
    # true_triples[h][r] only for (h, r) pairs present in test (holE.py:421-422): cut the known triples
    # down to those pairs with one sort-based pass instead of walking 3e7 rows in Python
    if len(data.known) and len(data.test):
        kq = (data.test[:, 0].astype(np.int64) << 32) | data.test[:, 2].astype(np.int64)
        kk = (data.known[:, 0].astype(np.int64) << 32) | data.known[:, 2].astype(np.int64)
        for h, t, r in data.known[np.isin(kk, kq)].tolist():
            data.true_triples[h][r].add(t)
    return data


# --------------------------------------------------------------------------------------
# model pieces on the engine
# --------------------------------------------------------------------------------------
def make_engine(entity_count, relation_count, dim, embeddings, id_to_type=None, device=0):
    eng = HoleEngine(entity_count, dim, device).set_embeddings(embeddings)
    eng.set_relation_count(max(1, relation_count))
    if id_to_type is not None:
        names = {}
        type_of = np.full(entity_count, -1, dtype=np.int32)
        for idx, t in id_to_type.items():
            type_of[idx] = names.setdefault(t, len(names))
        if (type_of < 0).any():
            raise ValueError(f"{int((type_of < 0).sum())} table rows have no type in the metadata "
                             f"(first: {int(np.flatnonzero(type_of < 0)[0])})")
        off, ids = D.build_type_csr(type_of, len(names))
        eng.set_types(type_of, off, ids)
    return eng


def evaluate_batch(eng, triple_batch, seed, step, margin):
    """holE.py:222-234 without the update: corrupt, score both, hinge.  Returns
    (loss[B], sigma_pos[B], sigma_neg[B]) device tensors."""
    t = torch.as_tensor(triple_batch, dtype=torch.int32).to(eng.device)
    side, neg = eng.corrupt_batch(t, seed, step)
    corrupt = t.clone()
    corrupt[:, 0 if side else 1] = neg
    vp, vn = eng.evaluate_triples(t), eng.evaluate_triples(corrupt)
    return torch.clamp(vp - vn + margin, min=0.0), vp, vn


def evaluate_batch_logloss(eng, triple_batch, seed, step, l2, negative_ratio):
    """holE.py:206-221 without the update: rows [(1 + k), B] = log(1 + exp(-label * score)) +
    l2 * l2_loss(embeddings) for the positives and k corrupt batches (virtual steps step*k + j,
    as in hole_train_step_logloss).  Forward only (validation); computed from the device scores."""
    t = torch.as_tensor(triple_batch, dtype=torch.int32).to(eng.device)
    k = int(negative_ratio)
    rows = [-torch.log(eng.evaluate_triples(t))]                 # log(1+exp(-s)) = -log(sigmoid(s))
    for j in range(k):
        side, neg = eng.corrupt_batch(t, seed, step * k + j)
        corrupt = t.clone()
        corrupt[:, 0 if side else 1] = neg
        rows.append(-torch.log1p(-eng.evaluate_triples(corrupt)))  # log(1+exp(s)) = -log(1 - sigmoid(s))
    l2_loss = 0.5 * (eng.table.double() ** 2).sum()
    return torch.stack(rows) + float(l2) * l2_loss.float()


def summarize(var):
    """holE.py:237-246: mean / stddev / max / min of a tensor."""
    mean = var.mean()
    return {"mean": float(mean), "stddev": float(torch.sqrt(((var - mean) ** 2).mean())),
            "max": float(var.max()), "min": float(var.min())}


ADAGRAD_SLOT = "embeddings/Adagrad"


def check_optimizer_flags(flags):
    """The training branches that have no AdaGrad form exit before anything is trained."""
    if getattr(flags, 'optimizer', 'sgd') != 'adagrad':
        return
    if flags.log_loss:
        raise SystemExit("--optimizer adagrad has no --log_loss branch (its L2 gradient would make the update dense)")
    if getattr(flags, 'score_variant', 'complex') != 'complex':
        raise SystemExit("--optimizer adagrad is not available with --score_variant ccorr_tanh")
    if not flags.adagrad_initial_accumulator > 0:
        raise SystemExit("--adagrad_initial_accumulator must be > 0")


def save_checkpoint(eng, output_dir, global_step, metadata_names=None):
    """saver.save(sess, output_dir + '/model.ckpt') (holE.py:359) + checkpoint state file."""
    E = eng.embeddings().cpu().numpy()
    tensors = {"embeddings": E, "batch/Variable": np.array(global_step, dtype=np.int32)}
    if eng.accum is not None:       # AdagradOptimizer's slot, under the name TF's Saver gives it
        tensors[ADAGRAD_SLOT] = eng.accumulator().cpu().numpy()
    tf_bundle.save_bundle(os.path.join(output_dir, 'model.ckpt'), tensors)
    tf_bundle.write_checkpoint_state(output_dir)


def load_checkpoint(output_dir):
    """saver.restore(sess, output_dir + '/model.ckpt') (holE.py:313-314)."""
    b = tf_bundle.load_bundle(os.path.join(output_dir, 'model.ckpt'), names={"embeddings", "batch/Variable"})
    return b["embeddings"], int(np.asarray(b.get("batch/Variable", 0)).reshape(-1)[0])


def load_accumulator(output_dir):
    """The AdaGrad slot of the checkpoint; a checkpoint without one is refused, as TF's Saver refuses to
    restore a variable the checkpoint does not hold."""
    b = tf_bundle.load_bundle(os.path.join(output_dir, 'model.ckpt'), names={ADAGRAD_SLOT})
    if ADAGRAD_SLOT not in b:
        raise SystemExit(f"--optimizer adagrad: the checkpoint in {output_dir} has no {ADAGRAD_SLOT} slot "
                         "(it was not trained with AdaGrad); resume it with --optimizer sgd")
    return b[ADAGRAD_SLOT]


# --------------------------------------------------------------------------------------
# training driver
# --------------------------------------------------------------------------------------
def run_training(data, flags=None, seed=0, max_steps=None, log=print):
    flags = flags or FLAGS
    batch_count = data.triple_count // flags.batch_size
    log('Embedding dimension: ', flags.embedding_dim, 'Batch size: ', flags.batch_size,
        'Batch count: ', batch_count)
    if flags.embedding_dim % 2:
        raise ValueError("embedding_dim must be even (holE.py:164-165 splits the row in halves)")
    check_optimizer_flags(flags)
    # Warning: this will clobber existing summaries (holE.py:253-260)
    if not flags.resume_checkpoint and os.path.isdir(flags.output_dir):
        raise Exception("WARNING: " + flags.output_dir + " already exists!")
    try:
        os.makedirs(flags.output_dir)
    except OSError as e:
        if e.errno != errno.EEXIST:
            raise

    global_step = 0
    adagrad = getattr(flags, 'optimizer', 'sgd') == 'adagrad'
    A = None
    if flags.resume_checkpoint:
        E, global_step = load_checkpoint(flags.output_dir)
        if adagrad:
            A = load_accumulator(flags.output_dir)      # (--optimizer sgd ignores a saved accumulator)
        # TODO (reference, holE.py:315): the epoch counter restarts
    else:
        E = D.init_embeddings(data.entity_count, flags.embedding_dim, np.random.default_rng(seed))
    eng = make_engine(data.entity_count, data.relation_count, flags.embedding_dim, E, data.id_to_type)
    if adagrad:      # tf.train.AdagradOptimizer(lr, initial_accumulator_value) in place of holE.py:296's SGD
        eng.set_optimizer("adagrad", flags.adagrad_initial_accumulator)
        if A is not None:
            eng.set_accumulator(A)
    if getattr(flags, 'score_variant', 'complex') != 'complex':
        if flags.log_loss:
            raise SystemExit("--score_variant ccorr_tanh has no --log_loss branch")
        eng.set_score_mode(flags.score_variant)      # archived FFT / tanh score (holE-20170724/graph.pbtxt:6221-6521)
    B = flags.batch_size
    triples_dev = torch.from_numpy(data.triples).to(eng.device)
    valid = data.validation_triples
    decay_steps = flags.learning_decay_steps * batch_count
    valid_every = max(1, batch_count // 16)      # holE.py:351 (divides by zero if batch_count < 16)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(seed)
    vrng = np.random.default_rng(seed + 1)
    valid_dev = torch.from_numpy(np.ascontiguousarray(valid)).to(eng.device) if len(valid) else None
    log_path = os.path.join(flags.output_dir, 'summaries.tsv')
    events = tf_events.EventFileWriter(flags.output_dir)      # summary_writer (holE.py:317)
    pocket_loss = 2.
    steps_done = 0
    t_start = time.time()
    try:
        with open(log_path, 'a') as slog:
            for epoch in range(1, flags.num_epochs + 1):
                log('Initializing projector...')
                tf_bundle.write_projector_config(flags.output_dir)
                log('Training epoch {}...'.format(epoch))
                perm = torch.randperm(data.triple_count, device=eng.device, generator=gen)
                shuffled = triples_dev[perm]
                batch = 1                       # for batch in range(1, batch_count)  (holE.py:340)
                while batch < batch_count:
                    if batch % valid_every == 0 and len(valid) > 0:
                        # The reference scores ONE shuffled batch of the validation file and notes
                        # "TODO: this should run the entire validation set" (holE.py:350): the whole file
                        # is scored on the device here (--valid_sample restores the sampled batch).
                        if getattr(flags, "valid_sample", False):
                            vb = valid[vrng.integers(0, len(valid), size=B)]
                        else:
                            vb = valid_dev
                        if flags.log_loss:
                            vloss = evaluate_batch_logloss(eng, vb, seed, global_step, flags.l2_regularization,
                                                           flags.negative_ratio)
                            parts = (("loss", vloss),)
                        else:
                            vloss, vp, vn = evaluate_batch(eng, vb, seed, global_step, flags.margin)
                            parts = (("pos", vp), ("neg", vn), ("loss", vloss))
                        vlm = float(vloss.mean())
                        lr_now = float(inverse_time_decay(flags.learning_rate, global_step, decay_steps,
                                                          flags.learning_decay_rate))
                        row = {"step": global_step, "valid_loss_mean": vlm, "learning_rate": lr_now}
                        for nm, var in parts:
                            row.update({f"{nm}_{k}": v for k, v in summarize(var).items()})
                        slog.write("\t".join(f"{k}={v}" for k, v in row.items()) + "\n")
                        slog.flush()
                        # the merged summaries of holE.py:352-353: the validation twin's scalars and
                        # histograms, the training graph's on the next training batch (scored, not
                        # trained on), and the learning rate -- under the reference's name scopes
                        scal, hist = {"batch/learn/learning_rate": lr_now}, {}
                        scopes = {"pos": "validation/positive/eval", "neg": "validation/corrupt/eval",
                                  "loss": "validation"}
                        for nm, var in parts:
                            sc_, hi_ = tf_events.summarize_tags(scopes[nm], var.float().cpu().numpy())
                            scal.update(sc_); hist.update(hi_)
                        if not flags.log_loss:
                            tb = shuffled[(batch - 1) * B:batch * B]
                            tl, tp, tn = evaluate_batch(eng, tb, seed, global_step, flags.margin)
                            for scope, var in (("batch/eval/positive/eval", tp), ("batch/eval/corrupt/eval", tn),
                                               ("batch/eval", tl)):
                                sc_, hi_ = tf_events.summarize_tags(scope, var.float().cpu().numpy())
                                scal.update(sc_); hist.update(hi_)
                        events.add_summary(global_step, scal, hist)
                        log('\tStep {} Validation Loss: {}...'.format(global_step, vlm))
                        if vlm < pocket_loss:       # pocket checkpoint (holE.py:357-360)
                            pocket_loss = vlm
                            save_checkpoint(eng, flags.output_dir, global_step)
                            log('Epoch {}, (Model saved with loss {})'.format(epoch, vlm))
                    # run up to the next validation point without returning to the host per step
                    nxt = min(batch_count, (batch // valid_every + 1) * valid_every)
                    n = nxt - batch
                    if max_steps is not None:
                        n = min(n, max_steps - steps_done)
                    lrs = [inverse_time_decay(flags.learning_rate, global_step + k, decay_steps,
                                              flags.learning_decay_rate) for k in range(n)]
                    if flags.log_loss:
                        for k in range(n):       # one library call per step (k corrupt batches inside)
                            eng.train_step_logloss(shuffled[(batch - 1 + k) * B:(batch + k) * B], seed,
                                                   global_step + k, lrs[k], flags.l2_regularization,
                                                   flags.negative_ratio)
                    else:
                        eng.train_steps(shuffled[(batch - 1) * B:(batch - 1 + n) * B], B, seed, global_step,
                                        flags.margin, lrs)
                    batch += n
                    global_step += n
                    steps_done += n
                    if max_steps is not None and steps_done >= max_steps:
                        raise StopIteration
            log('Done training -- epoch limit reached')
    except StopIteration:
        log('Done training -- step limit reached')
    finally:
        log('Stopping training...')
        events.close()
    torch.cuda.synchronize()
    if not os.path.exists(os.path.join(flags.output_dir, 'model.ckpt.index')):
        save_checkpoint(eng, flags.output_dir, global_step)    # never validated: still leave a model
    log('Trained {} steps in {:.1f}s'.format(steps_done, time.time() - t_start))
    return eng, global_step


# --------------------------------------------------------------------------------------
# link prediction
# --------------------------------------------------------------------------------------
def score_mrr(raw_positions, filtered_positions, log=print):
    """holE.py:475-490 (hits are percentages of the filtered positions)."""
    raw_positions = np.array(raw_positions)
    raw_mrr = np.mean(1.0 / raw_positions)
    mean_raw_pos = np.mean(raw_positions)
    filtered_positions = np.array(filtered_positions)
    filtered_mrr = np.mean(1.0 / filtered_positions)
    mean_filtered_pos = np.mean(filtered_positions)
    hits1 = np.mean(filtered_positions <= 1).sum() * 100
    hits3 = np.mean(filtered_positions <= 3).sum() * 100
    hits10 = np.mean(filtered_positions <= 10).sum() * 100
    log('\n\n\nRaw MRR: {} (mean position: {})'.format(raw_mrr, mean_raw_pos))
    log('Filtered MRR: {} (mean position: {})'.format(filtered_mrr, mean_filtered_pos))
    log('Hits at 1: {}, 3: {}, 10: {}'.format(hits1, hits3, hits10))
    return {"raw_mrr": float(raw_mrr), "raw_mean_pos": float(mean_raw_pos),
            "filtered_mrr": float(filtered_mrr), "filtered_mean_pos": float(mean_filtered_pos),
            "hits1": float(hits1), "hits3": float(hits3), "hits10": float(hits10)}


def _logit(p):
    return float(np.log(p) - np.log1p(-p))


def eval_link_prediction(eng, queries, known, relation_count, entity_count, sides=("tail", "head"),
                         threshold=None, results_path=None, precision=HOLE_RANK_BF16X3):
    """All-entity generalisation of holE.py:427-472 on the tensor cores: every test triple is
    ranked against all entity rows on each requested side, ascending by (score, id).
    Train/valid-true candidates do not advance the filtered rank (holE.py:454-463); a test
    triple that is itself in-sample is skipped, as the reference's `continue` does.
    threshold: the reference's confidence gate `min sigma over the candidates < infer_threshold`
    (holE.py:438), evaluated as "some candidate scores below logit(threshold)"; None disables
    it (it cannot fire for the live model, SURVEY.md section 0).
    precision: split-bf16 by default (ranks match the fp32 reference except within ~3e-5 of a
    tie); HOLE_RANK_BF16 is 3x cheaper and what bench.py times.
    Side "relation" ranks each triple's relation against all relation rows [0, relation_count),
    filtered by the known relations of its (head, tail).
    Returns (raw_positions, filtered_positions) lists."""
    queries = np.unique(np.asarray(queries, dtype=np.int32).reshape(-1, 3), axis=0)   # test sets dedupe
    raw_positions, filtered_positions = [], []
    queries = queries[~D.rows_in(queries, known)]
    if len(queries) == 0:
        return raw_positions, filtered_positions
    for side_name in sides:
        side = _SIDES[side_name]
        lo, hi = _candidate_range(side_name, relation_count, entity_count)
        foff, fids = D.build_filter_csr(queries, known, side_name)
        raw, filt, ts = eng.rank(queries, side, lo, hi, foff, fids, precision=precision)
        ok = np.ones(len(queries), bool)
        if threshold is not None:
            gate = torch.full((len(queries),), _logit(threshold), dtype=torch.float32, device=eng.device)
            below, _, _ = eng.rank(queries, side, lo, hi, true_score=gate, compute_true=False, precision=precision)
            ok = below.cpu().numpy() > 0
        raw, filt, ts = raw.cpu().numpy(), filt.cpu().numpy(), ts.cpu().numpy()
        sig = 1.0 / (1.0 + np.exp(-ts.astype(np.float64)))
        raw_positions += (raw[ok] + 1).tolist()
        filtered_positions += (filt[ok] + 1).tolist()
        if results_path:
            with open(results_path, 'a') as output:     # holE.py:445,456
                for (h, t, r), s in zip(queries[ok].tolist(), sig[ok]):
                    output.write('{:.6f}\t{}\t{}\t{}\t{}\n'.format(s, h, t, r, False))
    return raw_positions, filtered_positions


def eval_link_prediction_typed(eng, heads, candidate, true_triples, test_triples, threshold=None):
    """The reference's own protocol (holE.py:564-573 + 427-469): for every head, the triples
    product([head], candidate.tail_candidates, candidate.relations) are ranked JOINTLY,
    ascending by (sigma, (head, tail, relation)); in-sample tails are skipped without
    advancing the filtered rank; every test-true (tail, relation) records its ranks.
    Implemented as tensor-core counts: one query row per (test item, relation of the group),
    thresholded at the test item's own score, ties resolved by the (tail, relation) order.
    Returns (raw_positions, filtered_positions)."""
    rels = sorted(int(r) for r in candidate.relations)
    tails = np.array(sorted(set(int(t) for t in candidate.tail_candidates)), dtype=np.int64)
    heads = [int(h) for h in heads]
    if not rels or len(tails) == 0 or not heads:
        return [], []
    R = int(max(rels)) + 1
    dev = eng.device
    tail_pos = {int(t): i for i, t in enumerate(tails)}
    # temporary table [relation rows 0..R-1 | candidate tails (ascending id) | heads]
    rows = torch.cat([torch.arange(R), torch.from_numpy(tails), torch.tensor(heads, dtype=torch.int64)]).to(dev)
    table = eng.table.index_select(0, rows)
    tmp = HoleEngine(int(table.shape[0]), eng.dim, dev.index or 0)
    tmp.table = table
    c0, c1 = R, R + len(tails)
    items = []            # (head slot, t*, r*) of every recorded test item
    for hi, h in enumerate(heads):
        for r in rels:
            for t in sorted(test_triples.get(h, {}).get(r, ())):
                if t in tail_pos and t not in true_triples.get(h, {}).get(r, ()):
                    items.append((hi, t, r))
    if not items:
        tmp.close()
        return [], []
    # 1. the test items' own scores through the same MMA path
    q_true = np.array([[c1 + hi, c0 + tail_pos[t], r] for hi, t, r in items], dtype=np.int32)
    _, _, s_true = tmp.rank(q_true, HOLE_SIDE_TAIL, c0, c1)
    # 2. one counting row per (item, relation r'): candidates (t, r') before (t*, r*)
    q_rows, thr, foff, fids = [], [], [0], []
    for k, (hi, t, r) in enumerate(items):
        h = heads[hi]
        for r2 in rels:
            # ties: (t, r2) < (t*, r*)  <=>  t < t*  or  (t == t* and r2 < r*)
            q_rows.append([c1 + hi, c0 + tail_pos[t] + (1 if r2 < r else 0), r2])
            thr.append(k)
            f = sorted(tail_pos[x] + c0 for x in true_triples.get(h, {}).get(r2, ()) if x in tail_pos)
            fids += f
            foff.append(len(fids))
    q_rows = np.array(q_rows, dtype=np.int32)
    thr_t = s_true[torch.as_tensor(thr, device=dev)].contiguous()
    raw, filt, _ = tmp.rank(q_rows, HOLE_SIDE_TAIL, c0, c1, np.array(foff, dtype=np.int64),
                            np.array(fids, dtype=np.int32), true_score=thr_t, compute_true=False)
    raw = raw.cpu().numpy().reshape(len(items), len(rels)).sum(1)
    filt = filt.cpu().numpy().reshape(len(items), len(rels)).sum(1)
    ok = np.ones(len(items), bool)
    if threshold is not None:      # min sigma over the head's whole candidate product < threshold
        gate = torch.full((len(q_rows),), _logit(threshold), dtype=torch.float32, device=dev)
        below, _, _ = tmp.rank(q_rows, HOLE_SIDE_TAIL, c0, c1, true_score=gate, compute_true=False)
        ok = below.cpu().numpy().reshape(len(items), len(rels)).sum(1) > 0
    tmp.table = None
    tmp.close()
    return (raw[ok] + 1).tolist(), (filt[ok] + 1).tolist()


def predict_top_k(eng, test, known, relation_count, entity_count, k, path, precision=HOLE_RANK_BF16X3,
                  value=None, sides=("tail", "head")):
    """The all-entity generalisation of the reference's `max_triples` cut of the pop loop (holE.py:427-472):
    the k best NEW tails of every distinct (head, relation) pair of the test file and the k best new heads of
    every distinct (tail, relation) pair, filtered against the train + valid triples; with "relation" in
    `sides`, also the k best new relations of every distinct (head, tail) pair.  Writes one line per
    prediction to `path`:  side  head  tail  relation  position  score  value  in_test
    (position 1-based, score = raw s, value = value(s) (sigma by default), in_test = the predicted triple is
    a test triple: the reference's MATCH vs GUESS).  Returns the number of lines written."""
    value = value or (lambda s: 1.0 / (1.0 + np.exp(-s)))
    test = np.asarray(test, dtype=np.int64).reshape(-1, 3)
    test_set = set(map(tuple, test.tolist()))
    key_cols = {"tail": (0, 2), "head": (1, 2), "relation": (0, 1)}       # the query's known columns
    n = 0
    with open(path, 'w') as out:
        for side_name in sides:
            side, cols = _SIDES[side_name], list(key_cols[side_name])
            pairs = np.unique(test[:, cols], axis=0)
            if len(pairs) == 0:
                continue
            queries = np.zeros((len(pairs), 3), dtype=np.int32)     # the predicted column is ignored
            queries[:, cols] = pairs
            foff, fids = D.build_filter_csr(queries, known, side_name)
            lo, hi = _candidate_range(side_name, relation_count, entity_count)
            ids, scores = eng.topk(queries, side, lo, hi, k, foff, fids, precision=precision)
            ids, scores = ids.cpu().numpy(), scores.cpu().numpy().astype(np.float64)
            vals = value(scores)
            for i, q in enumerate(queries.tolist()):
                for pos in range(k):
                    c = int(ids[i, pos])
                    if c < 0:
                        break
                    h, t, r = q
                    if side == HOLE_SIDE_TAIL:
                        t = c
                    elif side == HOLE_SIDE_HEAD:
                        h = c
                    else:
                        r = c
                    out.write('{}\t{}\t{}\t{}\t{}\t{:.9g}\t{:.6f}\t{}\n'.format(
                        side_name, h, t, r, pos + 1, scores[i, pos], vals[i, pos], (h, t, r) in test_set))
                    n += 1
    return n


def write_nearest_neighbors(eng, test, relation_count, entity_count, k, path, id_to_metadata,
                            precision=HOLE_RANK_BF16X3, chunk=65536):
    """The k most similar rows (cosine of the whole embedding, HoleEngine.neighbors) of every distinct entity of
    the test file among the entity rows [relation_count, entity_count), and of every distinct relation of the test
    file among the relation rows [0, relation_count).  Writes one line per neighbour to `path`:
    kind  row  neighbour  position  similarity  row_metadata  neighbour_metadata
    (kind = entity / relation, position 1-based, metadata = entity_metadata.tsv's "id name").  Queries go to the
    device `chunk` rows at a time, which bounds the workspace.  Returns the number of lines written."""
    test = np.asarray(test, dtype=np.int64).reshape(-1, 3)
    groups = (("entity", np.unique(test[:, :2]), relation_count, entity_count),
              ("relation", np.unique(test[:, 2]), 0, relation_count))
    n = 0
    with open(path, 'w') as out:
        for kind, rows, lo, hi in groups:
            for c0 in range(0, len(rows), chunk):
                part = rows[c0:c0 + chunk]
                ids, sims = eng.neighbors(part, k, lo, hi, precision=precision)
                ids, sims = ids.cpu().numpy(), sims.cpu().numpy()
                for i, row in enumerate(part.tolist()):
                    for pos in range(k):
                        c = int(ids[i, pos])
                        if c < 0:
                            break
                        out.write('{}\t{}\t{}\t{}\t{:.9g}\t{}\t{}\n'.format(
                            kind, row, c, pos + 1, sims[i, pos], id_to_metadata.get(row, ''),
                            id_to_metadata.get(c, '')))
                        n += 1
    return n


def infer_triples(flags=None, log=print):
    """holE.py:530-582 with the all-entity filtered protocol."""
    flags = flags or FLAGS
    data = init_inference_data(flags)
    E, _ = load_checkpoint(flags.output_dir)
    if E.shape != (data.entity_count, flags.embedding_dim):
        raise ValueError(f"checkpoint has embeddings {E.shape}, expected "
                         f"{(data.entity_count, flags.embedding_dim)}")
    eng = HoleEngine(data.entity_count, flags.embedding_dim).set_embeddings(E)
    if getattr(flags, 'score_variant', 'complex') != 'complex':
        if getattr(flags, "infer_gate", False):
            raise SystemExit("--infer_gate is defined on sigma(score): not available with --score_variant ccorr_tanh")
        eng.set_score_mode(flags.score_variant)      # ranks on the raw score s (tanh is monotone)
    threshold = flags.infer_threshold if getattr(flags, "infer_gate", False) else None
    precision = HOLE_RANK_BF16 if getattr(flags, "rank_precision", "bf16x3") == "bf16" else HOLE_RANK_BF16X3
    raw, filt = eval_link_prediction(eng, data.test, data.known, data.relation_count, data.entity_count,
                                     threshold=threshold, results_path='inference_results.tsv',
                                     precision=precision)
    relations = getattr(flags, 'relation_prediction', False)
    k = getattr(flags, 'predict_top_k', 0)
    if k:
        value = np.tanh if getattr(flags, 'score_variant', 'complex') != 'complex' else None
        path = os.path.join(flags.output_dir, 'predictions.tsv')
        sides = ("tail", "head", "relation") if relations else ("tail", "head")
        n = predict_top_k(eng, data.test, data.known, data.relation_count, data.entity_count, k, path,
                          precision=precision, value=value, sides=sides)
        log('Wrote {} predictions to {}'.format(n, path))
    nn_k = getattr(flags, 'nearest_neighbors', 0)
    if nn_k:
        path = os.path.join(flags.output_dir, 'neighbors.tsv')
        n = write_nearest_neighbors(eng, data.test, data.relation_count, data.entity_count, nn_k, path,
                                    data.id_to_metadata, precision=precision)
        log('Wrote {} nearest-neighbour lines to {}'.format(n, path))
    if not raw:
        log('No test triple passed the confidence gate; no ranks recorded.')
        result = None
    else:
        result = score_mrr(raw, filt, log)
    if relations:
        # (h, ?, t) for every test triple: no confidence gate, nothing written to inference_results.tsv
        rraw, rfilt = eval_link_prediction(eng, data.test, data.known, data.relation_count, data.entity_count,
                                           sides=("relation",), precision=precision)
        log('\nRelation prediction:')
        if rraw:
            result = dict(result or {}, relation=score_mrr(rraw, rfilt, log))
        else:
            log('No test triple to rank (every one is in-sample).')
    return result


# --------------------------------------------------------------------------------------
def build_parser():
    """Flags of holE.py:598-619, same names and defaults."""
    parser = argparse.ArgumentParser()
    parser.add_argument('--learning_rate', type=float, default=0.1, help='Initial learning rate.')
    parser.add_argument('--learning_decay_steps', type=float, default=32, help='Learning rate decay steps (in epochs).')
    parser.add_argument('--learning_decay_rate', type=float, default=0.5, help='Learning decay rate.')
    parser.add_argument('--batch_size', type=int, default=512, help='Batch size.')
    parser.add_argument('--num_epochs', type=int, default=1000, help='Number of training epochs.')
    parser.add_argument('--embedding_dim', type=int, default=128, help='Embedding dimension.')
    parser.add_argument('--log_loss', action='store_true', help='Use logistic loss with --negative_ratio corrupt batches (holE.py:194-196, 206-220).')
    parser.add_argument('--l2_regularization', type=float, default=0.1, help='L2 regularization weight (log loss only).')
    parser.add_argument('--negative_ratio', type=int, default=1, help='Number of negative labels sampled in log_loss.')
    parser.add_argument('--margin', type=float, default=0.2, help='Hinge loss margin.')
    parser.add_argument('--padded_size', type=int, default=1024,
                        help='Accepted for compatibility; the Philox sampler draws from the full type list.')
    parser.add_argument('--output_dir', type=str, required=True, help='Tensorboard Summary directory.')
    parser.add_argument('--data_dir', type=str, required=True, help='Input data directory.')
    parser.add_argument('--reader_threads', type=int, default=4, help='Accepted for compatibility; unused.')
    parser.add_argument('--resume_checkpoint', action='store_true', help='Resume training on the checkpoint model.')
    parser.add_argument('--save_embeddings', action='store_true', help='(out of scope here) debug dump.')
    parser.add_argument('--infer', action='store_true', help='Infer new triples from the latest checkpoint model.')
    parser.add_argument('--infer_threshold', type=float, default=0.05, help='Max loss to save triples')
    parser.add_argument('--min_mentions', type=int, default=50000,
                        help='The minimum number of mentions for an entity to be a viable candidate in inference.')
    parser.add_argument('--infer_gate', action='store_true',
                        help='Apply the reference\'s `min sigma < infer_threshold` gate (off: it never fires).')
    parser.add_argument('--rank_precision', choices=['bf16', 'bf16x3'], default='bf16x3',
                        help='Tensor-core operand precision of --infer (bf16x3 = split-bf16, ~fp32 ranks).')
    parser.add_argument('--predict_top_k', type=int, default=0,
                        help='With --infer: write the K best new tails of every (head, relation) and heads of every '
                             '(tail, relation) pair of the test file to <output_dir>/predictions.tsv (0 = off).')
    parser.add_argument('--relation_prediction', action='store_true',
                        help='With --infer: also rank every test triple\'s relation against all relations, (h, ?, t) '
                             'filtered by the train + valid relations of (h, t), and log its MRR / Hits; with '
                             '--predict_top_k, also write the K best new relations of every (head, tail) pair of the '
                             'test file to predictions.tsv.  Writes nothing to inference_results.tsv; --infer_gate '
                             'does not apply to it.')
    parser.add_argument('--nearest_neighbors', type=int, default=0,
                        help='With --infer: write the K entity rows most similar (cosine of the embeddings) to every '
                             'entity of the test file, and the K relation rows most similar to every relation of it, '
                             'to <output_dir>/neighbors.tsv (0 = off; K <= 128).')
    parser.add_argument('--valid_sample', action='store_true',
                        help='Validate on one sampled batch as holE.py does (default: the whole triples-valid.txt).')
    parser.add_argument('--score_variant', choices=['complex', 'ccorr_tanh'], default='complex',
                        help="Score function: 'complex' = holE.py:191-198 (default); 'ccorr_tanh' = the archived "
                             "variant of the holE-20170724 run (tanh of the r-weighted circular correlation, "
                             "trained there with --margin 1.0); no --log_loss branch.")
    parser.add_argument('--optimizer', choices=['sgd', 'adagrad'], default='sgd',
                        help="sgd: holE.py's GradientDescentOptimizer; adagrad: tf.train.AdagradOptimizer in its "
                             "place (checkpoints then hold its slot embeddings/Adagrad); hinge loss, complex score only.")
    parser.add_argument('--adagrad_initial_accumulator', type=float, default=0.1,
                        help='AdagradOptimizer initial_accumulator_value (> 0).')
    parser.add_argument('--seed', type=int, default=0)
    parser.add_argument('--max_steps', type=int, default=None, help='Stop after this many steps (testing).')
    return parser


def main(argv=None):
    global FLAGS
    FLAGS, _ = build_parser().parse_known_args(argv)
    if FLAGS.save_embeddings:
        raise SystemExit("--save_embeddings (holE.py:501-527, a py2-only debug dump) is out of scope")
    if FLAGS.infer:
        infer_triples(FLAGS)
    else:
        check_optimizer_flags(FLAGS)
        training_data = init_data(FLAGS)
        run_training(training_data, FLAGS, seed=FLAGS.seed, max_steps=FLAGS.max_steps)


if __name__ == '__main__':
    main(sys.argv[1:])
