"""Drop-in for Codes/train.py:  python train.py <dataset_dir>   (run from the directory that holds config.ini).

Same CLI, same config.ini keys, same stdout lines and checkpoint path pattern as the reference (train.py:30-381); the
epoch body (train.py:180-356) runs on the B200 through engine.GanEngine: phase A for every batch, NUM_SUB_EPOCHS passes of
D updates, NUM_SUB_EPOCHS passes of G updates over one shuffled batch order, validation, checkpoint.
<dataset_dir> may also be a golden .npz fixture (tests/golden/askubuntu_sample.npz) holding the loaders' outputs.
"""
from __future__ import print_function

import configparser
import importlib
import os
import sys

import numpy as np
import torch

if __package__ in (None, ""):
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    _pkg = importlib.import_module("long-tail-gan_b200")
    __package__ = _pkg.__name__

from . import data_processing as dp                      # noqa: E402
from .data_processing import load_item_one_hot_features as load_item_features  # noqa: E402,F401
from .discriminator import discriminator                 # noqa: E402
from .engine import GanEngine, TrainData, longtail_summary   # noqa: E402
from .generator import generator_VAECF as generator      # noqa: E402
from .generator import MultiVAE                          # noqa: E402
from .dist import env_rank_world as dist_env_rank_world  # noqa: E402
from .dist import shard_range as dist_shard_range        # noqa: E402


def _load_dataset(dataset):
    """Returns (tables for TrainData, validation CSR pair, n_items, generator tuple, niche item ids)."""
    if dataset.endswith(".npz"):
        g = np.load(dataset)
        n_items = int(g["n_items"])
        tabs = dp.tables_from_golden(g)
        vad = (g["vad_tr_indptr"], g["vad_tr_indices"].astype(np.int32), g["vad_te_indptr"], g["vad_te_indices"].astype(np.int32))
        vae = MultiVAE([200, 600, n_items], lam=0.0, random_seed=98765)
        out, loss, params = vae.build_graph()
        return tabs, vad, n_items, (vae, out, loss, params, [200, 600, n_items], 20000, 0.2), np.sort(g["niche_tags"].astype(np.int64))
    DATA_DIR = dataset + "/"
    show2id_path = DATA_DIR + "item2id.txt"
    niche_tags_path = DATA_DIR + "niche_items.txt"
    user_tag_matrix_path = DATA_DIR + "item_counts.csv"
    item_list_path = DATA_DIR + "item_list.txt"
    pro_dir = DATA_DIR
    n_items = sum(1 for _ in open(os.path.join(pro_dir, "unique_item_id.txt")))
    print("Loading Items...", end="")
    SHOW2ID, IDs_present, NICHE_TAGS, ALL_TAGS, OTHER_TAGS = dp.load_pop_niche_tags(show2id_path, item_list_path, niche_tags_path, n_items)
    print("Done.")
    print("Loading Item Features...", end="")
    ITEM_FEATURE_DICT, FEATURE_LEN, ITEM_FEATURE_ARR = dp.load_item_one_hot_features(item_list_path, SHOW2ID, n_items)
    print("Done.")
    print("Loading Training Interaction Matrix...", end="")
    train_data, uid_start_idx = dp.load_train_data(os.path.join(pro_dir, "train_GAN.csv"), n_items)
    print("Done.")
    print("Loading Validation Matrix...", end="")
    vad_data_tr, vad_data_te, uid_start_idx_vad = dp.load_tr_te_data(os.path.join(pro_dir, "validation_tr.csv"),
                                                                     os.path.join(pro_dir, "validation_te.csv"), n_items)
    print("Done.")
    print("Loading User's Popular and Niche Items...", end="")
    user_popular_data = dp.load_user_items(os.path.join(pro_dir, "train_GAN_popular.csv"))
    user_niche_data = dp.load_user_items(os.path.join(pro_dir, "train_GAN_niche.csv"))
    print("Done.")
    print("Loading item overlap coefficients....", end="")
    OVERLAP_COEFFS = dp.load_overlap_coeff(show2id_path, user_tag_matrix_path)
    print("Done.")
    N = train_data.shape[0]
    user_x_niche_vectors, user_x_popular_n_vectors = dp.load_vectors(user_popular_data, user_niche_data, OVERLAP_COEFFS, ITEM_FEATURE_DICT, N)
    print("Vectors Loaded")
    print("Loading Items to Sample....", end="")
    USER_TAGS_TO_SAMPLE = dp.load_items_to_sample(user_popular_data, user_niche_data, NICHE_TAGS, OVERLAP_COEFFS, N)
    print("Done")
    tabs = dp.build_train_tables(train_data, user_popular_data, user_niche_data, user_x_niche_vectors, user_x_popular_n_vectors,
                                 USER_TAGS_TO_SAMPLE, ITEM_FEATURE_DICT, n_items)
    vad_data_tr.sort_indices(); vad_data_te.sort_indices()
    vad = (vad_data_tr.indptr, vad_data_tr.indices, vad_data_te.indptr, vad_data_te.indices)
    return tabs, vad, n_items, generator(pro_dir), np.asarray(sorted(NICHE_TAGS), dtype=np.int64)


def _dist_setup():
    """One process per GPU under torch.distributed.run (RANK / WORLD_SIZE / LOCAL_RANK in the environment): user-sharded data
    parallelism (SURVEY 8e). Returns (rank, world). A plain `python train.py` run is (0, 1) and touches no process group."""
    rank, world, local = dist_env_rank_world()
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        if not dist.is_initialized():
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world


def train_GAN(h0_size, h1_size, h2_size, h3_size, NUM_EPOCH, NUM_SUB_EPOCHS, BATCH_SIZE, DISPLAY_ITER, LEARNING_RATE, to_restore,
              model_name, dataset, GANLAMBDA, seed=0, max_epochs=None, save=True, quiet=False, init=None, diag=False):
    """train.py:30-356. Extra keyword arguments (seed, max_epochs, save, quiet, init=(vae params, E, d_params), diag) are ours.
    Launched under torch.distributed.run with N ranks, every global batch of BATCH_SIZE users is split over the ranks (BATCH_SIZE / N
    users each; gradients exchanged inside the step, engine._g_step_dp); rank 0 prints the reference's lines and writes checkpoints.
    to_restore = 1 (parsed and ignored by the reference, train.py:374) resumes from the newest model_<epoch> under the output path."""
    rank, world = _dist_setup()
    log = (lambda *a, **k: None) if (quiet or rank != 0) else print
    dataset_name = dataset.split("/")[-1].strip()
    if dataset_name == "":
        dataset_name = dataset.split("/")[-2].strip()
    if dataset_name.endswith(".npz"):
        dataset_name = dataset_name[:-4]
    output_path = "chkpt/" + dataset_name + "_" + model_name + "_" + str(GANLAMBDA) + "/"
    if save and not os.path.exists(output_path):
        os.makedirs(output_path)

    tabs, vad, n_items, gen, niche_tags = _load_dataset(dataset)
    item_pop = np.bincount(np.asarray(tabs["indices"], dtype=np.int64), minlength=n_items)   # training interactions per item
    generator_network, generator_out, g_vae_loss, g_params, p_dims, total_anneal_steps, anneal_cap = gen
    if world > 1:
        if BATCH_SIZE % world != 0:
            raise ValueError("BATCH_SIZE (%d) must be a multiple of the number of ranks (%d)" % (BATCH_SIZE, world))
        B_local = BATCH_SIZE // world
        n_local_total = int(np.ceil(float(len(tabs["indptr"]) - 1) / B_local))
        first, count = dist_shard_range(n_local_total, rank, world)   # contiguous block of local batches per rank; the tail is dropped
        data = TrainData(batch_size=B_local, first_batch=first, max_batches=count, **tabs)
    else:
        data = TrainData(batch_size=BATCH_SIZE, **tabs)
    N = data.N
    log("Number of Users: ", N)
    batches_per_epoch = int(np.ceil(float(N) / BATCH_SIZE))
    log("Batches Per Epoch: ", batches_per_epoch)
    y_data, y_generated, d_params, x_generated_id, x_popular_n_id, x_popular_g_id, x_niche_id, item_feature_arr, keep_prob = \
        discriminator(n_items, n_items, h0_size, h1_size, h2_size, h3_size)
    disc = y_data.owner
    if world > 1:
        # the reference leaves the discriminator initialiser unseeded (discriminator.py:14-41): every rank would draw its own
        import torch.distributed as dist
        for t in (disc.arena, disc.E):
            dist.broadcast(t, 0)
        disc.load_state_dict(dict(arena=disc.arena.clone(), E=disc.E.clone()))
    if init is not None:
        generator_network.set_params(init[0]); generator_network.reset_optimizer()
        disc.set_params(init[1], init[2])
    start_epoch, restored_words = 0, None
    if to_restore and save:
        found = latest_checkpoint(output_path)
        if found is not None:
            start_epoch, ck = found[0] + 1, torch.load(found[1], map_location="cpu")
            generator_network.load_state_dict(ck["vae"]); disc.load_state_dict(ck["disc"])
            restored_words = ck["words"]
            log("Restored", found[1], "-> resuming at global-epoch", start_epoch)
    engine = GanEngine(generator_network, disc, max(data.max_B, 1), data.max_P, seed=seed, lr=LEARNING_RATE, lam=GANLAMBDA,
                       total_anneal_steps=total_anneal_steps, anneal_cap=anneal_cap, max_active=data.max_active, world_size=world, rank=rank,
                       B_global=(data.batch_size * world if world > 1 else None))
    if restored_words is not None:   # rng step, the shared Adam step t (F6) and the G-update count behind the KL anneal
        engine.words[: len(restored_words)].copy_(restored_words.to(engine.words.device))
    if world > 1:
        import torch.distributed as dist
        from .engine import build_dp_shard_tables
        engine.attach_dp_tables(build_dp_shard_tables(data, tabs["indptr"], tabs["indices"], world, rank, len(data.batches), engine.R))
    rng = np.random.RandomState(seed)
    for _ in range(start_epoch):      # the batch order of a resumed run continues the original shuffle sequence
        rng.shuffle(np.arange(len(data.batches)))
    history = []
    n_epochs = NUM_EPOCH if max_epochs is None else min(NUM_EPOCH, max_epochs)
    for i in range(start_epoch, n_epochs):
        # ---- phase A (train.py:192-278): sample generated pairs for every batch with the epoch-start generator ----
        for bi in range(len(data.batches)):
            engine.run_phase_a(data, bi)
        torch.cuda.synchronize()
        cnts = torch.stack([bt["cnt"][0] for bt in data.batches]).to(torch.int64)
        if world > 1:
            dist.all_reduce(cnts)     # a global batch is skipped only when no rank produced a pair for it (train.py:254-255)
        cnts = cnts.cpu().tolist()
        user_err_cnt = int((~np.asarray(tabs["eligible"], dtype=bool)).sum())
        log("global-epoch:", i, "Data Creation Finished", "user_err_cnt:", user_err_cnt)
        indices = np.asarray([bi for bi, c in enumerate(cnts) if c > 0])   # train.py:254-255: batches without pairs are skipped
        rng.shuffle(indices)                                               # train.py:284-285
        curr_d_loss = float("nan")
        for j_disc in range(NUM_SUB_EPOCHS):                               # train.py:287-303
            for bi in indices:
                engine.run_d_step(data, int(bi))
            if len(indices):
                curr_d_loss = engine.last_losses(data.batches[int(indices[-1])]["B"], reduce=True)["d_loss"]
            log("global-epoch:%s, discr-epoch:%s, d_loss:%.5f" % (i, j_disc, curr_d_loss))
        log("")
        j_gen = 0
        dg = dict(sp=[], ybar=[], vae=[], gan=[])
        for j_gen in range(NUM_SUB_EPOCHS):                                # train.py:307-329
            for bi in indices:
                engine.run_g_step(data, int(bi))
                if diag and j_gen == NUM_SUB_EPOCHS - 1:   # what the adversarial term acts on, over the last G sub-epoch (parity runs)
                    Ld = engine.last_losses(data.batches[int(bi)]["B"], reduce=True)
                    if Ld["cnt"] > 0:
                        dg["sp"].append(Ld["sum_p"] / Ld["cnt"]); dg["ybar"].append(Ld["sum_y"] / Ld["cnt"])
                        dg["vae"].append(Ld["vae_loss"]); dg["gan"].append(Ld["gan_loss"])
            if len(indices):
                L = engine.last_losses(data.batches[int(indices[-1])]["B"], reduce=True)
                log("global-epoch:%s, generator-epoch:%s, g_loss:%.5f (vae_loss: %.5f + gan_loss: %.5f, anneal: %.5f)"
                    % (i, j_gen, L["g_loss"], L["vae_loss"], L["gan_loss"], L["anneal"]))
        log("")
        m = engine.evaluate(vad[0], vad[1], vad[2], vad[3], k=100, recall_ks=(20, 50), niche=niche_tags, item_pop=item_pop)   # train.py:333-348
        ndcg_vad, recall_at_20, recall_at_50 = m["ndcg@100"], m["recall@20"], m["recall@50"]
        log("global-epoch:", i, "gen-epoch:", j_gen, "Vad: NDCG:", np.mean(ndcg_vad), "Recall@20:", np.mean(recall_at_20), "Recall@50:",
            np.mean(recall_at_50), "Num_users:", len(ndcg_vad), len(recall_at_20), len(recall_at_50))
        log("")
        rec = dict(epoch=i, ndcg=float(np.mean(ndcg_vad)), r20=float(np.mean(recall_at_20)), r50=float(np.mean(recall_at_50)),
                   d_loss=curr_d_loss)
        rec.update(longtail_summary(m))
        if diag:
            rec.update(sp_mean=float(np.mean(dg["sp"])) if dg["sp"] else None, ybar_mean=float(np.mean(dg["ybar"])) if dg["ybar"] else None,
                       vae_loss_mean=float(np.mean(dg["vae"])) if dg["vae"] else None, gan_loss_mean=float(np.mean(dg["gan"])) if dg["gan"] else None)
        history.append(rec)
        if save:
            engine.gather_master()   # data parallel: the fp32 masters and Adam moments are row-sharded; no-op on one GPU
            if rank == 0:
                save_checkpoint(os.path.join(output_path, "model_" + str(i)), generator_network, disc, engine, p_dims,
                                (h0_size, h1_size, h2_size, h3_size))
            log("Model saved at global-epoch", i)
    return dict(history=history, vae=generator_network, disc=disc, engine=engine, data=data)


def latest_checkpoint(output_path):
    """(epoch, path) of the newest model_<epoch> file under output_path, or None."""
    best = None
    if os.path.isdir(output_path):
        for name in os.listdir(output_path):
            if name.startswith("model_") and name[6:].isdigit():
                if best is None or int(name[6:]) > best[0]:
                    best = (int(name[6:]), os.path.join(output_path, name))
    return best


def save_checkpoint(path, vae, disc, engine, p_dims, hs):
    """train.py:354 (tf.train.Saver over all variables incl. optimizer slots) -> one torch file at the same path."""
    torch.save(dict(vae=vae.state_dict(), disc=disc.state_dict(), words=engine.words.cpu(), p_dims=list(p_dims), hs=list(hs)), path)


def read_config(path="config.ini"):
    cp = configparser.RawConfigParser()
    if not cp.read(path):
        raise IOError("config.ini not found in the current directory (train.py:359-361 reads it from the CWD)")
    g = lambda k: cp.get("Long-Tail-GAN", k)  # noqa: E731
    NUM_EPOCH = int(g("NUM_EPOCH"))
    return dict(h0_size=int(g("h0_size")), h1_size=int(g("h1_size")), h2_size=int(g("h2_size")), h3_size=int(g("h3_size")),
                NUM_EPOCH=NUM_EPOCH, NUM_SUB_EPOCHS=int(NUM_EPOCH / 8), BATCH_SIZE=int(g("BATCH_SIZE")), DISPLAY_ITER=int(g("DISPLAY_ITER")),
                LEARNING_RATE=float(g("LEARNING_RATE")), to_restore=int(g("to_restore")), model_name=g("model_name"),
                GANLAMBDA=float(g("GANLAMBDA")))


if __name__ == "__main__":
    cfg = read_config("config.ini")
    cfg["dataset"] = sys.argv[1]
    me = os.environ.get("LTG_MAX_EPOCHS")   # (ours) bound the run without editing NUM_EPOCH, which also sets NUM_SUB_EPOCHS
    train_GAN(max_epochs=int(me) if me else None, **cfg)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        torch.cuda.synchronize(); dist.barrier()
        sys.stdout.flush()
        os._exit(0)   # graphs hold captured exchange kernels; leave without tearing the process group down under them
