"""Training step on the gathered self-play buffer (§8f f1): the consumer of `all_gather_trajectories`.

Mirrors the reference's `train.train` (train.py:109-148) and the compile settings of `ResidualCNN.build_model`
(model.py:58-87): the same 9-block net, loss = softmax cross-entropy with logits on the policy head (loss.py:3-4,
soft targets pi) + mean squared error on the value head (loss weights 1, 1; config.py:41), L2 kernel regularisation
REG_CONST = 6e-3 on every conv / dense kernel (not on biases or BatchNorm), SGD with Nesterov momentum 0.9 at
LEARNING_RATE = 1e-4, batch 32, 5 epochs, shuffled, the last 5 % of the (pre-shuffle) data held out for validation
as Keras' `validation_split` does.  Per SURVEY §8f this step is plain PyTorch (autograd, cuDNN convs): it is a
consumer of the hot path, not part of it.  Weights enter and leave in the Keras `save_weights` tensor layout
('<layer>/<param>' arrays, kernels (kh,kw,cin,cout), dense (in,out)), i.e. exactly what model.ResidualCNN loads into the
CUDA inference kernels, so a trained net goes straight back into self-play."""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .config import (BATCH_SIZE, DEF_DATA_RETENTION_RATE, EPOCHS, EVAL_GAMES, LEARNING_RATE, LOSS_WEIGHTS, NUM_ACTIONS,
                     NUM_SELF_PLAY, PAST_ITER_COUNT, REG_CONST)

BN_EPS, BN_MOMENTUM = 1e-3, 0.99          # Keras BatchNormalization defaults (moving = 0.99 * moving + 0.01 * batch)


class _ConvBN(nn.Module):
    def __init__(self, cin, cout, k, padding):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, k, padding=padding, bias=True)
        self.bn = nn.BatchNorm2d(cout, eps=BN_EPS, momentum=1.0 - BN_MOMENTUM)

    def forward(self, x):
        return self.bn(self.conv(x))


class TrainableResidualCNN(nn.Module):
    """model.py:58-145 in PyTorch (NCHW inside, Flatten in Keras' (H, W, C) order so dense kernels map 1:1)."""

    def __init__(self):
        super().__init__()
        self.layers = nn.ModuleDict()
        self.layers["1"] = _ConvBN(7, 64, 3, 0)                                    # model.py:62
        for b in range(9):                                                          # model.py:66-76, 120-145
            self.layers[str(2 + 3 * b)] = _ConvBN(64, 32, 1, 0)
            self.layers[str(3 + 3 * b)] = _ConvBN(32, 32, 3, 1)
            self.layers[str(4 + 3 * b)] = _ConvBN(32, 64, 1, 0)
        self.layers["29"] = _ConvBN(64, 16, 1, 0)                                   # policy conv, model.py:108
        self.layers["30"] = _ConvBN(64, 1, 1, 0)                                    # value conv, model.py:91
        self.policy_head = nn.Linear(400, NUM_ACTIONS)
        self.dense_1 = nn.Linear(25, 32)
        self.value_head = nn.Linear(32, 1)

    def forward(self, board_x):
        """board_x (B,7,7,7) channels-last (uint8 or float) -> (logits (B,294), value (B,))"""
        x = board_x.to(self.policy_head.weight.dtype).permute(0, 3, 1, 2)
        L = self.layers
        x = F.relu(L["1"](x))
        for b in range(9):
            y = F.relu(L[str(2 + 3 * b)](x))
            y = F.relu(L[str(3 + 3 * b)](y))
            x = F.relu(L[str(4 + 3 * b)](y) + x)
        p = F.relu(L["29"](x)).permute(0, 2, 3, 1).reshape(x.shape[0], -1)
        v = F.relu(L["30"](x)).permute(0, 2, 3, 1).reshape(x.shape[0], -1)
        return self.policy_head(p), torch.tanh(self.value_head(F.relu(self.dense_1(v))))[:, 0]

    # -- Keras tensor layout <-> torch -----------------------------------------------------------------
    def load_keras_weights(self, w):
        """w: dict '<layer>/<param>' -> array (model.read_weight_file of a .h5 / .npz)"""
        with torch.no_grad():
            for i, m in self.layers.items():
                m.conv.weight.copy_(torch.from_numpy(np.ascontiguousarray(np.transpose(w["conv2d_%s/kernel" % i], (3, 2, 0, 1)))))
                m.conv.bias.copy_(torch.from_numpy(np.asarray(w["conv2d_%s/bias" % i])))
                m.bn.weight.copy_(torch.from_numpy(np.asarray(w["batch_normalization_%s/gamma" % i])))
                m.bn.bias.copy_(torch.from_numpy(np.asarray(w["batch_normalization_%s/beta" % i])))
                m.bn.running_mean.copy_(torch.from_numpy(np.asarray(w["batch_normalization_%s/moving_mean" % i])))
                m.bn.running_var.copy_(torch.from_numpy(np.asarray(w["batch_normalization_%s/moving_variance" % i])))
            for name in ("policy_head", "dense_1", "value_head"):
                lin = getattr(self, name)
                lin.weight.copy_(torch.from_numpy(np.ascontiguousarray(np.asarray(w[name + "/kernel"]).T)))
                lin.bias.copy_(torch.from_numpy(np.asarray(w[name + "/bias"])))
        return self

    def keras_weights(self):
        out = {}
        for i, m in self.layers.items():
            out["conv2d_%s/kernel" % i] = m.conv.weight.detach().permute(2, 3, 1, 0).contiguous().cpu().numpy().astype(np.float32)
            out["conv2d_%s/bias" % i] = m.conv.bias.detach().cpu().numpy().astype(np.float32)
            out["batch_normalization_%s/gamma" % i] = m.bn.weight.detach().cpu().numpy().astype(np.float32)
            out["batch_normalization_%s/beta" % i] = m.bn.bias.detach().cpu().numpy().astype(np.float32)
            out["batch_normalization_%s/moving_mean" % i] = m.bn.running_mean.detach().cpu().numpy().astype(np.float32)
            out["batch_normalization_%s/moving_variance" % i] = m.bn.running_var.detach().cpu().numpy().astype(np.float32)
        for name in ("policy_head", "dense_1", "value_head"):
            lin = getattr(self, name)
            out[name + "/kernel"] = lin.weight.detach().t().contiguous().cpu().numpy().astype(np.float32)
            out[name + "/bias"] = lin.bias.detach().cpu().numpy().astype(np.float32)
        return out

    def save_weights(self, path):
        """Model.save_weights (model.py:38-41): `.h5` = a Keras `save_weights` file (h5lite.write_weights: /<layer>/<layer>/<param>:0
        datasets, layer_names / weight_names attributes in model.layers order), `.npz` = the same tensors by name; both are what
        model.ResidualCNN.load_weights reads."""
        w = self.keras_weights()
        if str(path).endswith(".npz"):
            np.savez(path, **w)
            return path
        from . import h5lite
        return h5lite.write_weights(path, w)

    def kernel_l2(self):
        """sum of squares of every conv / dense kernel (Keras kernel_regularizer=l2(REG_CONST), model.py:60)"""
        s = 0.0
        for m in self.layers.values():
            s = s + (m.conv.weight ** 2).sum()
        for lin in (self.policy_head, self.dense_1, self.value_head):
            s = s + (lin.weight ** 2).sum()
        return s


def loss_terms(model, board_x, pi_y, v_y):
    """(total, policy CE, value MSE, L2) as Keras reports them for one batch"""
    logits, value = model(board_x)
    ce = -(pi_y * F.log_softmax(logits, dim=1)).sum(1).mean()                 # loss.py:3-4, soft targets
    mse = F.mse_loss(value, v_y.to(value.dtype))
    l2 = REG_CONST * model.kernel_l2()
    return LOSS_WEIGHTS["policy_head"] * ce + LOSS_WEIGHTS["value_head"] * mse + l2, ce, mse, l2


def make_optimizer(model, lr=LEARNING_RATE):
    # model.py:83: SGD(lr, momentum=0.9, nesterov=True).  Keras: v = m v - lr g; w += m v - lr g  ==  torch's Nesterov form
    return torch.optim.SGD(model.parameters(), lr=lr, momentum=0.9, nesterov=True)


def train(model, board_x, pi_y, v_y, data_retention=1.0, epochs=EPOCHS, batch_size=BATCH_SIZE, validation_split=0.05,
          seed=None, log=None):
    """train.train (train.py:109-148) on device tensors: sample `data_retention` of the examples without replacement
    (:130-133), hold out the LAST validation_split of the sampled set (Keras semantics), shuffle every epoch.
    Returns the per-epoch history [{loss, policy, value, val_loss, ...}]."""
    dev = next(model.parameters()).device
    g = torch.Generator(device="cpu")
    if seed is not None:
        g.manual_seed(int(seed))
    n_all = board_x.shape[0]
    keep = torch.randperm(n_all, generator=g)[:int(data_retention * n_all)].to(dev)
    bx, py, vy = board_x.to(dev)[keep], pi_y.to(dev)[keep].float(), v_y.to(dev)[keep].float()
    n = bx.shape[0]
    n_val = int(n * validation_split)
    n_tr = n - n_val
    opt = make_optimizer(model)
    history = []
    for ep in range(epochs):
        model.train()
        perm = torch.randperm(n_tr, generator=g).to(dev)
        tot = np.zeros(4)
        for s in range(0, n_tr, batch_size):
            idx = perm[s:s + batch_size]
            opt.zero_grad(set_to_none=True)
            terms = loss_terms(model, bx[idx], py[idx], vy[idx])
            terms[0].backward()
            opt.step()
            tot += np.array([float(t.detach()) for t in terms]) * idx.numel()
        rec = dict(zip(("loss", "policy", "value", "l2"), (tot / max(n_tr, 1)).tolist()))
        if n_val:
            model.eval()
            with torch.no_grad():
                vt = loss_terms(model, bx[n_tr:], py[n_tr:], vy[n_tr:])
            rec.update(val_loss=float(vt[0]), val_policy=float(vt[1]), val_value=float(vt[2]))
        history.append(rec)
        if log:
            log("epoch %d/%d %s" % (ep + 1, epochs, rec))
    model.eval()
    return history


# ---- the outer loop on one box (train.evolve, train.py:235-317), every stage on the batched kernels ----------------
SAVE_TRAIN_DATA_DIR, SAVE_TRAIN_DATA_PREF = "generated-training-data", "data-for-iter-"
SAVE_WEIGHTS_DIR, MODEL_PREFIX = "saved-weights", "version"


def get_weights_path_from_version(version, directory=SAVE_WEIGHTS_DIR):
    return "{}/{}{:0>4}-weights.h5".format(directory, MODEL_PREFIX, version)


def combine_prev_iters_train_data(board_x, pi_y, v_y, iteration_count, save_dir=SAVE_TRAIN_DATA_DIR,
                                  pref=SAVE_TRAIN_DATA_PREF):
    """This iteration's examples pooled with the PAST_ITER_COUNT previous data files (train.py:321-352)."""
    from .utils import combine_train_data
    return combine_train_data(board_x, pi_y, v_y, iteration_count - PAST_ITER_COUNT, iteration_count - 1, save_dir, pref)


def generate_self_play(model, num_games=NUM_SELF_PLAY, n_slots=None, seed=0, max_iters=512, opponent=None, resign_fp=None,
                       **selfplay_kw):
    """generate_self_play_in_parallel (train.py:58-105) without the process pool: exactly `num_games` games are started across
    the ranks (work shares like train.py:74-79: num_games // world each, the remainder on the last rank), every one is played
    to its end, discarded games are dropped (train.py:62-64), and the records come back as (board_x, pi_y, v_y) NumPy arrays
    in convert_to_train_data's format — all-gathered over the ranks when torch.distributed is initialised.
    `opponent`: a second loaded ResidualCNN in its own Engine = the reference's model2 (selfplay.py:11-29).
    `resign_fp` (with resign_threshold in selfplay_kw): stats["resign_suggested"] = this run's calibrated threshold for that
    false-positive rate (BatchedSelfPlay.suggest_resign_threshold, from this rank's samples)."""
    import torch.distributed as dist

    from .selfplay import BatchedSelfPlay, all_gather_trajectories
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist.is_available() and dist.is_initialized() else (0, 1)
    share = num_games // world + (num_games % world if rank == world - 1 else 0)
    if n_slots is None:
        # the accurate trunk works in rounds of (SMs x 3 contexts) four-position tiles: batches that fill its rounds exactly (3,552 or
        # 7,104 slots on a 148-SM B200) run 4-11 % more simulations per second than 4,096 (profiles/r02h_selfplay_slots.log)
        import torch
        full = 12 * torch.cuda.get_device_properties(model.eng.device).multi_processor_count
        n_slots = 4 * full if share >= 16 * full else 2 * full if share >= 2 * full else max(32, share)
    slots = int(n_slots)
    sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=slots, seed=seed, max_iters=max_iters, rank=rank, world=world,
                         ring=True, opponent=opponent, **selfplay_kw)
    stats = sp.play_games(share)
    if resign_fp is not None and sp.resign:
        stats["resign_suggested"] = sp.suggest_resign_threshold(resign_fp)
    traj = all_gather_trajectories(sp.collect())
    return (traj["board_x"].cpu().numpy(), traj["pi_y"].cpu().numpy(), traj["v_y"].cpu().numpy().astype(np.float32)), stats


def evolve(cur_model_path, other_opponent_for_selfplay=None, iteration_count=0, best_model=None, max_iterations=1,
           num_self_play=NUM_SELF_PLAY, eval_games=EVAL_GAMES, data_dir=SAVE_TRAIN_DATA_DIR, weights_dir=SAVE_WEIGHTS_DIR,
           seed=0, epochs=EPOCHS, log=print, symmetry="off", resign_fp=None, **selfplay_kw):
    """train.evolve (train.py:235-317) with a bound on the number of iterations: self-play with the best (else current)
    model — against `other_opponent_for_selfplay` when given (train.py:62, selfplay.py:11-29: the generator plays the even
    plies, the opponent the odd ones) -> augment -> save data-for-iter-N.h5 -> pool with previous iterations -> train
    (retention min(1/iters, 0.5)) -> save versionNNNN-weights.h5 -> arena against the best model, promote on more than
    int(0.55 * eval_games) wins.  `cur_model_path=None` starts from a freshly initialised net like the reference's version 0
    (train.py:41-46 `model_path is None`).  symmetry: the self-play nets' ResidualCNN.set_symmetry mode ("off", "random",
    "mean"; orientation seed = seed).  resign_fp: opt-in self-play resignation calibrated to that false-positive rate — the
    first iteration plays track-only (threshold -1, never resigns) to collect calibration samples, iteration k then plays with
    the threshold suggested from iteration k - 1's samples (resign_plies / resign_probe / resign_samples in selfplay_kw).
    Returns (cur_model_path, best_model, iteration_count) after the last iteration."""
    import os

    from . import utils
    from .arena import evaluate
    from .engine import Engine
    from .model import ResidualCNN, read_weight_file
    engine = Engine()
    opp_engine = Engine() if other_opponent_for_selfplay is not None else None
    if cur_model_path is None:                                     # un-trained model: materialise it so that every stage can load it
        os.makedirs(weights_dir, exist_ok=True)
        torch.manual_seed(int(seed))
        cur_model_path = TrainableResidualCNN().save_weights(os.path.join(weights_dir, "%s-untrained-weights.h5" % MODEL_PREFIX))
    if resign_fp is not None:
        selfplay_kw = dict(selfplay_kw, resign_threshold=-1.0)
    for _ in range(int(max_iterations)):
        if resign_fp is not None:
            log("iteration %d: self-play resign threshold %.6f (false-positive target %g)"
                % (iteration_count, selfplay_kw["resign_threshold"], resign_fp))
        generator_path = best_model if best_model is not None else cur_model_path
        net = ResidualCNN(engine=engine).load_weights(generator_path).set_symmetry(symmetry, seed)
        opponent = (ResidualCNN(engine=opp_engine).load_weights(other_opponent_for_selfplay).set_symmetry(symmetry, seed)
                    if other_opponent_for_selfplay is not None else None)
        (board_x, pi_y, v_y), stats = generate_self_play(net, num_self_play, seed=seed + iteration_count, opponent=opponent,
                                                         resign_fp=resign_fp, **selfplay_kw)
        if resign_fp is not None:
            selfplay_kw["resign_threshold"] = stats["resign_suggested"]
        log("iteration %d: self-play with %s%s: %s" % (iteration_count, generator_path,
                                                       " vs %s" % other_opponent_for_selfplay if opponent is not None else "", stats))
        if len(board_x):
            board_x, pi_y, v_y = utils.augment_train_data(board_x, pi_y, v_y)
            utils.save_train_data(board_x, pi_y, v_y, version=iteration_count, directory=data_dir, prefix=SAVE_TRAIN_DATA_PREF)
        board_x, pi_y, v_y, iters_used = combine_prev_iters_train_data(board_x, pi_y, v_y, iteration_count, data_dir)
        if iters_used == 0:
            log("No training data for iteration %d! Re-iterating..." % iteration_count)
            continue
        retention = min(1.0 / iters_used, DEF_DATA_RETENTION_RATE)
        learner = TrainableResidualCNN().load_keras_weights(read_weight_file(cur_model_path)).to(net.eng.device)
        history = train(learner, torch.from_numpy(board_x), torch.from_numpy(pi_y), torch.from_numpy(v_y), retention,
                        epochs=epochs, seed=seed + iteration_count, log=log)
        os.makedirs(weights_dir, exist_ok=True)
        cur_model_path = learner.save_weights(get_weights_path_from_version(iteration_count, weights_dir))
        log("iteration %d: trained on %d examples (retention %.2f), final %s -> %s"
            % (iteration_count, len(board_x), retention, history[-1] if history else None, cur_model_path))
        if best_model is not None:
            cur_wins, best_wins, draws = evaluate(best_model, cur_model_path, eval_games, seed=seed + iteration_count)
            if cur_wins > int(0.55 * eval_games):
                best_model = cur_model_path
                log("Now using {} as the best model".format(best_model))
            else:
                log("Output model of this iteration is not better; retaining {} as the best model".format(best_model))
        iteration_count += 1
    return cur_model_path, best_model, iteration_count
