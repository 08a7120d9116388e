"""GNN-stage runners driven by exp_settings files: the device-side counterparts of
/root/reference/job_runner.py ``GCNTrain`` (:1247-1432), ``GCNTrainSPGNN`` (:1517-1920), ``GCNTest`` (:815-911)
and ``GCNTestSPGNN`` (:2017-2091), restricted to the GNN stage (graph → logits → per-class arg-max → branch accuracy;
the voxel painting / resampling / .mhd archiving around it needs CT volumes and is out of scope).

Data: stage-1 pickles ``<DB_PATH>/derived/conv_embedding/<uid>.pkl`` with keys ``fvs, adj, labels, fvs_out``
(job_runner.py:796-805, dataset.py:24-49), or synthetic scans when ``settings.SYNTHETIC_SCANS`` is set.
"""
from __future__ import annotations

import glob
import logging
import os
import pickle
import random
import time

import numpy as np
import torch

from . import ops, runner, synth
from ._lib import SpgnnError
from .settings import Settings, get_callable_by_name


class HeNorm:
    """initializer.py:12-30 for the GNN stage: reset every nn.Linear (conv/norm branches concern the CNN only)."""

    def __init__(self, **kwargs):
        self.mode = kwargs.get("mode", "fan_in")

    def initialize(self, module):
        for m in module.modules():
            if isinstance(m, torch.nn.Linear):
                m.reset_parameters()


class XavierUniform:
    def __init__(self, **kwargs):
        self.gain = kwargs.get("gain", torch.nn.init.calculate_gain("relu"))

    def initialize(self, module):
        for m in module.modules():
            if type(m) is torch.nn.Linear or isinstance(m, torch.nn.Linear):
                torch.nn.init.xavier_uniform_(m.weight, gain=self.gain)
                if m.bias is not None:
                    m.bias.data.fill_(0.01)


class ScanSource:
    """uid → dict(fvs, adj, labels, fvs_out): pickles of ConvEmbeddingExtractor or the synthetic generator."""

    def __init__(self, settings):
        self.synthetic = int(getattr(settings, "SYNTHETIC_SCANS", 0) or 0)
        self.ragged = bool(getattr(settings, "SYNTHETIC_RAGGED", True))
        self.seed = int(getattr(settings, "SYNTHETIC_SEED", 1234))
        self.fv_dim = settings.MODEL.get("fv_dim", 1024)
        if self.synthetic:
            self.uids = [f"synthetic_{i:06d}" for i in range(self.synthetic)]
        else:
            if not settings.DB_PATH:
                raise SpgnnError("settings.DB_PATH is not set (or set SYNTHETIC_SCANS=N for synthetic airway trees)")
            self.path = os.path.join(settings.DB_PATH, "derived", "conv_embedding")
            self.uids = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(self.path, "*.pkl")))
            if not self.uids:
                raise SpgnnError(f"no stage-1 pickles under {self.path}")

    def __call__(self, uid):
        if self.synthetic:
            s = synth.make_scan(int(uid.rsplit("_", 1)[1]), seed=self.seed, ragged=self.ragged, fv_dim=self.fv_dim)
            return dict(fvs=s.fvs, adj=s.adj, labels=s.labels, fvs_out=s.fvs_out, meta=dict(uid=uid))
        with open(os.path.join(self.path, uid + ".pkl"), "rb") as fp:
            d = pickle.load(fp)
        d.setdefault("meta", {})["uid"] = uid
        return d


def host_batch(scans, pin=True, packed=True):
    """collate (utils.py:76-84) + the float()/long() casts of job_runner.py:1872-1875, as ONE set of host buffers
    (``packed``: the lossless wire format of runner.HostBatch / csrc/wire.cu, about half the H2D bytes)."""
    n = [int(np.asarray(s["adj"]).shape[0]) for s in scans]
    adj = torch.from_numpy(np.concatenate([(np.asarray(s["adj"]) != 0).astype(np.uint8).reshape(-1) for s in scans]))
    fvs = torch.from_numpy(np.concatenate([np.asarray(s["fvs"], dtype=np.float32) for s in scans]))
    fvs_out = torch.from_numpy(np.concatenate([np.asarray(s["fvs_out"], dtype=np.float32) for s in scans]))
    labels = torch.from_numpy(np.concatenate([np.asarray(s["labels"]).astype(np.int64).reshape(-1) for s in scans]))
    return runner.HostBatch(n, adj, fvs, fvs_out, labels, pin=pin, packed=packed)


class _Runner:
    uses_pos_enc = False

    def __init__(self, settings=None, settings_module=None, output_path=None, cpk_path=None):
        self.settings = settings if settings is not None else settings_module
        if isinstance(self.settings, str):
            self.settings = Settings(self.settings)
        s = self.settings
        if self._always_reload:                       # BaselineTest.__init__ (job_runner.py:566-575): testing reloads
            s.RELOAD_CHECKPOINT = True
            if cpk_path is not None:
                s.RELOAD_CHECKPOINT_PATH = cpk_path
        self.output_path = output_path
        self.logger = logging.getLogger(type(self).__name__)
        if not torch.cuda.is_available():
            raise SpgnnError("spgnn_b200 runners need a CUDA device (no CPU fallback)")
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.exp_path = os.path.join(s.MODEL_ROOT_PATH, s.EXP_NAME)
        self.epoch_n, self.current_iteration = 0, 0
        self.source = ScanSource(s)
        model_kw = dict(s.MODEL)                      # the reference pops 'method' from the shared dict; copy instead
        self.model = get_callable_by_name(model_kw.pop("method"))(**model_kw).to(self.device)
        init_kw = dict(s.INITIALIZER)
        self.model.init(get_callable_by_name(init_kw.pop("method"))(**init_kw))
        cw = [s.CLASS_WEIGHTS[k] for k in sorted(s.CLASS_WEIGHTS.keys())][1:]          # job_runner.py:1867
        self.class_w = torch.tensor(cw, dtype=torch.float32, device=self.device)
        self.pos_enc_dim = getattr(s, "POS_ENC_DIM", 39) if self.uses_pos_enc else 0
        self.optimizer = None                         # training runners build it before reloading
        self.base_lr = None
        self.metric = {}                              # the reference's model_metrics_save_dict
        if type(self)._reload_in_base:
            self.reload_model_from_cache()

    _reload_in_base = True
    _always_reload = False

    # ---- checkpoints: the container of job_runner.py:336-350 (update_model_state / save_model)
    def save_model(self, **kwargs):
        os.makedirs(self.exp_path, exist_ok=True)
        if "metric" in kwargs and not isinstance(kwargs["metric"], dict):
            self.metric = {"metric": kwargs.pop("metric")}
        state = {"iteration": self.current_iteration, "epoch_n": self.epoch_n,
                 "model_dict": {k: v.detach().cpu().clone() for k, v in self.model.state_dict().items()},
                 "metric": dict(self.metric)}
        if self.optimizer is not None:
            state["optimizer_dict"] = self.optimizer.state_dict()
            state["scheduler_dict"] = {"gamma": getattr(self, "gamma", 1.0), "base_lrs": [self.base_lr],
                                       "last_epoch": self.epoch_n, "_last_lr": [self.optimizer.lr]}
        state.update(kwargs)
        path = os.path.join(self.exp_path, f"{self.current_iteration}.pth")
        torch.save(state, path)
        self.logger.info("saved model into %s.", path)
        return path

    def reload_model_from_cache(self):
        """job_runner.py:298-331 + load_pretrained_model (:87-123): only when RELOAD_CHECKPOINT is set; an explicit
        RELOAD_CHECKPOINT_PATH or the newest ``*.pth`` of the experiment; a missing checkpoint is logged and training
        starts from scratch; RELOAD_DICT_LIST names, position by position, which of (model, metric, optimizer,
        scheduler) are restored; model tensors whose shape differs are skipped; iteration resumes at saved + 1."""
        s = self.settings
        if not s.RELOAD_CHECKPOINT:
            return None
        path = s.RELOAD_CHECKPOINT_PATH
        if path is None:
            found = glob.glob(os.path.join(self.exp_path, "*.pth"))
            if not found:
                self.logger.error("%s has no checkpoint files with pth extensions.", self.exp_path)
                return None
            path = max(found, key=os.path.getctime)
        self.logger.info("reloading model from %s.", path)
        state = torch.load(path, map_location="cpu", weights_only=False)
        ignored = set(getattr(s, "RELOAD_CHECKPOINT_IGNORE", []) or [])
        slots = ("model", "metric", "optimizer", "scheduler")
        for slot, key in zip(slots, s.RELOAD_DICT_LIST):
            if key not in state:
                continue
            if slot == "model":
                own = self.model.state_dict()
                ok = {k: v for k, v in state[key].items()
                      if k in own and k not in ignored and own[k].shape == v.shape}
                self.model.load_state_dict(ok, strict=False)
                self.logger.info("loaded %d/%d tensors from %s", len(ok), len(own), path)
            elif slot == "metric":
                self.metric = dict(state[key]) if isinstance(state[key], dict) else {"metric": state[key]}
            elif slot == "optimizer" and self.optimizer is not None:
                self.optimizer.load_state_dict(state[key])
            elif slot == "scheduler" and self.optimizer is not None:
                sd = state[key]
                self.gamma = sd.get("gamma", getattr(self, "gamma", 1.0))
                if sd.get("base_lrs"):
                    self.base_lr = sd["base_lrs"][0]
                if sd.get("_last_lr"):
                    self.optimizer.set_lr(sd["_last_lr"][0])
        self.current_iteration = state["iteration"] + 1 if "iteration" in state else 0
        self.epoch_n = state.get("epoch_n", 0)
        return state

    def to_device(self, scans):
        return runner.batch_to_device(host_batch(scans), pos_enc_dim=self.pos_enc_dim, device=self.device)


class GCNTrain(_Runner):
    """GCNTrain.run / .train (job_runner.py:1350-1416): epochs × scan batches × GCN_STEPS full-batch steps."""
    _reload_in_base = False

    def __init__(self, settings=None, **kw):
        super().__init__(settings, **kw)
        s = self.settings
        self.model.set_gcn_only()
        opt_kw = dict(s.OPTIMIZER)
        method = opt_kw.pop("method", "torch.optim.SGD")
        name = method.rpartition(".")[2]
        if name in ("Adam", "AdamW"):
            unknown = set(opt_kw) - {"lr", "betas", "eps", "weight_decay", "amsgrad", "maximize"}
            if unknown:      # e.g. 'foreach', 'fused', 'capturable': refuse rather than train differently in silence
                raise SpgnnError(f"OPTIMIZER keys {sorted(unknown)} are not supported by the device optimiser")
            opt_kw.setdefault("lr", 1e-3)                  # torch's defaults; AdamW decays by 0.01 unless told
            if name == "AdamW":
                opt_kw.setdefault("weight_decay", 1e-2)
            self.optimizer = runner.FlatAdam(self.model.parameters(), decoupled=name == "AdamW", **opt_kw)
        else:
            if not method.endswith("SGD"):
                raise SpgnnError("only torch.optim.SGD, Adam and AdamW are implemented for the device optimiser")
            unknown = set(opt_kw) - {"lr", "momentum", "dampening", "weight_decay", "nesterov"}
            if unknown:      # e.g. 'groups', 'maximize', 'foreach': refuse rather than train differently in silence
                raise SpgnnError(f"OPTIMIZER keys {sorted(unknown)} are not supported by the device optimiser")
            opt_kw.setdefault("lr", 1e-4)
            self.optimizer = runner.FlatSGD(self.model.parameters(), **opt_kw)
        self.base_lr = self.optimizer.lr
        sched_kw = dict(s.SCHEDULER)
        if not sched_kw.pop("method", "torch.optim.lr_scheduler.ExponentialLR").endswith("ExponentialLR"):
            raise SpgnnError("only torch.optim.lr_scheduler.ExponentialLR is implemented")
        self.gamma = sched_kw.get("gamma", 1.0)
        self.reload_model_from_cache()                # after the optimiser exists, so its state can be restored
        uids = list(self.source.uids)
        n_val = max(1, len(uids) // 10) if len(uids) > 1 else 0
        self.val_uids, self.tr_uids = uids[:n_val], uids[n_val:] or uids
        self.history = []

    def train_batch(self, scans, steps=None):
        s = self.settings
        self.model.train()
        g = self.to_device(scans)
        losses = []
        n_steps = s.GCN_STEPS if steps is None else steps
        # many steps on one batch: capture the step once and replay it (launch-bound at the reference's batch size)
        graphed = None
        if getattr(s, "USE_CUDA_GRAPH", True) and n_steps >= 16 and self.optimizer.world == 1:
            graphed = runner.GraphedTrainStep(self.model, g, self.optimizer, self.class_w, s.SAMPLING_RATE, warmup=3)
            first = 3                                      # the warm-up steps are real training steps
        else:
            first = 0
        self.current_iteration += first
        for n in range(first, n_steps):
            loss = graphed() if graphed is not None else \
                runner.train_step(self.model, g, self.optimizer, self.class_w, s.SAMPLING_RATE)
            if n % s.LOG_STEPS == 0:
                losses.append(float(loss.item()))
                self.logger.info("Step %d-%d, LOSS: %.5f, LR:%.5f.", self.epoch_n, self.current_iteration, losses[-1],
                                 self.optimizer.lr)
            self.current_iteration += 1
        if graphed is not None:
            graphed.reset_salt()
        return losses

    @torch.no_grad()
    def validate(self, uids=None):
        self.model.eval()
        accs = []
        for uid in (self.val_uids if uids is None else uids):
            g = self.to_device([self.source(uid)])
            logits, decision = runner.infer(self.model, g)
            accs.append(branch_accuracy(decision, g.ndata["y"]))
        return float(np.mean(accs)) if accs else float("nan")

    def run(self, max_epochs=None, steps=None):
        s = self.settings
        n_epochs = s.NUM_EPOCHS if max_epochs is None else max_epochs
        while self.epoch_n < n_epochs:
            sample = random.sample(self.tr_uids, min(s.TRAIN_SAMPLE_SIZE, len(self.tr_uids)))
            for i in range(0, len(sample), s.TRAIN_BATCH_SIZE):
                self.history += self.train_batch([self.source(u) for u in sample[i:i + s.TRAIN_BATCH_SIZE]], steps)
            if self.epoch_n % s.SAVE_EPOCHS == 0 or self.epoch_n == n_epochs - 1:
                self.save_model(metric=self.validate())
            self.optimizer.set_lr(self.optimizer.lr * self.gamma)          # ExponentialLR, once per epoch
            self.epoch_n += 1
        return self.history


class GCNTrainSPGNN(GCNTrain):
    uses_pos_enc = True


class GCNTrainSAGE(GCNTrain):
    """GCNTrainSAGE.train (job_runner.py:1460-1514): every GCN step draws ``node_sample_rate`` of the batch's nodes,
    walks them in mini-batches of NODE_BATCH_SIZE seeds through ``MultiLayerNeighborSampler(node_ks)`` blocks and
    takes one optimiser step per mini-batch with the class-weighted CE over the seeds (no node mask here).  The
    blocks come from ``sampling.DeviceBlockSampler``: the same distribution as DGL's sampler, drawn from the
    counter hash of the dropout masks (seeded by ``ops.manual_seed``) instead of torch's generator."""

    def train_batch(self, scans, steps=None, max_minibatches=None):
        from . import sampling
        s = self.settings
        self.model.train()
        g = self.to_device(scans)
        sampler = sampling.DeviceBlockSampler(self.model.sage.node_ks)
        node_bs = int(getattr(s, "NODE_BATCH_SIZE", 64))
        losses = []
        for n in range(s.GCN_STEPS if steps is None else steps):
            nids = random.sample(range(g.num_nodes), int(g.num_nodes * self.model.sage.node_sample_rate))
            loader = sampling.DeviceNodeDataLoader(g, nids, sampler, device=self.device, batch_size=node_bs,
                                                   shuffle=True, drop_last=False)
            loss = None
            for k, (input_nodes, seeds, blocks) in enumerate(loader):
                if max_minibatches is not None and k >= max_minibatches:
                    break
                self.optimizer.zero_grad()
                out, _ = self.model.forward_batch(blocks, blocks[0].srcdata["fvs"])
                loss = ops.masked_cross_entropy(out, blocks[-1].dstdata["y"], self.class_w, rate=1.0)
                loss.backward()
                self.optimizer.step()
            if n % s.LOG_STEPS == 0 and loss is not None:
                losses.append(float(loss.item()))
                self.logger.info("Step %d-%d, LOSS: %.5f, LR:%.5f.", self.epoch_n, self.current_iteration, losses[-1],
                                 self.optimizer.lr)
            self.current_iteration += 1
        return losses


def branch_accuracy(decision, y):
    """Fraction of (tree, class 1..21) pairs whose arg-max node carries that label: the branch-level part of
    job_runner.py:158-165 + :878-893 (voxel-level relabelling is out of scope)."""
    n_cls = decision.shape[-1]
    want = torch.arange(1, n_cls + 1, device=y.device).expand_as(decision)
    return float((y[decision] == want).float().mean().item())


class GCNTest(_Runner):
    """GCNTest.run (job_runner.py:840-911): one graph at a time → logits → softmax → per-class arg-max node."""
    _always_reload = True

    def run(self, uids=None):
        self.model.eval()
        results, t_total = {}, 0.0
        with torch.no_grad():
            for uid in (self.source.uids if uids is None else uids):
                t0 = time.time()
                g = self.to_device([self.source(uid)])
                logits, decision = runner.infer(self.model, g)
                torch.cuda.synchronize()
                t_total += time.time() - t0
                results[uid] = dict(decision=decision[0].cpu().numpy(), acc=branch_accuracy(decision, g.ndata["y"]),
                                    node_labels=logits.argmax(1).cpu().numpy())
        if self.output_path:
            os.makedirs(self.output_path, exist_ok=True)
            with open(os.path.join(self.output_path, "gnn_predictions.pkl"), "wb") as fp:
                pickle.dump(results, fp)
        self.logger.info("tested %d scans, %.4f s/scan, mean branch acc %.4f", len(results),
                         t_total / max(len(results), 1), float(np.mean([r["acc"] for r in results.values()])))
        return results


class GCNTestSPGNN(GCNTest):
    uses_pos_enc = True
