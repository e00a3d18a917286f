"""Train driver: the B200 counterpart of the reference's `src/ann3depth.py`.

Same CLI (`dataset --model --steps --batchsize --ckptdir --id --ckptfreq --sumfreq --datadir --timeout`,
src/ann3depth.py:221-254) and the same loop shape: build the model op once (`setup_model`, :134-145), then
`while not should_stop: run(op)` (:126-127) under stop-at-step / stop-at-signal hooks, periodic
checkpoints with resume (MonitoredTrainingSession, :113-125) and loss summaries (:103-104).
The cluster flags (`--cluster-spec --job-name --task-index`) are accepted and ignored: the
parameter-server cluster (:39-67, :78-92) is replaced by one process per GPU
(`torchrun --nproc-per-node N -m ann3depth_b200.ann3depth ...`; RANK / WORLD_SIZE / LOCAL_RANK from
the environment) with an NCCL gradient allreduce.  Exit code = number of the signal that stopped the
run, 0 otherwise (:129).
"""
from __future__ import annotations

import argparse
import logging
import os
import signal
import sys
import time

import torch

from . import data, models
from .augment import from_flag as augment_from_flag
from .summary import EventWriter, SummaryHook, TraceHook
from .init import glorot_params

logger = logging.getLogger("ann3depth")


class StopAtSignalHook:
    """src/tfhelper.py:160-189: remember the signal, request a stop after the current step."""

    def __init__(self, signals=None):
        self.signal_received = 0
        for s in signals or [signal.SIGUSR1, signal.SIGUSR2, signal.SIGALRM, signal.SIGINT, signal.SIGTERM]:
            signal.signal(s, self._handler)

    def _handler(self, signum, frame):
        self.signal_received = signum


CKPT_FORMAT = 2


def save_checkpoint(op, ckptdir, comm=None, write=True):
    """Variables, optimizer slots and global_step, keyed by the reference's TF variable names in TF layouts (HWIO conv
    kernels, [in, out] dense kernels): the file survives changes of the packed arena layout, like a TF Saver checkpoint
    (MonitoredTrainingSession(checkpoint_dir=...), src/ann3depth.py:113-125).
    Data parallel: EVERY rank must call this at the same step (`comm` set, `write` only on the chief) -- the sharded
    optimizer keeps each rank's f32 master weights / Adam slots current only for the slice it owns, so they are
    all-gathered first (dp.DataParallel.gather_master)."""
    net = op.net
    if comm is not None:
        if getattr(comm, "stream", None) is not None:
            with torch.cuda.stream(comm.stream):
                comm.stream.wait_stream(torch.cuda.current_stream())
                comm.gather_master(net)
            torch.cuda.current_stream().wait_stream(comm.stream)
        else:
            comm.gather_master(net)
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    if not write:
        return
    os.makedirs(ckptdir, exist_ok=True)
    state = {"format": CKPT_FORMAT, "variables": net.arena.export_tf(), "global_step": net.global_step}
    if net.arena.m is not None:
        state["adam_m"] = net.arena.export_tf(net.arena.m)
        state["adam_v"] = net.arena.export_tf(net.arena.v)
    if hasattr(net, "adam_t"):
        state["adam_t"] = dict(net.adam_t)
    tmp = os.path.join(ckptdir, "model.ckpt.tmp")
    torch.save(state, tmp)
    os.replace(tmp, os.path.join(ckptdir, "model.ckpt"))


def restore_checkpoint(op, ckptdir):
    path = os.path.join(ckptdir, "model.ckpt")
    if not os.path.exists(path):
        return False
    state = torch.load(path, map_location="cpu")
    if state.get("format") != CKPT_FORMAT:
        raise ValueError(f"{path}: unknown checkpoint format {state.get('format')!r} (expected {CKPT_FORMAT})")
    net = op.net
    net.arena.load_tf(state["variables"])          # also refreshes the bf16 mirror
    if hasattr(net, "refresh_derived"):
        net.refresh_derived()               # filters derived from the arena (MSDN pool-fused fine/first)
    if "adam_m" in state and net.arena.m is not None:
        net.arena.load_tf(state["adam_m"], net.arena.m)
        net.arena.load_tf(state["adam_v"], net.arena.v)
    net.global_step = int(state["global_step"])
    if hasattr(net, "step_dev"):
        net.step_dev.fill_(net.global_step)
    if "adam_t" in state and hasattr(net, "adam_t"):
        net.adam_t.update(state["adam_t"])
    return True


class StopConsensus:
    """Data parallel: signals (SIGALRM / SIGTERM / SIGUSR1 ...) and the chief's checkpoint timer fire at different step
    boundaries on different ranks, but leaving the loop or entering the checkpoint's all-gathers on one rank alone would
    leave the others blocked in NCCL collectives forever.  Every `every` steps the ranks MAX-reduce (signal number,
    checkpoint due) over the gloo control plane and all act on the reduced values at the same step."""

    def __init__(self, world, every=8):
        self.world, self.every = world, max(int(every), 1)

    def decide(self, step, signal_received, ckpt_due):
        """-> (signal number agreed to stop on, or 0; take a checkpoint now)"""
        if self.world == 1:
            return signal_received, ckpt_due
        if step % self.every:
            return 0, False
        import torch.distributed as dist
        t = torch.tensor([int(signal_received), int(bool(ckpt_due))], dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return int(t[0]), bool(t[1])


def setup_model(args, comm=None):
    """src/ann3depth.py:134-145."""
    model = getattr(models, args.model)
    inp = data.inputs(args.datadir, args.dataset, args.batchsize, seed=100 + int(os.environ.get("RANK", 0)))
    aug = augment_from_flag(getattr(args, "augment", "none"))          # the training op only; evaluation sees raw inputs
    kw = {"loss": args.loss} if getattr(args, "loss", "silog") != "silog" else {}   # parse_args admits it for msdn only
    op = model(inp.images, inp.depths, comm=comm, augment=aug, **kw)
    op.net.load_params(glorot_params(seed=1, model=args.model))
    return op, inp


class Validator:
    """--evalfreq: depth metrics of the training net's current parameters on the test split.  The inference net shares
    the training net's parameter arena (no host round trip) and re-derives its pool-fused first-layer filter from it
    before each pass; every rank evaluates its shard of the file and the metrics are summed over the gloo group."""

    def __init__(self, args, op, rank, world):
        from . import evaluate
        self.args, self.op, self.rank, self.world = args, op, rank, world
        self.shard = (rank, world)
        inp = self._inputs()
        self.eval_op = getattr(models, args.model)(inp.images, inp.depths, train=False)
        inp.close()
        self.eval_op.net.arena = op.net.arena
        self.meters = evaluate.make_meters(self.eval_op, self.eval_op.net.ctx, getattr(args, "evalscale", "none"))
        self.last_step = None

    def _inputs(self):
        return data.inputs(self.args.datadir, self.args.dataset, self.args.batchsize, "test", epochs=1, shard=self.shard)

    def run(self, writer=None):
        from . import evaluate
        net = self.op.net
        if hasattr(net, "flush"):
            net.flush()                 # data parallel: dense rows other ranks own are current only after the publish
        self.eval_op.net.refresh_derived()
        inp = self._inputs()
        self.eval_op.net.images, self.eval_op.net.depths = inp.images, inp.depths
        for m in self.meters.values():
            m.reset()
        try:
            evaluate.evaluate_split(self.eval_op, inp, self.meters)
        finally:
            inp.close()
        step = self.op.global_step
        scalars = {}
        for name, m in self.meters.items():
            m.reduce()
            for k, v in m.result().items():
                if k in evaluate.METRICS and v is not None:
                    scalars[f"eval/{name}/{k}"] = v
        if writer is not None:
            writer.add_scalars(step, scalars)
            writer.flush()
        if self.rank == 0:
            logger.info(f"step {step} eval " + " ".join(f"{k}={v:.4g}" for k, v in scalars.items()))
        self.last_step = step
        return scalars


def main(argv=None):
    logging.basicConfig(level=logging.DEBUG, stream=sys.stdout,
                        format="%(asctime)s %(name)s %(levelname)s %(message)s")
    args = parse_args(argv)
    logger.debug(args)
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    chief = rank == 0
    logger.info(f"This is rank {rank} of {world} -- Chief? {chief}")

    comm = None
    if world > 1:
        import torch.distributed as dist
        from . import ops
        from .dp import DataParallel
        dist.init_process_group("gloo")      # control plane only; gradients go over liba3d's NCCL communicator
        ids = [ops.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = DataParallel(models.get_context(local_rank), rank, world, ids[0])

    run_id = args.model + ("" if not args.id else f"_{args.id}")
    ckptdir = str(os.path.join(args.ckptdir, run_id))
    logger.info(f"Checkpoint dir is {ckptdir}.")
    logger.info(f"Loading model {args.model}.")
    op, inp = setup_model(args, comm)
    size_train = op.net.arena.num_real_params() * 4 / 1024 / 1024          # tfhelper.estimate_size_of
    logger.debug(f"Trainable variables have about {size_train:.1f} MB")
    if restore_checkpoint(op, ckptdir):
        logger.info(f"Restored checkpoint at global step {op.global_step}.")

    validator = Validator(args, op, rank, world) if args.evalfreq > 0 else None
    stop_hook = StopAtSignalHook()
    # chief-only observability, as in the reference (src/ann3depth.py:98-111): loss summaries every --sumfreq
    # steps and a per-kernel trace of the first step after a (re)start and of every 5000th step, both in ckptdir
    writer = EventWriter(ckptdir) if chief else None
    summary_hook = SummaryHook(ckptdir, args.sumfreq, writer) if chief else None
    trace_hook = TraceHook(ckptdir, 5000, writer) if chief else None
    # the reference arms the alarm only for cluster jobs (`if args.job_name != 'local'`, src/ann3depth.py:107-109):
    # a plain single-process run is not stopped after --timeout seconds
    if args.timeout and (world > 1 or args.job_name != "local"):
        logger.info(f"Starting alarm: {args.timeout} s timeout.")
        signal.alarm(args.timeout)

    logger.info("Starting session.")
    consensus = StopConsensus(world)
    last_ckpt = last_log = time.time()
    last_log_step = op.global_step
    stop_signal = 0
    while op.global_step < args.steps:                                         # StopAtStepHook(last_step)
        ckpt_due = chief and time.time() - last_ckpt > args.ckptfreq
        stop_signal, take_ckpt = consensus.decide(op.global_step, stop_hook.signal_received, ckpt_due)
        if take_ckpt:
            save_checkpoint(op, ckptdir, comm, write=chief)
            last_ckpt = time.time()
        if stop_signal:                                                        # StopAtSignalHook.after_run
            break
        inp.next_batch()
        if trace_hook is not None:
            trace_hook.run(op)
        else:
            op.run()
        if summary_hook is not None:
            summary_hook.after_run(op, args.batchsize * world)
        if op.global_step % args.sumfreq == 0:
            torch.cuda.synchronize()
            now = time.time()
            losses = {k: float(v) for k, v in op.losses.items()}
            rate = (op.global_step - last_log_step) / max(now - last_log, 1e-9)
            logger.info(f"step {op.global_step} losses {losses} global_step/sec {rate:.2f} "
                        f"images/sec {rate * args.batchsize * world:.1f}")
            last_log, last_log_step = now, op.global_step
        if validator is not None and op.global_step % args.evalfreq == 0:
            validator.run(writer)
    if validator is not None and not stop_signal and validator.last_step != op.global_step:
        validator.run(writer)                                                  # the final step
    if world > 1 and not stop_signal:
        # the step limit is reached by all ranks together; a signal that arrived since the last consensus point still
        # decides the exit code (and every rank takes part in the final checkpoint either way)
        import torch.distributed as dist
        t = torch.tensor([int(stop_hook.signal_received)], dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stop_signal = int(t[0])
    elif not stop_signal:
        stop_signal = stop_hook.signal_received
    torch.cuda.synchronize()
    save_checkpoint(op, ckptdir, comm, write=chief)
    if chief:
        writer.close()
    if hasattr(inp, "close"):
        inp.close()
    logger.info("Session stopped.")
    return stop_signal


def parse_args(argv=None):
    """src/ann3depth.py:221-254 -- same flags and defaults."""
    parser = argparse.ArgumentParser()
    parser.add_argument("dataset", default="nyu", type=str, nargs="?", help="The dataset to use.")
    parser.add_argument("--model", "-m", default="msdn", type=str, help="Enter a model name.")
    parser.add_argument("--steps", "-s", default=1000000, type=int, help="Total steps")
    parser.add_argument("--batchsize", "-b", default=32, type=int, help="Batchsize")
    parser.add_argument("--ckptdir", "-p", default="checkpoints", help="Checkpoint directory")
    parser.add_argument("--id", default="", type=str, help="Checkpoint path suffix.")
    parser.add_argument("--ckptfreq", "-f", default=900, type=int, help="Create a checkpoint every N seconds.")
    parser.add_argument("--sumfreq", "-r", default=100, type=int, help="Create a summary every N steps.")
    parser.add_argument("--datadir", "-d", default="data", type=str, help="The data directory containing the datasets.")
    parser.add_argument("--timeout", "-k", default=4200, type=int, help="The time after which the process dies.")
    parser.add_argument("--evalfreq", default=0, type=int,
                        help="Evaluate the test split every N steps and at the last step (0: never; beyond the reference).")
    parser.add_argument("--evalscale", default="none", choices=["none", "median", "affine"],
                        help="Alignment of each prediction before the --evalfreq metrics, as evaluate --scale: median "
                             "scale, or least-squares scale and shift per image (affine).")
    parser.add_argument("--augment", default="none", choices=["none", "eigen"],
                        help="Training-time augmentation: 'eigen' = random scale, rotation, crop, flip and colour of "
                             "Eigen et al. 2014, section 3.3, on the GPU (beyond the reference).")
    parser.add_argument("--loss", default="silog", choices=["silog", "ssi"],
                        help="Training objective of MSDN: the reference's scale-invariant log loss (silog), or the "
                             "scale-and-shift-invariant loss of Ranftl et al. 2020 (ssi) for ground truth known only up "
                             "to a scale and a shift per image (beyond the reference).")
    parser.add_argument("--cluster-spec", default="", type=str, help="(ignored: no parameter servers)")
    parser.add_argument("--job-name", default="local", type=str, help="(ignored)")
    parser.add_argument("--task-index", default=0, type=int, help="(ignored)")
    args = parser.parse_args(argv)
    if args.loss != "silog" and args.model != "msdn":
        parser.error(f"--loss {args.loss} applies to --model msdn only ({args.model} trains on its own objective)")
    return args


if __name__ == "__main__":
    sys.exit(main())
