"""Training / sampling loop: mirror of txt2vid/gan/trainer.py (train, test, add_params_to_parser,
save_frames, save_sentences) with the same parameters and iteration order, driving the B200-native
modules.  Differences that do not change results:
  * the real-video pyramid (trainer.py:131-165) runs as bit-exact index kernels on the GPU;
  * `real_pred` for the G step is computed without recording a D-parameter graph: the reference
    back-propagates the G loss into D's (already stepped, about to be zeroed) gradients
    (trainer.py:247,262) -- wasted work with no observable effect on lossG, G's gradients or D.  With
    --end2end and a conditional discriminator the graph through the caption embedding IS kept (see _g_phase);
  * an optional `dist` argument (txt2vid_b200.parallel) all-reduces gradients before each optimiser step.
"""
import sys

import torch

from . import kernels as K
from .blocks import Subsample
from .util import RollingAvg, Stopwatch, ensure_exists, status


def add_params_to_parser(parser):
    """Same flags, defaults and (inverted) store_false quirks as gan/trainer.py:15-42."""
    a = parser.add_argument
    a('--data_is_imgs', action='store_true', default=False, help='is the data images? If not, assume it is videos')
    a('--img_model', action='store_true', default=False, help='does the GAN only do images?')
    a('--log_period', type=int, default=20, help='period to log')
    a('--loss_window_size', type=int, default=20, help='window size for logging')
    a('--no_mean_discrim_loss', action='store_false', default=True,
      help='divides each discrim step loss by discrim_steps')
    a('--no_mean_gen_loss', action='store_false', default=True, help='divides each gen step loss by gen_steps')
    a('--sample_batch_size', type=int, default=None, help='batch size to gen samples')
    a('--discrim_steps', type=int, default=1, help='Number of discriminator steps to use per iteration')
    a('--gen_steps', type=int, default=1, help='Number of generator steps to use per iteration')
    a('--gp_lambda', type=float, default=-1, help='GP lambda hyper-param (negative to disable GP)')
    a('--save_initial', action='store_true', default=False, help='save initial model')
    a('--save_initial_examples', action='store_true', default=False, help='save initial sample')
    a('--save_model_period', type=int, default=100, help='number of iters until model is saved')
    a('--save_example_period', type=int, default=100, help='number of iters until model is saved')
    a('--use_writer', action='store_true', default=False, help='write losses to SummaryWriter (tensorboardX)')
    a('--out', type=str, default='out', help='dir output path')
    a('--out_samples', type=str, default='out_samples', help='dir output path')
    a('--subsample_input', action='store_true', default=False, help='should subsampling be applied to the input?')
    return parser


def multiscale_data(x, cond, frame_sizes, subsample_input, subsampler=None):
    """Real-video pyramid (gan/trainer.py:131-165): level i < last = nearest resize of the CURRENT
    (already subsampled) clip to frame_sizes[i]; last = the clip; after every level (the last one
    included: its draw is discarded) x <- x[::2, :, bt::2], cond <- cond[::2] when subsample_input."""
    n = len(frame_sizes)
    if n == 1:
        return [x], (None if cond is None else [cond])
    subsampler = subsampler or Subsample()
    xs, conds = [], []
    for i in range(n):
        if i != n - 1:
            fs = frame_sizes[i]
            xs.append(K.pyramid_level(x.contiguous(), fs, fs))      # index kernel; no CPU path (T2VError off-GPU)
        else:
            xs.append(x)
        if cond is not None:
            conds.append(cond)
        if subsample_input:
            x, _ = subsampler(x)
            if cond is not None:
                cond = cond[::2]
    return xs, (conds if conds else None)


def save_frames(frames, path=None, channel_first=True, is_images=False):
    import torchvision.utils as vutils
    if channel_first:
        if is_images:
            frames = frames.unsqueeze(2)
        frames = frames.permute(0, 2, 1, 3, 4).contiguous()
    n = frames.size(1)
    vutils.save_image(frames.view(-1, frames.size(2), frames.size(3), frames.size(4)), path, normalize=True, nrow=n)


def save_sentences(captions, path=None, vocab=None):
    with open(path, 'w') as f:
        for cap in captions:
            f.write(vocab.to_words(cap))
            f.write('\n')


def test(gan=None, num_samples=1, dataset=None, device=None, params=None, channel_first=True, vocab=None):
    """Eval-mode sampling (gan/trainer.py:44-90): one batch per sample index, full-resolution output."""
    ensure_exists(params.out_samples)
    gan.gen.eval()
    for i in range(num_samples):
        for j, data in enumerate(dataset):
            x = data[0]
            B = x.size(0)
            if channel_first:
                x = x.permute(0, 2, 1, 3, 4)
            y = [a.to(device) if isinstance(a, torch.Tensor) else a for a in data[1:]]
            cond = None
            if gan.cond_encoder is not None and len(y) >= 2:
                _, _, cond = gan.cond_encoder.encode(y[0], y[1])
            z = torch.randn(B, gan.gen.latent_size, device=device)
            with torch.no_grad():
                fake = as_levels(gan(z, cond=cond))
            save_frames(x, path='%s/real_%d.png' % (params.out_samples, i), channel_first=channel_first,
                        is_images=params.img_model)
            if cond is not None:
                save_sentences(y[0], path='%s/sentences_%d_%d.txt' % (params.out_samples, i, j), vocab=vocab)
            for f in fake:
                h, w = (f.size(2), f.size(3)) if params.img_model else (f.size(3), f.size(4))
                path = '%s/%dx%d_%d_%d.jpg' % (params.out_samples, h, w, i, j)
                status("saving to %s" % path)
                save_frames(f, path=path, channel_first=channel_first, is_images=params.img_model)
            break


def as_levels(fake):
    """generator output as a list of pyramid levels: a single-scale generator (TGAN) returns one tensor"""
    return [fake] if torch.is_tensor(fake) else fake


def encode_captions(gan, y, end2end):
    cond = None
    if gan.cond_encoder is not None and len(y) >= 2:
        _, _, cond = gan.cond_encoder.encode(y[0], y[1])
        if not end2end:
            cond = cond.detach()
    return cond


def _d_phase(gan, x, cond, device, params, losses, z, channel_first, end2end, j=0, st=None):
    """pyramid + G forward (first D step only) + D loss backward (trainer.py:199-240)."""
    if st is None:
        B = x.size(0)
        if not params.data_is_imgs and channel_first:
            x = x.permute(0, 2, 1, 3, 4)
        if params.img_model and not params.data_is_imgs:
            x = x.squeeze(2)
        xs, conds = multiscale_data(x, cond, params.frame_sizes, params.subsample_input)
        if z is None:
            z = torch.randn(B, gan.gen.latent_size, device=device)
        fake = as_levels(gan(z, cond=conds[0] if conds is not None else None))
        st = {"xs": xs, "conds": conds, "z": z, "fake": fake}
    loss = gan.discrim_step(real=st["xs"], fake=[f.detach() for f in st["fake"]], cond=st["conds"],
                            loss=losses.discrim_loss, gp_lambda=params.gp_lambda)
    if not params.no_mean_discrim_loss:
        loss = loss / params.discrim_steps
    from . import ops
    with ops.skip_leaf_input_grads():       # d(loss)/d(x_hat) of the penalty's interpolated clips is never read
        loss.backward(retain_graph=j != params.discrim_steps - 1 or end2end)
    st["lossD"] = loss.detach()
    return st


def _g_phase(gan, st, params, losses, j=0, end2end=False):
    """real_pred + G loss backward (trainer.py:247-262).  D's parameter gradients are never needed here (the reference
    computes and discards them), so D is frozen for the whole phase.  real_pred itself is computed without a graph --
    EXCEPT with end2end and a conditional discriminator: there the conditional real prediction depends on the
    (undetached) caption embedding (cond_gan.py:108-112), and relativistic losses send a generator-step gradient
    through it into the caption encoder, whose parameters are in optG (train/gan.py:84-85)."""
    xs, conds = st["xs"], st["conds"]
    dparams = [p_ for d in gan.discrims for p_ in d.parameters()]
    for p_ in dparams:
        p_.requires_grad_(False)
    try:
        if j == 0:
            # trainer.py:247 -- draws the caption permutation again (numpy RNG) although only real_pred is used
            need_graph = end2end and conds is not None and any(c.requires_grad for c in conds)
            with torch.enable_grad() if need_graph else torch.no_grad():
                _, _, st["real_pred"] = gan.all_discrim_forward(real=xs, cond=conds, fake=None, loss=None)
        else:
            st["fake"] = as_levels(gan(st["z"], cond=conds[0] if conds is not None else None))
        loss = gan.gen_step(fake=st["fake"], real_pred=st["real_pred"], cond=conds, loss=losses.gen_loss)
        if not params.no_mean_gen_loss:
            loss = loss / params.gen_steps
        loss.backward(retain_graph=j != params.gen_steps - 1)
    finally:
        for p_ in dparams:
            p_.requires_grad_(True)
    st["lossG"] = loss.detach()
    return st


def train_iteration(gan, x, y, device, optD, optG, params, losses, channel_first=True, end2end=True, dist=None,
                    z=None):
    """Body of one `train()` iteration (gan/trainer.py:199-267).  x: (B,T,C,H,W) loader order.
    Returns (lossD, lossG, fake, real_levels, conds) with the losses as 0-d device tensors (no host sync)."""
    from . import hostrng
    if torch.is_tensor(x) and x.dtype == torch.uint8:       # frames as stored: ToTensor + Normalize(0.5, 0.5) on the device
        x = K.u8_normalize(x.contiguous())
    hostrng.CURRENT.begin_iteration()
    cond = encode_captions(gan, y, end2end)
    st, total_d, total_g = None, 0, 0
    for j in range(params.discrim_steps):
        st = _d_phase(gan, x, cond, device, params, losses, z, channel_first, end2end, j, st)
        if dist is not None:
            dist.reduce_grads(optD)
        optD.step()
        total_d = total_d + st["lossD"]
    for j in range(params.gen_steps):
        st = _g_phase(gan, st, params, losses, j, end2end)
        if dist is not None:
            dist.reduce_grads(optG)
        optG.step()
        total_g = total_g + st["lossG"]
    return total_d, total_g, st["fake"], st["xs"], st["conds"]


def hostrng_ring():
    from . import hostrng
    return hostrng.StaticDraws.RING


class GraphedTrainStep(object):
    """The training iteration as ONE replayed CUDA graph (no tracing compiler: the eager iteration above is
    captured as is): pyramid, G fwd, D fwd/bwd incl. gradient penalty, all-reduce of the D grads, Adam D,
    real_pred, G-step fwd/bwd, all-reduce of the G grads, Adam G.  `graphs` is the 1-tuple of that graph.
    Everything the host decides per iteration reaches the kernels through device buffers refreshed before each replay: the batch, the caption
    embedding (the Bi-LSTM runs eagerly -- variable lengths), the host-RNG draws (hostrng.StaticDraws, same
    generators and order as the reference), Adam's bias corrections.  z comes from the CUDA generator inside
    the graph.  With discrim_steps > 1 (the WGAN-GP recipe: 5 critic steps per generator step) the graph holds every
    critic step, each with its all-reduce and Adam step; each of those Adam steps reads its own row of bias corrections.
    Needs gen_steps = 1, a fixed batch shape and an even frame count per level."""

    def __init__(self, gan, optD, optG, params, losses, device, channel_first=True, end2end=False, dist=None,
                 warmup=2):
        assert params.gen_steps == 1 and not end2end
        self.gan, self.optD, self.optG, self.params, self.losses = gan, optD, optG, params, losses
        self.device, self.channel_first, self.dist = device, channel_first, dist
        self.warmup, self.calls, self.graphs = warmup, 0, None
        self.static_x = self.static_cond = self.draws = None
        self.side = torch.cuda.Stream(device=device)
        # per-replay host values (RNG draws, Adam bias corrections) go through a ring of pinned staging slots: the
        # H2D copies are asynchronous, so a slot is rewritten only after the copies issued from it have executed
        self.ring = hostrng_ring()
        self.stage_evt = [None] * self.ring
        self.replays = 0

    # ---- per-replay host work
    def _stage_adam(self, opt, step, slot):
        """row j of opt.dyn <- the bias corrections of Adam step `step + j` (one row per captured step)"""
        b1, b2 = opt.param_groups[0]["betas"]
        lr = opt.param_groups[0]["lr"]
        h = opt._dyn_host[slot]
        h.copy_(torch.tensor([[lr / (1.0 - b1 ** t), 1.0 / (1.0 - b2 ** t) ** 0.5]
                              for t in range(step, step + h.shape[0])], dtype=torch.float32))
        K.multi_copy([h], [opt.dyn])            # UVA read of the pinned slot (see hostrng.StaticDraws.refresh)

    def _capture(self, x, cond):
        """Capture only: nothing executes here.  The caller replays right afterwards."""
        dev = self.device
        self.static_x = x.clone()
        self.static_cond = None if cond is None else cond.clone()
        for opt, n in ((self.optD, self.params.discrim_steps), (self.optG, 1)):
            opt.dyn = torch.zeros(n, 2, device=dev, dtype=torch.float32)
            opt._dyn_host = [torch.zeros(n, 2, dtype=torch.float32).pin_memory() for _ in range(self.ring)]
            opt._step_count = max([st_["step"] for st_ in opt.state.values()] or [0])
            opt.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        pool = torch.cuda.graph_pool_handle()
        self.draws.begin_iteration()
        # ONE graph for the whole iteration; the two NCCL all-reduces are captured with it (thread-local capture
        # mode: NCCL's watchdog thread may touch the CUDA API meanwhile).  Separate graphs with eager all-reduces
        # between them leave cross-stream waits in front of each replay: measured at two GPUs the step then
        # flips between 90 and 130 ms.
        g = torch.cuda.CUDAGraph()
        dynD = self.optD.dyn
        with torch.cuda.graph(g, pool=pool, stream=self.side, capture_error_mode="thread_local"):
            st = None
            for j in range(self.params.discrim_steps):
                st = _d_phase(self.gan, self.static_x, self.static_cond, dev, self.params, self.losses, None,
                              self.channel_first, False, j, st)
                if self.dist is not None:
                    self.dist.reduce_grads(self.optD)
                self.optD.dyn = dynD[j]
                self.optD.step()
                # the iteration's lossD is the sum over its critic steps, as train_iteration returns it
                lossD = st["lossD"] if j == 0 else lossD + st["lossD"]
            self.optD.dyn = dynD
            st["lossD"] = lossD
            st = _g_phase(self.gan, st, self.params, self.losses)
            if self.dist is not None:
                self.dist.reduce_grads(self.optG)
            self.optG.step()
        self.state = st
        self.graphs = (g,)

    def __call__(self, x, y):
        """x (B,T,C,H,W) on the device (or pinned host), y = [tokens, lengths] -> (lossD, lossG) device scalars."""
        from . import hostrng, ops
        if not x.is_cuda:
            x = x.to(self.device, non_blocking=True)
            y = [a.to(self.device, non_blocking=True) if isinstance(a, torch.Tensor) else a for a in y]
        self.calls += 1
        if self.graphs is None and self.calls <= self.warmup:
            rec = hostrng.set_current(hostrng.RecordingDraws())
            try:
                self.side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(self.side):
                    ld, lg, _, _, _ = train_iteration(self.gan, x, y, self.device, self.optD, self.optG,
                                                      self.params, self.losses, self.channel_first, False, self.dist)
                torch.cuda.current_stream().wait_stream(self.side)
            finally:
                hostrng.set_current(hostrng.EagerDraws())
            self._calls_rec = rec.calls
            return ld, lg
        cond = encode_captions(self.gan, y, False)
        if self.graphs is None:
            self.draws = hostrng.StaticDraws(self._calls_rec, self.device)
            hostrng.set_current(self.draws)
            try:
                self._capture(K.u8_normalize(x.contiguous()) if x.dtype == torch.uint8 else x, cond)
            finally:
                hostrng.set_current(hostrng.EagerDraws())
        if x.is_cuda and x.dtype == torch.uint8 and x.is_contiguous() and self.static_x.is_contiguous():
            # frames as stored: ToTensor + Normalize fused into the fill of the graph's static input (t2v_u8_normalize)
            K.u8_normalize(x, out=self.static_x)
        elif x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and self.static_x.is_contiguous():
            # an SM copy kernel, not cudaMemcpyAsync: a copy-engine D2D copy would queue behind the prefetcher's
            # H2D chunks of the NEXT batch (data.data_prefetcher) and delay this step by the whole transfer
            K.multi_copy([x], [self.static_x])
        else:
            self.static_x.copy_(x, non_blocking=True)
        if cond is not None:
            if cond.dtype == torch.float32 and cond.is_contiguous() and self.static_cond.is_contiguous():
                K.multi_copy([cond], [self.static_cond])
            else:
                self.static_cond.copy_(cond)
        slot = self.replays % self.ring
        self.replays += 1
        if self.stage_evt[slot] is not None:
            self.stage_evt[slot].synchronize()
        self.draws.refresh(slot)
        self._stage_adam(self.optD, self.optD._step_count + 1, slot)
        self._stage_adam(self.optG, self.optG._step_count + 1, slot)
        self.stage_evt[slot] = torch.cuda.Event()
        self.stage_evt[slot].record()
        self.graphs[0].replay()
        self.optD._step_count += self.params.discrim_steps
        self.optG._step_count += 1
        ops.bump_weight_epoch()          # eager users of the modules must re-pack the updated weights
        return self.state["lossD"], self.state["lossG"]

    def sync_optimizer_state(self):
        """write the replayed step counts back into the optimisers' state (for checkpoints)"""
        for opt in (self.optD, self.optG):
            if not hasattr(opt, "_step_count"):
                continue
            for st_ in opt.state.values():
                st_["step"] = opt._step_count

    def begin_eager_step(self):
        """An eager iteration between replays (a ragged last batch): the fused Adam must take its bias corrections
        from the step count, not from the device slot the replays stage, and the count must advance."""
        self.sync_optimizer_state()
        self._saved_dyn = []
        for opt in (self.optD, self.optG):
            self._saved_dyn.append(getattr(opt, "dyn", None))
            opt.dyn = None

    def end_eager_step(self):
        for opt, dyn in zip((self.optD, self.optG), self._saved_dyn):
            opt.dyn = dyn
            if hasattr(opt, "_step_count"):
                opt._step_count = max([st_["step"] for st_ in opt.state.values()] or [opt._step_count])


class LaggedLosses(object):
    """Loss logging without stalling the launch pipeline (graph mode): every iteration's (lossD, lossG) is written into
    a pinned host slot by an SM copy kernel over UVA -- a cudaMemcpyAsync D2H would queue behind the prefetcher's H2D
    pieces, and float(tensor) waits for everything enqueued so far -- and handed to the rolling averages `lag`
    iterations later, when its event has long fired.  drain() delivers what is pending (before a log line / a
    checkpoint name / the end of an epoch).  With lag = 0 this is the reference's float(loss) per iteration."""

    def __init__(self, sink, lag=2, device=None):
        self.sink, self.lag = sink, lag
        self.cuda = device is not None and torch.device(device).type == 'cuda' and lag > 0
        self.pending = []
        if self.cuda:
            self.slots = [torch.zeros(2).pin_memory() for _ in range(lag + 1)]
            self.events = [torch.cuda.Event() for _ in range(lag + 1)]
            self.i = 0

    def push(self, ld, lg):
        if not self.cuda:
            self.sink(float(ld), float(lg))
            return
        k = self.i % (self.lag + 1)
        self.i += 1
        K.multi_copy([torch.stack((ld.detach().float().reshape(()), lg.detach().float().reshape(())))], [self.slots[k]])
        self.events[k].record()
        self.pending.append(k)
        while len(self.pending) > self.lag:
            self._deliver(self.pending.pop(0))

    def _deliver(self, k):
        self.events[k].synchronize()
        self.sink(float(self.slots[k][0]), float(self.slots[k][1]))

    def drain(self):
        while self.pending:
            self._deliver(self.pending.pop(0))


def train(gan=None, num_epoch=None, dataset=None, device=None, optD=None, optG=None, params=None, vocab=None,
          losses=None, channel_first=True, end2end=True, dist=None):
    """gan/trainer.py:111-333."""
    if getattr(params, 'debug', False):
        status("Parameter settings:")
        print(locals())
    if params.sample_batch_size is None:
        params.sample_batch_size = params.batch_size
    ensure_exists(params.out)
    ensure_exists(params.out_samples)
    from .data import data_prefetcher

    gen_loss, discrim_loss = RollingAvg(params.loss_window_size), RollingAvg(params.loss_window_size)
    avg_data_load, avg_iter = RollingAvg(params.log_period), RollingAvg(params.log_period)
    data_load_watch, iter_watch = Stopwatch(), Stopwatch()

    def _log_losses(d, g):
        discrim_loss.update(d)
        gen_loss.update(g)

    main_rank = dist is None or getattr(dist, "is_main", True)     # checkpoints / samples / logs: rank 0 only
    graphed = None
    if getattr(params, 'cuda_graphs', False) and torch.device(device).type == 'cuda' and not end2end \
            and params.gen_steps == 1:
        graphed = GraphedTrainStep(gan, optD, optG, params, losses, torch.device(device), channel_first=channel_first,
                                   end2end=False, dist=dist)
    lagged = LaggedLosses(_log_losses, lag=2 if graphed is not None else 0, device=device)

    for epoch in range(num_epoch):
        if params.log_period > 0:
            status('Epoch %d started' % (epoch + 1))
        data_load_watch.start()
        iter_watch.start()
        i = 0
        prefetcher = data_prefetcher(dataset, device=device, normalize=graphed is None)
        x, y = prefetcher.next(preload=False)
        while x is not None:
            iteration = epoch * len(dataset) + i + 1
            data_load_watch.stop()
            avg_data_load.update(data_load_watch.elapsed_time)

            if graphed is not None and x.size(0) == params.batch_size:
                ld, lg = graphed(x, y)
                st = getattr(graphed, "state", None) or {}
                fake, xs, cond = st.get("fake", []), st.get("xs", [x]), st.get("conds")
            else:
                if graphed is not None:
                    graphed.begin_eager_step()               # ragged last batch: plain Adam steps, counted
                ld, lg, fake, xs, cond = train_iteration(gan, x, y, device, optD, optG, params, losses,
                                                         channel_first=channel_first, end2end=end2end, dist=dist)
                if graphed is not None:
                    graphed.end_eager_step()
            prefetcher.preload()                 # the next batch's bulk copy is enqueued behind this iteration's launch
            # the reference's two host syncs per iteration (trainer.py:243,264); in graph mode the values reach the
            # rolling averages two iterations late so that the host stays ahead of the device
            lagged.push(ld, lg)
            saving = (iteration == 1 and params.save_initial) or iteration % params.save_example_period == 0
            if saving or (params.log_period > 0 and iteration % params.log_period == 0):
                lagged.drain()

            if main_rank and ((iteration == 1 and params.save_initial) or iteration % params.save_example_period == 0):
                if graphed is not None:
                    graphed.sync_optimizer_state()           # replays advance the step count outside optimizer.state
                to_save = {'optG': optG.state_dict(), 'optD': optD.state_dict()}
                to_save.update(gan.save_dict())
                torch.save(to_save, '%s/iter_%d_lossG_%.4f_lossD_%.4f' % (params.out, iteration, gen_loss.get(),
                                                                          discrim_loss.get()))
                del to_save
            if main_rank and params.log_period > 0 and iteration % params.log_period == 0:
                sys.stdout.flush()
                mem = (torch.cuda.max_memory_allocated() / 1e9, torch.cuda.max_memory_reserved() / 1e9) \
                    if torch.cuda.is_available() else (0.0, 0.0)
                status('[%d/%d; %d/%d] - Iter %d, Loss_D: %.4f Loss_G: %.4f (%.2fGB used; %.2fGB cached) - '
                       '%.4f sec/iter; %.4f sec/batch load' % (epoch, num_epoch, i, len(dataset), iteration,
                                                                discrim_loss.get(), gen_loss.get(), mem[0], mem[1],
                                                                avg_iter.get(), avg_data_load.get()))
                if torch.cuda.is_available():
                    torch.cuda.reset_peak_memory_stats()
            if main_rank and params.save_example_period > 0 and ((iteration == 1 and params.save_initial_examples) or
                                                                 iteration % params.save_example_period == 0):
                status('saving to %s (iteration %d)' % (params.out_samples, iteration))
                save_frames(xs[0], '%s/real_samples.png' % params.out_samples, is_images=params.img_model)
                for f in fake:
                    h, w = (f.size(2), f.size(3)) if params.img_model else (f.size(3), f.size(4))
                    save_frames(f.detach(), path='%s/fake_samples_epoch_%03d_iter_%06d_%dx%d.png' %
                                (params.out_samples, epoch, iteration, h, w), channel_first=channel_first,
                                is_images=params.img_model)
                if cond is not None and vocab is not None:
                    save_sentences(y[0], path='%s/sentences_epoch%03d_iter_%06d.txt' % (params.out_samples, epoch,
                                                                                       iteration), vocab=vocab)
            data_load_watch.start()
            iter_watch.stop()
            avg_iter.update(iter_watch.elapsed_time)
            iter_watch.start()
            x, y = prefetcher.next(preload=False)
            i += 1
        lagged.drain()
