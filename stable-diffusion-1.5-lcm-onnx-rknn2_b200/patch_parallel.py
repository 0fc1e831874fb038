"""Patch-parallel SDXL denoising over NVLink (BASELINE config C5, SURVEY.md §8e).

One image is latency-bound (30 serial UNet forwards, CFG batch 2), so the *single image* is
sharded: the world of N ranks is `cfg_ways x strips`:

  * cfg_ways = 2 (when N is even and the pass is classifier-free guided): ranks [0, N/2) run the
    unconditional half of the CFG batch, ranks [N/2, N) the conditional half — no exchange at
    all inside the UNet, one all-gather of the noise prediction per step;
  * strips = N / cfg_ways: each rank of a half owns `H/strips` latent rows of every feature map.
    Exchanges per layer (all inside the strip group, synchronous, so results do not depend on
    the rank count beyond fp32 summation order of the GroupNorm merge):
      X1  one halo row to each neighbour in front of every 3x3 conv          (`halo_exchange`)
      X2  all-gather of the self-attention K/V rows                           (`gather_rows`)
      X3  all-gather of per-(image, group) GroupNorm (mean, M2) records       (`all_gather`)
    Cross-attention, LayerNorm, FFN and the 1x1 convs are token-local.

Every rank keeps the full latent (64 KB): after the per-step all-gather of the strip outputs all
ranks run the same CFG combine + `LCMScheduler.step` kernels on identical inputs, so latents stay
bit-identical across ranks without a broadcast.  The VAE decode runs on rank 0, or (`vae_strips`)
as row strips over all N ranks with the same three exchanges (`VAEDecoderB200.decode_strips`).

Communicators: `DistComm` = torch.distributed (NCCL over NVLink on GPUs; gloo in the CPU tests);
`ThreadComm` = N virtual ranks as threads of one process on one device (test double that lets
the single-GPU `pytest -m gpu` run exercise the strip arithmetic end to end).
"""
from __future__ import annotations

import threading
from typing import List, Optional

import torch


class StripComm:
    """Collectives of one strip group.  Subclasses provide `all_gather(x) -> [world, *x.shape]`."""

    rank: int = 0
    world: int = 1

    def all_gather(self, x: torch.Tensor) -> torch.Tensor:
        raise NotImplementedError

    def gather_rows(self, x: torch.Tensor) -> torch.Tensor:
        """[B, n, ...] per rank -> [B, world*n, ...] in rank order (X2; strip outputs)."""
        g = self.all_gather(x.contiguous())                     # [R, B, n, ...]
        R, B, n = g.shape[:3]
        if B == 1:
            return g.reshape(1, R * n, *g.shape[3:])            # a view: no copy
        return g.transpose(0, 1).reshape(B, R * n, *g.shape[3:])

    def halo_exchange(self, t: torch.Tensor) -> None:
        """t [B, h+2, W, C]: rows 1 and h go to the neighbours, rows 0 and h+1 are filled from
        them (zeros at the image border) (X1)."""
        h = t.shape[1] - 2
        if self.world == 1:
            t[:, 0].zero_()
            t[:, h + 1].zero_()
            return
        edge = torch.stack([t[:, 1], t[:, h]], dim=1)           # [B, 2, W, C]: my first / last row
        g = self.all_gather(edge)                               # [R, B, 2, W, C]
        if self.rank > 0:
            t[:, 0].copy_(g[self.rank - 1, :, 1])
        else:
            t[:, 0].zero_()
        if self.rank < self.world - 1:
            t[:, h + 1].copy_(g[self.rank + 1, :, 0])
        else:
            t[:, h + 1].zero_()


class SingleComm(StripComm):
    """world == 1: exercises the split kernels (stats | apply, halo-padded convs) on one rank."""

    def all_gather(self, x):
        return x.unsqueeze(0)


class DistComm(StripComm):
    """torch.distributed process group (NCCL over NVLink 5 / NVSwitch on the GPU box)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self._dist = dist
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)

    def all_gather(self, x):
        x = x.contiguous()
        # concatenation along dim 0 (the layout every backend accepts), viewed as [world, ...]
        out = torch.empty((self.world * x.shape[0],) + tuple(x.shape[1:]), device=x.device, dtype=x.dtype)
        self._dist.all_gather_into_tensor(out, x, group=self.group)
        return out.view((self.world,) + tuple(x.shape))


class PeerComm(StripComm):
    """All-gathers as ONE kernel of ours over NVLink peer memory (`dl_peer_allgather`, csrc/peer.cu):
    stores into every peer's symmetric staging buffer, epoch flags in the peers' signal pads, no
    NCCL call and no pack / unpack kernels.  The buffers come from torch's symmetric-memory
    allocator (plumbing: it only maps the same allocation into every rank of the group)."""

    def __init__(self, group=None, slot_bytes: int = 16 << 20):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.rank = dist.get_rank(self.group)
        self.world = dist.get_world_size(self.group)
        self.slot_bytes = int(slot_bytes)
        dev = torch.device("cuda", torch.cuda.current_device())
        self._stage = symm_mem.empty(2 * self.world * self.slot_bytes, dtype=torch.uint8, device=dev)
        self._hdl = symm_mem.rendezvous(self._stage, self.group)
        self._stage_ptrs = [int(p) for p in self._hdl.buffer_ptrs]
        # our own epoch flags (one u32 per peer) in a second symmetric allocation: the handle's
        # signal pads stay reserved for torch's barrier
        self._flags = symm_mem.empty(64, dtype=torch.int32, device=dev)
        self._flags.zero_()
        self._fhdl = symm_mem.rendezvous(self._flags, self.group)
        self._flag_ptrs = [int(p) for p in self._fhdl.buffer_ptrs]
        self._state = torch.zeros(4, device=dev, dtype=torch.int32)
        torch.cuda.synchronize(dev)
        self._fhdl.barrier()                      # every rank's flags are zero before the first call
        torch.cuda.synchronize(dev)

    def all_gather(self, x):
        from . import lib
        x = x.contiguous()
        out = torch.empty((self.world,) + tuple(x.shape), device=x.device, dtype=x.dtype)
        lib.peer_allgather(x, out, self._stage_ptrs, self._flag_ptrs, self.rank, self.slot_bytes, self._state)
        return out

    def halo_exchange(self, t):
        """Rows 1 and h of t [B, h+2, W, C] go to the neighbours' rows h+1 / 0 — through the same
        gather kernel (both boundary rows of every rank; neighbours pick theirs)."""
        super().halo_exchange(t)

    # ---- all-gather fused into the producing GEMM ----------------------------------------------
    def _fused_setup(self, nbytes: int):
        import torch.distributed._symmetric_memory as symm_mem
        if getattr(self, "_fbuf_bytes", 0) >= nbytes:
            return
        # (re)allocation is collective and happens on the first call of a geometry, never under capture
        self._fbuf_bytes = max(int(nbytes), 32 << 20)
        dev = self._state.device
        self._fbuf = symm_mem.empty(2 * self._fbuf_bytes, dtype=torch.uint8, device=dev)
        self._fbuf_hdl = symm_mem.rendezvous(self._fbuf, self.group)
        self._fbuf_ptrs = [int(p) for p in self._fbuf_hdl.buffer_ptrs]
        self._fcalls = 0

    def gather_linear(self, linear_fn, B: int, rows: int, cols: int):
        """[B, R*rows, cols] bf16 = all-gather over the group of every rank's [B, rows, cols] GEMM
        output, with the gather fused into the GEMM: `linear_fn(out_view, peer_ptrs)` must launch
        the igemm whose epilogue TMA-stores each tile into `out_view` (this rank's row block of the
        local buffer) and into the same view of every peer's buffer.  A flag-only barrier kernel
        then orders the peers' NVLink writes before the consumer.  Halves of the symmetric buffer
        alternate per call (callers issue an even number of calls per captured graph)."""
        from . import lib
        R, esz = self.world, 2
        nbytes = B * R * rows * cols * esz
        self._fused_setup(nbytes)
        half = (self._fcalls & 1) * self._fbuf_bytes
        self._fcalls += 1
        full = self._fbuf[half:half + nbytes].view(torch.bfloat16).view(B, R * rows, cols)
        mine = full[:, self.rank * rows:(self.rank + 1) * rows]
        off = half + self.rank * rows * cols * esz                 # byte offset of my row block
        peers = [self._fbuf_ptrs[r] + off for r in range(R) if r != self.rank]
        linear_fn(mine, peers)
        lib.peer_barrier(self._stage_ptrs, self._flag_ptrs, self.rank, self.slot_bytes, self._state)
        return full


class _ThreadHub:
    def __init__(self, world: int):
        self.world = world
        self.barrier = threading.Barrier(world)
        self.slots: List[Optional[torch.Tensor]] = [None] * world


class ThreadComm(StripComm):
    """Virtual rank `rank` of `world` threads sharing one device (tests only)."""

    def __init__(self, hub: _ThreadHub, rank: int):
        self.hub, self.rank, self.world = hub, rank, hub.world

    @staticmethod
    def make(world: int) -> List["ThreadComm"]:
        hub = _ThreadHub(world)
        return [ThreadComm(hub, r) for r in range(world)]

    def all_gather(self, x):
        x = x.contiguous()
        if x.is_cuda:
            torch.cuda.current_stream(x.device).synchronize()   # my data is complete
        self.hub.slots[self.rank] = x
        self.hub.barrier.wait()
        out = torch.stack(list(self.hub.slots), dim=0)
        if x.is_cuda:
            torch.cuda.current_stream(x.device).synchronize()   # copies done before slots are reused
        self.hub.barrier.wait()
        return out


class Topology:
    """rank -> (cfg half, strip index) for a world of N ranks."""

    def __init__(self, world: int, rank: int, cfg: bool):
        self.world, self.rank = world, rank
        self.cfg_ways = 2 if (cfg and world % 2 == 0) else 1
        self.strips = world // self.cfg_ways
        self.cfg_index = rank // self.strips        # 0 = unconditional half, 1 = conditional
        self.strip_index = rank % self.strips

    def strip_ranks(self, cfg_index: int) -> List[int]:
        return list(range(cfg_index * self.strips, (cfg_index + 1) * self.strips))


def assemble_eps(g: torch.Tensor, topo: Topology, batch: int):
    """World all-gather of the per-rank strip outputs -> (eps_uncond, eps_text) full maps
    (or (eps, None) without CFG).  g: [world, b_local, hl, W, 4] with b_local = batch when the
    CFG halves live on different ranks, 2*batch when every rank runs the doubled batch."""
    W, C = g.shape[3], g.shape[4]
    hl = g.shape[2]

    def rows(block):                                   # [strips, b, hl, W, C] -> [b, strips*hl, W, C]
        s, b = block.shape[:2]
        if b == 1:
            return block.reshape(1, s * hl, W, C)
        return block.transpose(0, 1).reshape(b, s * hl, W, C)

    if topo.cfg_ways == 2:
        return rows(g[:topo.strips]), rows(g[topo.strips:])
    full = rows(g)
    if full.shape[0] == 2 * batch:
        return full[:batch], full[batch:]
    return full, None


class PatchParallelDenoiser:
    """The LCM loop of `LCMPipelineB200` with the UNet sharded over a world communicator."""

    def __init__(self, pipe, world_comm: StripComm, strip_comm_factory=None):
        """pipe: LCMPipelineB200 of this rank.  world_comm spans all ranks; strip_comm_factory
        (ranks -> StripComm) builds the communicator of this rank's strip group (default: the
        world itself when there is no CFG split)."""
        self.pipe = pipe
        self.world = world_comm
        self._strip_factory = strip_comm_factory
        self._strip_comms = {}
        self._graphs = {}
        self.force_split = False     # tests: run the strip kernels even for a one-strip group

    def _strip_comm(self, topo: Topology) -> Optional[StripComm]:
        if topo.strips == 1 and not self.force_split:
            return None                              # whole image on this rank: the fused single-GPU kernels
        if topo.cfg_ways == 1:
            return self.world
        key = topo.cfg_index
        if key not in self._strip_comms:
            self._strip_comms[key] = self._strip_factory(topo)
        return self._strip_comms[key]

    @torch.no_grad()
    def _prepare(self, prompt_embeds, pooled_embeds, B, H, W, guidance_scale):
        """Per-rank conditioning of this rank's role -> (topo, comm, pe, add, w_emb, repeat, cfg_scale)."""
        pipe = self.pipe
        cfg_scale = pipe.cfg_scale_for(guidance_scale)
        topo = Topology(self.world.world, self.world.rank, cfg_scale is not None)
        comm = self._strip_comm(topo)
        w_emb = pipe._w_emb(B, guidance_scale)
        pe_all, add = pipe._conditioning(prompt_embeds, pooled_embeds, None, None, None, cfg_scale,
                                         8 * H, 8 * W)
        repeat = 1
        if cfg_scale is not None:
            if topo.cfg_ways == 2:                  # my half of the [uncond, cond] conditioning
                sl = slice(topo.cfg_index * B, (topo.cfg_index + 1) * B)
                pe_all = pe_all[sl]
                add = (add[0][sl], add[1][sl]) if add is not None else None
            else:
                repeat = 2
        return topo, comm, pe_all, add, w_emb, repeat, cfg_scale

    @torch.no_grad()
    def _loop(self, topo, comm, pe, add, we, repeat, cfg_scale, lat_nchw, noise_nchw, steps, record=None,
              teacher=None):
        """Device tensors in, final latents NHWC out; no host sync (graph-capturable)."""
        from . import lib
        pipe = self.pipe
        dev = pipe.device
        B, C, H, W = lat_nchw.shape
        sched = pipe.schedule(steps)                   # the pipeline's scheduler config
        kvs = pipe.unet.encode_context(pe)
        aug = pipe.unet.addition_embedding(*add) if add is not None else None
        tembs = pipe.unet.time_embeddings(sched.timesteps, B * repeat, we, aug)
        x = torch.empty(B, H, W, C, device=dev, dtype=torch.float32)
        lib.nchw_to_nhwc_f32(lat_nchw, x)
        noise = None
        if steps > 1:
            noise = torch.empty(steps - 1, B, H, W, C, device=dev, dtype=torch.float32)
            lib.nchw_to_nhwc_f32(noise_nchw[:steps - 1].reshape((steps - 1) * B, C, H, W),
                                 noise.view((steps - 1) * B, H, W, C))
        den = torch.empty_like(x)
        tx = None
        if teacher is not None:          # parity tests: step i starts from a given trajectory (teacher forcing)
            tx = torch.empty(steps, B, H, W, C, device=dev, dtype=torch.float32)
            lib.nchw_to_nhwc_f32(teacher.to(dev, torch.float32).reshape(steps * B, C, H, W).contiguous(),
                                 tx.view(steps * B, H, W, C))
        for i in range(steps):
            if tx is not None:
                x = tx[i]
            strip = pipe.unet.forward(x, tembs[i], kvs, repeat=repeat, comm=comm)
            e_u, e_t = assemble_eps(self.world.all_gather(strip), topo, B)
            if e_t is not None:
                eps = torch.empty_like(x)
                lib.cfg_combine(e_u.contiguous(), e_t.contiguous(), cfg_scale, eps)
                if record is not None:
                    record.setdefault("noise_pred_raw", []).append(
                        torch.cat([e_u, e_t], 0).permute(0, 3, 1, 2).clone())
            else:
                eps = e_u.contiguous()
            x_next = torch.empty_like(x)
            lib.lcm_step_ex(eps, x, noise[i] if sched.has_noise(i) else None, x_next, den, sched.coeffs(i),
                            sched.prediction_type, sched.clip_range)
            if record is not None:
                record.setdefault("noise_pred", []).append(eps.permute(0, 3, 1, 2).clone())
                record.setdefault("latents", []).append(x_next.permute(0, 3, 1, 2).clone())
            x = x_next
        return x

    @torch.no_grad()
    def denoise(self, prompt_embeds, pooled_embeds, latents_nchw, step_noise_nchw, steps: int,
                guidance_scale: float, record: dict = None, use_graph: bool = False, teacher_latents=None):
        """Inputs as `LCMPipelineB200.generate` (host or device, identical on every rank).
        Returns the final latents NHWC fp32 (identical on every rank).  use_graph: the whole
        loop — kernels and collectives — is captured once per geometry and replayed (one image
        at N ranks is otherwise bound by launch latency, not by the GPUs)."""
        pipe = self.pipe
        dev = pipe.device
        B, C, H, W = latents_nchw.shape
        topo, comm, pe_all, add, w_emb, repeat, cfg_scale = self._prepare(
            prompt_embeds, pooled_embeds, B, H, W, guidance_scale)
        with torch.cuda.device(dev):
            pe = pe_all.to(dev, torch.bfloat16).contiguous()
            if add is not None:
                add = (add[0].to(dev).contiguous(), add[1].to(dev).contiguous())
            we = w_emb.to(dev) if w_emb is not None else None
            lat0 = latents_nchw.to(dev, torch.float32).contiguous()
            nz = step_noise_nchw.to(dev, torch.float32).contiguous() if steps > 1 else None
            if not use_graph or record is not None or teacher_latents is not None:
                return self._loop(topo, comm, pe, add, we, repeat, cfg_scale, lat0, nz, steps, record,
                                  teacher=teacher_latents)
            key = (B, H, W, steps, cfg_scale)
            g = self._graphs.get(key)
            if g is None:
                st = dict(pe=pe.clone(), add=None if add is None else (add[0].clone(), add[1].clone()),
                          we=None if we is None else we.clone(), lat=lat0.clone(),
                          nz=None if nz is None else nz.clone())
                args = lambda: (topo, comm, st["pe"], st["add"], st["we"], repeat, cfg_scale, st["lat"],  # noqa: E731
                                st["nz"], steps)
                s = torch.cuda.Stream(device=dev)
                s.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(s):
                    self._loop(*args())                           # warm-up (lazy init, NCCL channels)
                torch.cuda.current_stream(dev).wait_stream(s)
                torch.cuda.synchronize(dev)
                graph = torch.cuda.CUDAGraph()
                f0 = getattr(comm, "_fcalls", 0)
                with torch.cuda.graph(graph, stream=s, capture_error_mode="thread_local"):
                    st["out"] = self._loop(*args())
                if (getattr(comm, "_fcalls", 0) - f0) % 2:
                    raise RuntimeError("patch parallel: a captured loop must issue an even number of fused "
                                       "gathers (the peer buffers alternate halves per call)")
                st["graph"] = graph
                g = self._graphs[key] = st
            g["pe"].copy_(pe)
            if add is not None:
                g["add"][0].copy_(add[0]); g["add"][1].copy_(add[1])
            if we is not None:
                g["we"].copy_(we)
            g["lat"].copy_(lat0)
            if nz is not None:
                g["nz"].copy_(nz)
            g["graph"].replay()
            return g["out"]

    @torch.no_grad()
    def generate(self, prompt_embeds, pooled_embeds, latents_nchw, step_noise_nchw, steps: int,
                 guidance_scale: float, record: dict = None, decode_rank: int = 0, use_graph: bool = False,
                 vae_strips: bool = False):
        """-> u8 images [B,H,W,3] on `decode_rank` (None elsewhere).  vae_strips: the decode is
        sharded too — every rank of the WORLD (there is no CFG batch in the decoder, so all
        cfg_ways x strips ranks form one strip group) decodes H/N latent rows
        (`VAEDecoderB200.decode_strips`) and every rank returns the full image."""
        if vae_strips and getattr(self.pipe, "vae_kind", "kl") == "taesd":
            raise RuntimeError("vae_strips: the tiny autoencoder (AutoencoderTiny) has no strip-parallel decode; "
                               "decode on one rank (vae_strips=False)")
        lat = self.denoise(prompt_embeds, pooled_embeds, latents_nchw, step_noise_nchw, steps,
                           guidance_scale, record, use_graph=use_graph)
        if vae_strips and self.world.world > 1:
            with torch.cuda.device(self.pipe.device):
                return self.pipe.vae.decode_strips(lat, self.world)
        if self.world.rank != decode_rank:
            return None
        with torch.cuda.device(self.pipe.device):
            return self.pipe.vae.decode(lat)


def dist_denoiser(pipe, cfg: bool = True, peer: bool = False) -> "PatchParallelDenoiser":
    """PatchParallelDenoiser over the default torch.distributed world: builds the two strip
    groups of the CFG halves (every rank must call this: `new_group` is collective).
    peer=True: exchanges run as `dl_peer_allgather` kernels over NVLink peer memory instead of
    NCCL all-gathers."""
    import torch.distributed as dist
    make = PeerComm if peer else DistComm
    world = make()
    groups, comms = {}, {}
    if cfg and world.world % 2 == 0 and world.world > 2:
        topo = Topology(world.world, world.rank, True)
        for c in range(2):
            groups[c] = dist.new_group(topo.strip_ranks(c))
        if peer:                                  # rendezvous is collective inside its group
            comms[topo.cfg_index] = PeerComm(groups[topo.cfg_index])

    def factory(topo: Topology):
        if topo.cfg_index in comms:
            return comms[topo.cfg_index]
        return make(groups[topo.cfg_index])

    return PatchParallelDenoiser(pipe, world, factory)
