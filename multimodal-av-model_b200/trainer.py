"""MultimodalTrainer — drop-in for /root/reference/model/trainer.py:12-252 with the hot path on sm_100a kernels.

Same constructor, attributes and methods (SURVEY.md §8b):

    MultimodalTrainer(visual_encoder, audio_encoder, fusion_module, decoder1, tokenizer,
                      learning_rate=1e-4, device="cuda", lambda_=0.1)
    .train_epoch(dataloader) -> float          .evaluate(dataloader) -> (avg_loss, avg_wer)
    .ctc_decode(pred_ids)                      .crop_or_pad_feat(feat, target_len)
    .align(batch) -> token time spans of both speakers' reference transcripts (not in the reference; CTC forced alignment)
    attributes: visual_encoder audio_encoder fusion_module decoder1 tokenizer optimizer device lambda_ ctc_loss

Differences that matter (all deliberate, none changes a result):
  * the CTC loss, InfoNCE, fusion module, CTC head and beam search are this package's kernels
  * mixed precision is bf16 autocast (no GradScaler needed); the reference uses fp16 + GradScaler (trainer.py:9,40)
  * the reference's per-sample label sanity prints (trainer.py:77-85, 3B host syncs per step) are dropped
  * evaluate() decodes a whole batch with one beam-search launch instead of 2B Python loops
  * train_epoch() never blocks on the GPU inside the loop: the next batch's host->device copies are issued (side
    stream) as soon as the current step is enqueued, and each step's loss goes to the host through a non-blocking
    copy into the pinned `loss_log` (the reference's `loss.item()` per batch, trainer.py:125, is one sync per step)
  * when torch.distributed is initialised the step is utterance-sharded data parallel: every rank runs its own
    batch, gradients are averaged with a bucketed NCCL all-reduce overlapped with backward (ddp.py)
"""
from __future__ import annotations

import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .align import TimedTokenSpan, forced_align, fused_frame_encoder_index, merge_tokens_batch
from .beam_search import beam_search_batch, fast_decode
from .contrastive import contrastive_loss_with_mask
from .ctc import CTCLoss
from .ddp import GradBucketReducer, broadcast_buffers, broadcast_module
from .context_graph import ContextGraph
from .prefix_beam import ctc_prefix_beam_search


def word_error_rate(refs, hyps):
    """jiwer.wer(refs, hyps) semantics: total word-level edit distance / total reference words."""
    try:
        from jiwer import wer as _wer
        return _wer(refs, hyps)
    except Exception:
        pass
    edits = words = 0
    for r, h in zip(refs, hyps):
        r, h = r.split(), h.split()
        prev = list(range(len(h) + 1))
        for i, rw in enumerate(r, 1):
            cur = [i] + [0] * len(h)
            for j, hw in enumerate(h, 1):
                cur[j] = min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (rw != hw))
            prev = cur
        edits += prev[-1]
        words += len(r)
    return edits / words if words else (0.0 if edits == 0 else float("inf"))


def _log_softmax_again(lp):
    """evaluate() re-normalises the decoder's log-probs (trainer.py:212,221); kept for bit-faithful inputs to
    the eval CTC loss and the beam search."""
    x = lp.detach().float().contiguous()
    out = torch.empty_like(x)
    V = x.shape[-1]
    with _lib.device_guard(x.device):
        _lib.check(_lib.lib().avctc_log_softmax_forward(x.data_ptr(), _lib.F32, out.data_ptr(), _lib.F32, x.numel() // V, V,
                                                        _lib.stream_ptr(x.device)), "avctc_log_softmax_forward")
    return out


class StagedBatch(dict):
    """A collated batch whose host->device copies have been issued (MultimodalTrainer.stage): device tensors, the
    per-clip wait callables and the host-side lengths the audio encoder uses."""


_END = object()          # train_epoch: the dataloader is exhausted


class MultimodalTrainer:
    cache_frozen_casts = True       # encoders.install_frozen_cast_cache on the two encoders (frozen weights only)

    def __init__(self, visual_encoder, audio_encoder, fusion_module, decoder1, tokenizer, learning_rate=1e-4,
                 device="cuda", lambda_=0.1):
        self.visual_encoder = visual_encoder.to(device)
        self.audio_encoder = audio_encoder.to(device)
        self.fusion_module = fusion_module.to(device)
        self.decoder1 = decoder1.to(device)
        self.tokenizer = tokenizer
        self.device = device
        self.lambda_ = lambda_
        self.ctc_loss = CTCLoss(blank=tokenizer.blank_id, zero_infinity=True)
        self.parameters = (list(self.visual_encoder.parameters()) + list(self.audio_encoder.parameters()) +
                           list(self.fusion_module.parameters()) + list(self.decoder1.parameters()))
        self.optimizer = torch.optim.Adam([
            {"params": self.visual_encoder.parameters(), "lr": learning_rate},
            {"params": self.audio_encoder.parameters(), "lr": 2e-5},
            {"params": self.fusion_module.parameters(), "lr": learning_rate},
            {"params": self.decoder1.parameters(), "lr": learning_rate}],
            **({"fused": True} if str(device).startswith("cuda") else {}))   # same update rule, one kernel per group
        self.autocast_dtype = torch.bfloat16
        if self.cache_frozen_casts:
            from .encoders import install_frozen_cast_cache
            for m in (self.visual_encoder, self.audio_encoder):
                install_frozen_cast_cache(m)
        self.projection_layer = None
        self.verbose = True
        self.beam_width = 5                       # trainer.py:230,237
        self.batch_speakers = True                # BiLSTM + CTC head over both speakers at once (hot_path_loss)
        self.overlap_contrastive = True           # InfoNCE on a side stream, under the BiLSTM kernels (hot_path_loss)
        self.gpu_heavy_first = False              # train_step enqueue order (see there); measured slower on B200, kept as a switch
        self.prefetch_batches = True              # train_epoch: stage batch i+1 while step i runs on the GPU
        self.loss_log = None                      # pinned fp32 ring: per-step total loss of the current epoch (async D2H)
        self.loss_log_count = 0                   # steps logged this epoch; entries are valid after a synchronize
        self.last_epoch_steps = 0                 # steps of the last train_epoch that did not raise
        self.world_size = dist.get_world_size() if dist.is_initialized() else 1
        self._reducer = None
        if self.world_size > 1:
            for m in (self.visual_encoder, self.audio_encoder, self.fusion_module, self.decoder1):
                broadcast_module(m)
            never = list(getattr(self.fusion_module, "never_used_parameters", lambda: [])())
            self._reducer = GradBucketReducer(self.parameters, never_used=never)

    # ------------------------------------------------------------------------------------------ helpers
    def crop_or_pad_feat(self, feat, target_len):
        if feat.size(0) >= target_len:
            return feat[:target_len]
        pad = torch.zeros(target_len - feat.size(0), feat.size(1), device=feat.device)
        return torch.cat([feat, pad], dim=0)

    def ctc_decode(self, pred_ids):
        """Greedy collapse of trainer.py:168-177: blanks are skipped WITHOUT resetting `prev`."""
        out, prev = [], None
        blank = self.tokenizer.blank_id
        for idx in pred_ids:
            if idx == blank:
                continue
            if idx != prev:
                out.append(idx)
            prev = idx
        return out

    def _to_dev(self, batch):
        """Host -> device.  Pinned host tensors are copied on a side stream (small tensors first, the two 44 MB lip
        clips last); `lips` entries are zero-argument callables that make the main stream wait for exactly the clip it
        is about to consume, so the audio encoder runs while the lip frames are still in flight."""
        dev = self.device
        on_gpu = str(dev).startswith("cuda")
        any_host = on_gpu and any(torch.is_tensor(v) and not v.is_cuda for v in batch.values())
        if not any_host:
            g = lambda k: batch[k].to(dev, non_blocking=True)
            gt = lambda k: g(k) if k in batch else None          # transcripts: absent when only decoding
            lips = [g("lip1").permute(0, 2, 1, 3, 4).contiguous(), g("lip2").permute(0, 2, 1, 3, 4).contiguous()]
            return dict(lips=[(lambda t=t: t) for t in lips], audio=g("audio"), masks=[g("mask1"), g("mask2")],
                        texts=[gt("text1"), gt("text2")], lens=[gt("text1_lengths"), gt("text2_lengths")])
        main = torch.cuda.current_stream(dev)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        cs = self._copy_stream            # (the caching allocator orders cross-stream reuse through record_stream)
        out, events = {}, {}
        with torch.cuda.stream(cs):
            for k in ("audio", "mask1", "mask2", "text1", "text2", "text1_lengths", "text2_lengths"):
                if k.startswith("text") and k not in batch:
                    continue
                out[k] = batch[k].to(dev, non_blocking=True)
            events["small"] = cs.record_event()
            for k in ("lip1", "lip2"):
                out[k] = batch[k].to(dev, non_blocking=True).permute(0, 2, 1, 3, 4).contiguous()
                events[k] = cs.record_event()
        for t in out.values():
            t.record_stream(main)
        main.wait_event(events["small"])

        def lip(k):
            def get():
                torch.cuda.current_stream(dev).wait_event(events[k])
                return out[k]
            return get
        return dict(lips=[lip("lip1"), lip("lip2")], audio=out["audio"], masks=[out["mask1"], out["mask2"]],
                    texts=[out.get("text1"), out.get("text2")], lens=[out.get("text1_lengths"), out.get("text2_lengths")])

    def _host_lengths(self, batch, key):
        """Utterance lengths (samples that are not padding, label 3) from the HOST copy of a mask, when there is one:
        lets the audio encoder draw its SpecAugment spans without reading the lengths back from the GPU."""
        m = batch.get(key)
        if not torch.is_tensor(m):
            return {}
        # a device-resident mask is read back HERE, before the step's work is enqueued — once per tensor: the same
        # (unmodified) mask tensor seen again, e.g. a batch kept resident in HBM across steps, reuses the lengths
        cache = self.__dict__.setdefault("_hl_cache", {})
        hit = cache.get(key)
        if hit is not None and hit[0]() is m and hit[1] == m._version:
            return {"host_lengths": hit[2]}
        # count_nonzero, not (m != 3).sum(-1): the bool -> int64 sum of a [B, 80000] host mask costs milliseconds of
        # host time per call (47 ms on 8 cores in the build container) against 0.2 ms, with the GPU idle meanwhile
        lens = torch.count_nonzero(m != 3, dim=-1).cpu()
        import weakref
        cache[key] = (weakref.ref(m), m._version, lens)
        return {"host_lengths": lens}

    def stage(self, batch):
        """Issue the host->device copies of one collated batch and return it as a StagedBatch that train_step accepts
        in place of the batch.  Nothing here waits for the GPU; train_epoch calls it one batch ahead."""
        if isinstance(batch, StagedBatch):
            return batch
        kw = [{}, {}]
        if hasattr(self.audio_encoder, "prefetch_features"):
            kw = [self._host_lengths(batch, "mask1"), self._host_lengths(batch, "mask2")]
        d = StagedBatch(self._to_dev(batch))
        d["enc_kw"] = kw
        return d

    _LOSS_LOG_CAP = 1 << 16

    def _log_loss(self, loss):
        """Device scalar -> pinned host ring, non-blocking: the per-step read-back without a per-step sync."""
        if not loss.is_cuda:
            return
        if self.loss_log is None:
            self.loss_log = torch.zeros(self._LOSS_LOG_CAP, dtype=torch.float32).pin_memory()
        self.loss_log[self.loss_log_count % self._LOSS_LOG_CAP].copy_(loss.detach().float(), non_blocking=True)
        self.loss_log_count += 1

    def _side_stream(self, ref):
        """Stream for work that is independent of the main chain (None on CPU tensors or when switched off)."""
        if not ref.is_cuda or not self.overlap_contrastive or torch.cuda.is_current_stream_capturing():
            return None
        st = getattr(self, "_aux_stream", None)
        if st is None or st.device != ref.device:
            st = self._aux_stream = torch.cuda.Stream(device=ref.device)
            # the projection layer's gradients are produced on the side stream and accumulated by nodes created on the
            # main stream: intended (autograd synchronises the two), so the advisory warning about it is switched off
            quiet = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
            if quiet is not None:
                quiet(False)
        return st

    def _ensure_projection(self, D):
        if self.projection_layer is None:           # trainer.py:105-106: created lazily, once per epoch
            self.projection_layer = nn.Linear(D, 128).to(self.device)
            if self.world_size > 1:
                broadcast_module(self.projection_layer)

    def hot_path_loss(self, visual_feats, audio_feats, middle_feats, masks, texts, lens):
        """trainer.py:98-119 from encoder features on (two speakers): returns (total, ctc1, ctc2, con1, con2)."""
        ctc, con, mask_ds = [], [], []
        for s in range(2):
            t_enc = audio_feats[s].shape[1]
            mask_ds.append(F.interpolate(masks[s].unsqueeze(1).float(), size=t_enc, mode="nearest").squeeze(1).long())
            self._ensure_projection(audio_feats[s].shape[2])
        # The two contrastive losses depend on nothing the fusion -> BiLSTM -> head -> CTC chain produces, and that chain
        # is dominated by the persistent BiLSTM kernels, which occupy 64 of the 148 SMs: the InfoNCE kernels (forward
        # here, backward through autograd, which replays an op on the stream its forward ran on) go to a side stream
        # and run on the idle SMs underneath it.  Same kernels, same values.
        side = self._side_stream(middle_feats[0])
        if side is not None:
            main = torch.cuda.current_stream(middle_feats[0].device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                for s in range(2):
                    middle_feats[s].record_stream(side); mask_ds[s].record_stream(side)
                    con.append(contrastive_loss_with_mask(middle_feats[s], mask_ds[s].reshape(-1),
                                                          projection_layer=self.projection_layer))
        else:
            for s in range(2):
                con.append(contrastive_loss_with_mask(middle_feats[s], mask_ds[s].reshape(-1),
                                                      projection_layer=self.projection_layer))
        if self.batch_speakers and hasattr(self.fusion_module, "forward_pair"):
            # the recurrent model and the CTC head see both speakers as one batch of 2B sequences (same values, half
            # the sequential steps); everything whose result depends on the batch it is computed in stays per speaker
            fused, in_lens = self.fusion_module.forward_pair(visual_feats, audio_feats, mask_ds)
            if fused[0].shape == fused[1].shape:
                lp = self.decoder1(torch.cat(fused, dim=0))
                log_probs = (lp[:fused[0].shape[0]], lp[fused[0].shape[0]:])
            else:
                log_probs = (self.decoder1(fused[0]), self.decoder1(fused[1]))
        else:
            fused, in_lens, log_probs = [None, None], [None, None], [None, None]
            for s in range(2):
                fused[s], in_lens[s] = self.fusion_module(visual_feats[s], audio_feats[s], mask=mask_ds[s])
                log_probs[s] = self.decoder1(fused[s])
        for s in range(2):
            ctc.append(self.ctc_loss(log_probs[s].transpose(0, 1), texts[s], in_lens[s], lens[s]))
        self._last_log_probs = log_probs[0]
        if side is not None:
            main.wait_stream(side)
            for c in con:
                c.record_stream(main)
        total = (ctc[0] + ctc[1]) / 2 + self.lambda_ * (con[0] + con[1]) / 2
        return total, ctc[0], ctc[1], con[0], con[1]

    def _forward_backward(self, batch):
        if isinstance(batch, Exception):          # a staging error (train_epoch._stage_next) fails THIS step, inside the
            raise batch                           # step protocol, so that under DDP the peers are not left waiting
        if hasattr(self.audio_encoder, "begin_step"):
            self.audio_encoder.begin_step()       # the feature-extractor cache serves the second call of THIS step only
        with torch.autocast("cuda", dtype=self.autocast_dtype, enabled=str(self.device).startswith("cuda")):
            d = self.stage(batch)
            kw = d["enc_kw"]
            # Enqueue order.  Default: audio encoder (small H2D) first so that the two 44 MB lip clips copy behind it.
            # gpu_heavy_first enqueues the conv front ends before the ~1500 small transformer launches; on B200 the
            # step is GPU-bound (~47 ms of kernels) and that order measured 3 ms slower (tools/exp_step.py).
            heavy_first = self.gpu_heavy_first and hasattr(self.audio_encoder, "prefetch_features")
            if heavy_first:
                self.audio_encoder.prefetch_features(d["audio"])
                vis = [self.visual_encoder(d["lips"][0]()), self.visual_encoder(d["lips"][1]())]
            aud, mid = [], []
            for s in range(2):
                a, m = self.audio_encoder(d["audio"], attention_mask=(d["masks"][s] != 3), **kw[s])
                aud.append(a); mid.append(m)
            if not heavy_first:
                vis = [self.visual_encoder(d["lips"][0]()), self.visual_encoder(d["lips"][1]())]
            total, c1, c2, k1, k2 = self.hot_path_loss(vis, aud, mid, d["masks"], d["texts"], d["lens"])
        total.backward()
        return total, c1, c2, k1, k2

    def train_step(self, batch):
        """One optimisation step on one collated batch, or on a StagedBatch from stage() (the body of the reference's
        loop, trainer.py:64-125).  Returns the detached total loss (device tensor; no host sync)."""
        if self._reducer is not None:
            self._reducer.zero_grad()           # .grad = zeroed views into the all-reduce buckets
        else:
            self.optimizer.zero_grad()
        err = None
        try:
            total, c1, c2, k1, k2 = self._forward_backward(batch)
        except Exception as e:
            if self._reducer is None:
                raise
            err = e
        if self._reducer is not None:
            # every rank reduces every bucket and applies the same update, also when ITS step raised (it then contributes
            # zeros and is left out of the average, ddp.GradBucketReducer.finish); the error surfaces afterwards
            self._reducer.finish(ok=err is None)
        self.optimizer.step()
        if err is not None:
            raise err
        self._last_parts = (c1.detach(), c2.detach(), k1.detach(), k2.detach())
        return total.detach()

    # ------------------------------------------------------------------------------------------ epochs
    def _stage_next(self, it):
        """Next batch of the iterator, staged; _END when exhausted.  A staging error is returned, not raised: it
        belongs to that batch's turn in the loop (same `except Exception: continue` policy as a failing step)."""
        try:
            batch = next(it)
        except StopIteration:
            return _END
        if not self.prefetch_batches or not str(self.device).startswith("cuda"):
            return batch
        try:
            return self.stage(batch)
        except Exception as e:
            return e

    def train_epoch(self, dataloader):
        for m in (self.visual_encoder, self.audio_encoder, self.fusion_module, self.decoder1):
            m.train()
        self.projection_layer = None
        total_loss = torch.zeros((), device=self.device)
        self.loss_log_count = 0
        n = 0
        it = iter(dataloader)
        cur = self._stage_next(it)
        batch_idx = -1
        while cur is not _END:
            batch_idx += 1
            loss = None
            try:
                loss = self.train_step(cur)
            except Exception as e:                      # same policy as trainer.py:162-164
                print(f"Error at batch {batch_idx}: {e}", flush=True)
            # the next batch's copies run (side stream) under this step's GPU work; an error of the iterator itself
            # propagates, as it does out of the reference's `for` statement
            cur = self._stage_next(it)
            if loss is None:
                continue
            try:
                total_loss += loss.float()
                self._log_loss(loss)
                if self.verbose and batch_idx % 100 == 0:
                    c1, c2, k1, k2 = (float(x) for x in self._last_parts)
                    print(f"[Batch {batch_idx}] CTC1: {c1:.4f}, CTC2: {c2:.4f}, Contrast1: {k1:.4f}, "
                          f"Contrast2: {k2:.4f}, Total: {float(loss):.4f}", flush=True)
                    pred = torch.argmax(self._last_log_probs[0], dim=-1).cpu().tolist()
                    print(f"[pred] {self.tokenizer.decode(self.ctc_decode(pred))}", flush=True)
                n += 1
            except Exception as e:
                print(f"Error at batch {batch_idx}: {e}", flush=True)
        self.last_epoch_steps = n
        return float(total_loss) / max(len(dataloader), 1)

    def evaluate(self, dataloader):
        for m in (self.visual_encoder, self.audio_encoder, self.fusion_module, self.decoder1):
            m.eval()
            if self.world_size > 1:
                broadcast_buffers(m)          # BatchNorm running statistics: rank 0's, on every rank
        refs, hyps = [[], []], [[], []]
        total_loss = 0.0
        blank = self.tokenizer.blank_id
        with torch.no_grad():
            for batch in dataloader:
                if hasattr(self.audio_encoder, "begin_step"):
                    self.audio_encoder.begin_step()
                d = self._to_dev(batch)
                with torch.autocast("cuda", dtype=self.autocast_dtype, enabled=str(self.device).startswith("cuda")):
                    lps, losses = [], []
                    # collate_fn pads mask1 and mask2 with 3 at the same positions (dataset/collate_fn.py:39-44), so both
                    # speakers see the same attention mask and, in eval mode, bit-identical audio features
                    # (trainer.py:206-207,215-216 computes them twice): one encoder pass serves both when the masks agree
                    att = [d["masks"][0] != 3, d["masks"][1] != 3]
                    shared = None
                    if torch.equal(att[0], att[1]):
                        shared, _ = self.audio_encoder(d["audio"], attention_mask=att[0])
                    for s in range(2):
                        vis = self.visual_encoder(d["lips"][s]())
                        aud = shared if shared is not None else self.audio_encoder(d["audio"], attention_mask=att[s])[0]
                        t_enc = aud.shape[1]
                        mask_ds = F.interpolate(d["masks"][s].unsqueeze(1).float(), size=t_enc, mode="nearest").squeeze(1).long()
                        fused, il = self.fusion_module(vis, aud, mask_ds)
                        if hasattr(self.decoder1, "log_probs"):       # both normalisations inside the head kernel
                            lp = self.decoder1.log_probs(fused, passes=2)
                        else:
                            lp = _log_softmax_again(self.decoder1(fused))
                        losses.append(self.ctc_loss(lp.transpose(0, 1), d["texts"][s], il, d["lens"][s]))
                        lps.append(lp)
                total_loss += (losses[0].item() + losses[1].item()) / 2
                B = lps[0].shape[0]
                if lps[0].shape[1:] == lps[1].shape[1:]:
                    ids = beam_search_batch(torch.cat(lps, 0), beam_width=self.beam_width, blank=blank)   # all 2B at once
                else:       # collate_fn pads lip1 and lip2 separately (dataset/collate_fn.py:18-23): T_v1 != T_v2 is the
                    ids = []   # normal case on real data; each speaker then decodes exactly its own padded T (trainer.py:230,237)
                    for lp_s in lps:
                        ids.extend(beam_search_batch(lp_s, beam_width=self.beam_width, blank=blank))
                lens_h = [d["lens"][0].cpu().tolist(), d["lens"][1].cpu().tolist()]
                texts_h = [d["texts"][0].cpu(), d["texts"][1].cpu()]
                for i in range(B):
                    for s in range(2):
                        hyps[s].append(fast_decode(ids[s * B + i], self.tokenizer))
                        refs[s].append(self.tokenizer.decode(texts_h[s][i][:lens_h[s][i]].tolist()))
        wer1 = word_error_rate(refs[0], hyps[0])
        wer2 = word_error_rate(refs[1], hyps[1])
        avg_wer = (wer1 + wer2) / 2
        avg_loss = total_loss / max(len(dataloader), 1)
        if self.verbose:
            print(f"[Eval] WER1: {wer1:.3f}, WER2: {wer2:.3f}, Avg: {avg_wer:.3f}, Loss: {avg_loss:.4f}")
        return avg_loss, avg_wer

    # ------------------------------------------------------------------------------------------ alignment
    hop_seconds = 320 / 16000                 # wav2vec2 encoder frame hop at 16 kHz

    def align(self, batch):
        """Who said what, when: force-aligns each speaker's reference transcript (text{s}, text{s}_lengths) to the CTC
        head's log-probs, computed in eval mode with the encoder -> fusion -> decoder1 path the training loss sees, one
        forced_align call per speaker.  Returns spans[s][b] = list of TimedTokenSpan, one per target token: frames of
        the fused sequence [start, end), the piece text, and [start_sec, end_sec] in the mixed recording.

        The fused sequence is not wall-clock: the fusion compacts the speaker's speech frames and resamples them to T_v.
        Fused frame f maps to speech-frame rank nearest_src_index(T_v, Tp)[f] (Tp = the batch's largest speech-frame
        count), that rank to its encoder frame k, and k to k * hop_seconds; a span covers [sec(k_start),
        sec(k_{end-1}) + hop_seconds].  Raises (forced_align) if a transcript is too long for its input length."""
        for m in (self.visual_encoder, self.audio_encoder, self.fusion_module, self.decoder1):
            m.eval()
        blank = self.tokenizer.blank_id
        res = []
        with torch.no_grad():
            if hasattr(self.audio_encoder, "begin_step"):
                self.audio_encoder.begin_step()
            d = self._to_dev(batch)
            with torch.autocast("cuda", dtype=self.autocast_dtype, enabled=str(self.device).startswith("cuda")):
                for s in range(2):
                    vis = self.visual_encoder(d["lips"][s]())
                    aud, _ = self.audio_encoder(d["audio"], attention_mask=(d["masks"][s] != 3))
                    t_enc = aud.shape[1]
                    mask_ds = F.interpolate(d["masks"][s].unsqueeze(1).float(), size=t_enc, mode="nearest").squeeze(1).long()
                    fused, il = self.fusion_module(vis, aud, mask_ds)
                    lp = self.decoder1(fused)
                    paths, scores = forced_align(lp, d["texts"][s], il, d["lens"][s], blank=blank)
                    res.append((merge_tokens_batch(paths, scores, il, blank=blank),
                                fused_frame_encoder_index(mask_ds.cpu(), lp.shape[1])))
        out = []
        for spans, enc in res:
            spk = []
            for b, row in enumerate(spans):
                k = enc[b].tolist()
                spk.append([TimedTokenSpan(token=sp.token, start=sp.start, end=sp.end, score=sp.score,
                                           piece=self._piece(sp.token), start_sec=k[sp.start] * self.hop_seconds,
                                           end_sec=k[sp.end - 1] * self.hop_seconds + self.hop_seconds)
                            for sp in row])
            out.append(spk)
        return out

    # ------------------------------------------------------------------------------------------ transcription
    def transcribe(self, batch, beam_width=None, nbest=1, lm=None, lm_weight=0.5, token_bonus=0.0, context=None):
        """What each speaker said: a CTC prefix beam search over the CTC head's log-probs, computed in eval mode with the
        encoder -> fusion -> decoder1 path that align() uses, decoded on the fusion's input lengths.  The batch needs no
        transcripts.  beam_width defaults to self.beam_width (at most 15).  Returns out[s][b] = [(text, score), ...],
        best first, up to nbest per utterance; score is the hypothesis' natural-log probability, or with `lm` (an
        NgramLM over this tokenizer's pieces) the fused score acoustic + lm_weight * ln P_LM + token_bonus * length.
        `context` biases both speakers' searches towards a phrase list: a ContextGraph, or phrase strings encoded with
        self.tokenizer at the default weight; the score then includes each hypothesis' bias."""
        if context is not None and not isinstance(context, ContextGraph):
            context = ContextGraph.from_text(context, self.tokenizer)
        for m in (self.visual_encoder, self.audio_encoder, self.fusion_module, self.decoder1):
            m.eval()
        bw = self.beam_width if beam_width is None else beam_width
        blank = self.tokenizer.blank_id
        out = []
        with torch.no_grad():
            if hasattr(self.audio_encoder, "begin_step"):
                self.audio_encoder.begin_step()
            d = self._to_dev(batch)
            with torch.autocast("cuda", dtype=self.autocast_dtype, enabled=str(self.device).startswith("cuda")):
                for s in range(2):
                    vis = self.visual_encoder(d["lips"][s]())
                    aud, _ = self.audio_encoder(d["audio"], attention_mask=(d["masks"][s] != 3))
                    t_enc = aud.shape[1]
                    mask_ds = F.interpolate(d["masks"][s].unsqueeze(1).float(), size=t_enc, mode="nearest").squeeze(1).long()
                    fused, il = self.fusion_module(vis, aud, mask_ds)
                    lp = self.decoder1(fused)
                    hyps = ctc_prefix_beam_search(lp, il, beam_width=bw, nbest=nbest, blank=blank, lm=lm,
                                                  lm_weight=lm_weight, token_bonus=token_bonus, context=context)
                    out.append([[(fast_decode(h.tokens, self.tokenizer), h.score) for h in row] for row in hyps])
        return out

    def _piece(self, token):
        tok = self.tokenizer
        if hasattr(tok, "id_to_piece"):
            return tok.id_to_piece(token)
        if hasattr(tok, "id_to_token"):
            return tok.id_to_token[token]
        return tok.decode([token])
