"""Llama with an audio prefix — drop-in for modelling/audio.py of the reference.

Front-end: mel-spectrogram -> log10 -> cepstral mean normalisation stay PyTorch (torchaudio FFT); the Whisper-style
stem Conv1d(k3,s1)+GELU -> Conv1d(k3,s2)+GELU (audio.py:26-31,51-60) runs on this package's kernels on CUDA/bf16
(`AudioStemFn`: convolutions as tcgen05 GEMMs over overlapping-row views of the padded channels-last activations, fused
bias+GELU passes, col2im for the stride-2 input gradient), with `nn.Sequential` kept as the parameter container so
reference state_dicts load unchanged. The decoder blocks behind it run on the fused sm_100a path.

Extension over the reference: `LlamaAudio.forward(..., prefix_lm=True)` makes the audio positions a bidirectional
prefix (mask(q, kv) = (kv < P) | (q >= kv), P = number of audio positions) — the prefix-LM objective the
reference's README plans (README.md:16) but runs as plain causal attention (audio.py:65-70). The default
(`prefix_lm=False`) keeps the reference behaviour.
"""

from typing import NamedTuple

import torch
from torch import Tensor, nn

from .. import ops
from .llama import Llama, LlamaConfig, PrefixLM

# False: the stem runs through nn.Conv1d / nn.GELU (cuDNN), the tests' reference for AudioStemFn
_OWN_STEM = True



class AudioStemFn(torch.autograd.Function):
    """prefix [B, T/2, C] = GELU(Conv1d_k3s2(GELU(Conv1d_k3s1(mel)))) for mel [B, Cin, T] (T even), channels-last inside.

    A k = 3 convolution over a channels-last slab padded by one zero row on each side reads, for output row t, the 3*C
    CONSECUTIVE elements that start at padded row stride*t: the im2col matrix is a view with overlapping rows
    (row pitch stride*C, row length 3*C), which the GEMM's TMA descriptor walks directly. Batch slabs are laid back to
    back, so one GEMM covers the batch; the one or two rows per slab that straddle a boundary are padding rows and are
    zeroed by the bias+GELU pass that follows.
    """

    @staticmethod
    def forward(ctx, mel: Tensor, w1: Tensor, b1: Tensor, w2: Tensor, b2: Tensor):
        B, Cin, T = mel.shape
        C = w1.shape[0]
        assert T % 2 == 0 and Cin % 8 == 0 and C % 8 == 0 and w1.shape == (C, Cin, 3) and w2.shape == (C, C, 3)
        Tp, half = T + 2, (T + 2) // 2
        dev = mel.device
        x0p = torch.zeros(B, Tp, Cin, device=dev, dtype=torch.bfloat16)
        x0p[:, 1 : T + 1] = mel.transpose(1, 2)
        # conv 1 (stride 1): rows r = b*Tp + t  ->  output lands at padded row r + 1 of the next layer's input
        M1 = B * Tp - 2
        a1 = x0p.as_strided((M1, 3 * Cin), (Cin, 1))
        w1r = w1.detach().permute(0, 2, 1).reshape(C, 3 * Cin).contiguous()        # [C, j*Cin + c]
        z1 = torch.empty(B * Tp, C, device=dev, dtype=torch.bfloat16)
        ops.bf16_gemm(a1, w1r, out=z1[1 : 1 + M1])
        y1 = ops.gelu_bias_fwd_(z1, b1.detach(), Tp, 1, T + 1)                     # padded input of conv 2
        # conv 2 (stride 2): rows r = b*half + t read padded rows 2t, 2t+1, 2t+2; t = half-1 is a padding row
        M2 = B * half - 1
        a2 = y1.as_strided((M2, 3 * C), (2 * C, 1))
        w2r = w2.detach().permute(0, 2, 1).reshape(C, 3 * C).contiguous()
        z2 = torch.empty(B * half, C, device=dev, dtype=torch.bfloat16)
        ops.bf16_gemm(a2, w2r, out=z2[:M2])
        y2 = ops.gelu_bias_fwd_(z2, b2.detach(), half, 0, half - 1)
        ctx.save_for_backward(x0p, z1, y1, z2, w2r)
        ctx.dims = (B, Cin, T, C)
        return y2.view(B, half, C)[:, : half - 1]

    @staticmethod
    def backward(ctx, dout: Tensor):
        x0p, z1, y1, z2, w2r = ctx.saved_tensors
        B, Cin, T, C = ctx.dims
        Tp, half = T + 2, (T + 2) // 2
        M1, M2 = B * Tp - 2, B * half - 1
        dev = dout.device
        dy2 = torch.zeros(B, half, C, device=dev, dtype=torch.bfloat16)
        dy2[:, : half - 1] = dout
        dz2 = ops.gelu_bwd(dy2.view(B * half, C), z2, half, 0, half - 1)
        db2 = dz2.sum(0, dtype=torch.float32).to(torch.bfloat16)
        # dW2 [C, 3C] = dz2^T . im2col(y1): contraction over the (batch x time) rows; both operands are consumed as
        # stored (MN-major UMMA operands), the im2col matrix again as the overlapping-row view of y1
        dw2 = ops.bf16_gemm_tn(dz2[:M2], y1.as_strided((M2, 3 * C), (2 * C, 1))).view(C, 3, C).permute(0, 2, 1).contiguous()
        # input gradient of conv 2: column gradient, then overlap-add back onto the padded rows
        dcol = torch.zeros(B * half, 3 * C, device=dev, dtype=torch.bfloat16)
        ops.bf16_gemm(dz2[:M2], w2r.t().contiguous(), out=dcol[:M2])
        dy1p = ops.conv_s2k3_col2im(dcol, B, Tp, C)
        del dcol
        dz1 = ops.gelu_bwd(dy1p.view(B * Tp, C), z1, Tp, 1, T + 1)
        db1 = dz1.sum(0, dtype=torch.float32).to(torch.bfloat16)
        dw1 = ops.bf16_gemm_tn(dz1[1 : 1 + M1], x0p.as_strided((M1, 3 * Cin), (Cin, 1)))
        dw1 = dw1.view(C, 3, Cin).permute(0, 2, 1).contiguous()
        return None, dw1, db1, dw2, db2


class AudioConfig(NamedTuple):
    sample_rate: int = 16_000
    n_fft: int = 512
    win_length: int = 400
    hop_length: int = 160
    n_mels: int = 128


class LlamaAudio(Llama):
    def __init__(self, config: LlamaConfig, audio_config: AudioConfig = AudioConfig()):
        super().__init__(config)
        self.audio_config = audio_config
        # Whisper-style stem: stride-1 conv then stride-2 conv, GELU after each
        self.audio_embed = nn.Sequential(
            nn.Conv1d(audio_config.n_mels, config.embed_dim, 3, 1, 1),
            nn.GELU(),
            nn.Conv1d(config.embed_dim, config.embed_dim, 3, 2, 1),
            nn.GELU(),
        )

    def build_cache(self, inference: bool = False):
        super().build_cache(inference)
        from torchaudio.transforms import MelSpectrogram

        self.melspec = MelSpectrogram(**self.audio_config._asdict(), norm="slaney", mel_scale="slaney")
        self.melspec.to(self.tok_embeddings.weight.device)

    def embed_audio(self, audio: Tensor) -> Tensor:
        """waveform [B, T] -> prefix embeddings [B, P, embed_dim]."""
        mel = self.melspec(audio)[..., :-1].clip(1e-12).log10()  # drop the last frame: even length
        mel = mel - mel.mean(2, keepdim=True)
        mel = mel.to(dtype=self.tok_embeddings.weight.dtype)
        c1, c2 = self.audio_embed[0], self.audio_embed[2]
        if (_OWN_STEM and mel.is_cuda and mel.dtype is torch.bfloat16 and c1.weight.dtype is torch.bfloat16
                and mel.shape[2] % 2 == 0 and mel.shape[1] % 8 == 0):
            if self.config.activation_checkpointing:
                from torch.utils.checkpoint import checkpoint

                return checkpoint(AudioStemFn.apply, mel, c1.weight, c1.bias, c2.weight, c2.bias, use_reentrant=False)
            return AudioStemFn.apply(mel, c1.weight, c1.bias, c2.weight, c2.bias)
        if self.config.activation_checkpointing:
            from torch.utils.checkpoint import checkpoint

            emb = checkpoint(self.audio_embed, mel, use_reentrant=False)
        else:
            emb = self.audio_embed(mel)
        return emb.transpose(1, 2)

    def forward(self, audio: Tensor | None, tokens: Tensor, *, input_pos: Tensor | None = None,
                labels: Tensor | None = None, prefix_lm: bool | Tensor = False) -> Tensor:
        """prefix_lm: False (reference behaviour: causal over [audio ; text]), True (the audio positions are a bidirectional
        prefix), or an int tensor [B] of per-sequence prefix lengths (utterances shorter than the padded audio: only
        their own frames are bidirectional)."""
        if input_pos is not None:
            raise NotImplementedError("llamax_b200: input_pos (inference) is outside the fine-tuning hot path")
        label_count = self._count_labels(labels)
        x = self.tok_embeddings(tokens)
        n_prefix = 0
        if audio is not None:
            prefix = self.embed_audio(audio)
            n_prefix = prefix.shape[1]
            x = torch.cat([prefix, x], dim=1)
        if isinstance(prefix_lm, Tensor):
            block_mask = PrefixLM(prefix_lm.clamp(max=n_prefix))
        else:
            block_mask = PrefixLM(n_prefix) if (prefix_lm and n_prefix > 0) else None
        x = self._run_layers(x, block_mask)
        if n_prefix:
            x = x[:, n_prefix:]  # loss / logits on text positions only
        return self._head(x, labels, label_count)
