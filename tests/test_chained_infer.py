"""Chained low-res -> super-res inference (lvg_infer/chained.py) against the reference's schedule
(generate.py:56-88, generator_sres.py:662-681), with stand-in generators: the host logic on CPU; on cuda under -m gpu
the CUDA-graph capture / replay of the super-res batches and the pinned-host copies on the side stream."""
import pytest
import torch

from lvg_infer.chained import generate_video, segment_windows, to_uint8


class _Lres(torch.nn.Module):
    def forward(self, batch, seq_length, generator_emb=None):
        return torch.randn(batch, 3, seq_length, 6, 8, generator=generator_emb, device=generator_emb.device).tanh()


class _Sres(torch.nn.Module):
    """Per-sample, per-window function with the call surface of the reference's super-res generator."""
    temporal_context = 2

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.randn(3, 3))

    def sample_latent_z(self, batch, generator=None):
        return torch.randn(batch, 5, generator=generator, device=generator.device)

    def SG3(self, z, lr):
        c = self.temporal_context
        mid = lr[:, :, c:-c] + 0.25 * lr[:, :, :-2 * c] - 0.5 * lr[:, :, 2 * c:]            # uses the context frames
        y = torch.einsum('oc,nctHW->notHW', self.w, mid) * z[:, :1, None, None, None].tanh()
        return torch.nn.functional.interpolate(y, scale_factor=(1, 2, 2), mode='nearest')

    def sample_video_segments(self, lr_video, segment_length, generator_z=None):        # generator_sres.py:662-681
        z = self.sample_latent_z(lr_video.size(0), generator_z)
        for win in segment_windows(lr_video, segment_length, self.temporal_context):
            yield self.SG3(z, win)


@pytest.mark.parametrize('seq_length,seg,k', [(40, 8, 3), (64, 16, 8), (7, 4, 1), (48, 8, 2)])
def test_same_frames_as_the_reference_schedule(seq_length, seg, k):
    lres, sres = _Lres(), _Sres()
    # the reference's schedule (generate.py:56-68)
    gen = torch.Generator().manual_seed(5)
    lr_len = -(-seq_length // seg) * seg + 2 * sres.temporal_context
    lr_ref = lres(1, lr_len, generator_emb=gen)
    ref = torch.cat(list(sres.sample_video_segments(lr_ref, seg, generator_z=gen)), dim=2)[:, :, :seq_length]
    # ours
    gen = torch.Generator().manual_seed(5)
    lr, chunks = generate_video(lres, sres, seq_length, generator=gen, segment_length=seg, segments_per_batch=k, as_uint8=False)
    got = torch.empty(3, seq_length, *ref.shape[-2:])
    seen = 0
    for first, frames in chunks:
        assert first == seen and frames.shape[0] == 3
        got[:, first:first + frames.shape[1]] = frames                                   # consumed before the next chunk is requested
        seen += frames.shape[1]
    assert seen == seq_length and torch.equal(lr, lr_ref)
    torch.testing.assert_close(got, ref[0], rtol=1e-6, atol=1e-6)


def test_sink_and_uint8():
    lres, sres = _Lres(), _Sres()
    got = []
    lr, it = generate_video(lres, sres, 20, generator=torch.Generator().manual_seed(1), segment_length=4, segments_per_batch=2,
                            sink=lambda first, frames: got.append((first, frames.clone())))
    assert list(it) == [] and [f for f, _ in got] == [0, 8, 16] and got[-1][1].shape[1] == 4
    assert all(fr.dtype == torch.uint8 for _, fr in got)
    x = torch.tensor([-1.0, 0.0, 1.0, 3.0])
    assert to_uint8(x).tolist() == [0, 128, 255, 255]


def test_window_validation():
    with pytest.raises(ValueError):
        segment_windows(torch.zeros(1, 3, 21, 2, 2), 8, 2)


class _SresOps(_Sres):
    """The super-res stand-in with its activation through this repository's bias_act kernel (cuda only)."""

    def __init__(self):
        super().__init__()
        self.b = torch.nn.Parameter(torch.randn(3) * 0.1)

    def SG3(self, z, lr):
        from torch_utils.ops import bias_act
        return bias_act.bias_act(super().SG3(z, lr), self.b, act='lrelu', clamp=256)


@pytest.mark.gpu
def test_reference_generators_chained_on_cuda():
    """generate_video on cuda, eager and graph-captured, against the reference's one-segment-at-a-time schedule."""
    dev = torch.device('cuda')
    torch.manual_seed(0)
    lres, sres = _Lres(), _SresOps().to(dev)
    seq, seg = 88, 16                       # 6 segments (96 frames), cut to 88: the last batch is shorter and runs eagerly
    with torch.no_grad():
        gen = torch.Generator(dev).manual_seed(49)
        lr_len = -(-seq // seg) * seg + 2 * sres.temporal_context
        lr_ref = lres(1, lr_len, generator_emb=gen)
        ref = torch.cat(list(sres.sample_video_segments(lr_ref, seg, generator_z=gen)), dim=2)[0, :, :seq].cpu()
    for graph in (False, True):
        for as_uint8 in (False, True):
            gen = torch.Generator(dev).manual_seed(49)
            lr, chunks = generate_video(lres, sres, seq, generator=gen, segment_length=seg, segments_per_batch=4, as_uint8=as_uint8,
                                        graph=graph)
            got = torch.empty(3, seq, *ref.shape[-2:], dtype=torch.uint8 if as_uint8 else torch.float32)
            seen = 0
            for first, frames in chunks:
                assert first == seen and frames.shape[0] == 3 and frames.device.type == 'cpu'
                got[:, first:first + frames.shape[1]] = frames                           # consumed before the next chunk is requested
                seen += frames.shape[1]
            assert seen == seq and torch.equal(lr, lr_ref), (graph, as_uint8)
            if as_uint8:                    # a last-bit difference of the float frames may round to the neighbouring level
                assert int((got.int() - to_uint8(ref).int()).abs().max()) <= 1, graph
            else:
                torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-5)
