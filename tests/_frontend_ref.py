"""Reference front end, deployment call and detector loop for any analysis frame (fft_size, hop_size), composed from
the oracle's pieces (om.frame, om.mel_forward, ost.vad_pcm16 / SimpleQueue, the CTC decoder).  At 400/160 every
function here computes what the oracle's own pcm_to_mel / deploy_forward / StreamOracle / stream_vs_offline do."""
import numpy as np

from oracle import model as om
from oracle import prediction as op
from oracle import streaming as ost

# frames models are commonly trained with, and 400/160 (the default) as the control
CONFIGS = [(512, 160), (480, 160), (320, 160), (256, 128), (200, 80), (512, 256), (400, 200), (500, 125), (512, 512)]
CONTROL = (400, 160)
ALL = CONFIGS + [CONTROL]


def cfg_id(c):
    return "%d_%d" % c


def mel_basis(fft, n_mel):
    """librosa.filters.mel(16000, fft, n_mel, 300, 8000).T: [fft/2 + 1, n_mel] float32."""
    return np.ascontiguousarray(om.slaney_mel_basis(n_fft=fft, n_mels=n_mel).T.astype(np.float32))


def weights(fft, n_mel=40, seed=1234, fc_gain=1.0):
    """The oracle's random model with the mel basis of an fft-point frame."""
    ow = om.init_weights(seed=seed, n_mel=n_mel)
    ow.mel_basis = mel_basis(fft, n_mel)
    ow.fc_w = (ow.fc_w * fc_gain).astype(np.float32)
    return ow


def linearspec(frames, fft, dtype=np.float32):
    """abs(rfft(frames, [fft])) -> [S, n, fft/2 + 1]."""
    return np.abs(np.fft.rfft(frames.astype(dtype), n=fft, axis=-1)).astype(dtype)


def pcm_to_mel(pcm, basis, fft, hop, dtype=np.float32):
    """PCM [S, L] (float, already scaled) -> mel [S, n, M] with a rectangular fft-sample frame every hop samples."""
    frames = om.frame(np.asarray(pcm), fft, hop)
    return np.matmul(linearspec(frames, fft, dtype), basis.astype(dtype)).astype(dtype)


def deploy_forward(pcm, state, w, fft, hop, dtype=np.float32):
    pcm = np.asarray(pcm)
    if pcm.ndim == 1:
        pcm = pcm[None, :]
    return om.mel_forward(pcm_to_mel(pcm.astype(dtype), w.mel_basis, fft, hop, dtype), state, w, None, dtype)


class StreamRef(ost.StreamOracle):
    """ost.StreamOracle with the model's frame: the carried tail is (len - fft) % hop + fft - hop samples."""

    def __init__(self, weights, n_streams, fft, hop, **kw):
        super().__init__(weights, n_streams, **kw)
        self.fft, self.hop = fft, hop

    def step(self, chunk_i16, decide_on=None):
        chunk_i16 = np.asarray(chunk_i16, dtype=np.int16)
        data = om.pcm16_to_float(chunk_i16)
        speech = ost.vad_pcm16(chunk_i16, self.vad_thres)
        for s in np.nonzero(~speech)[0]:
            self.state[:, s, :] = 0
            self.queues[s].clear()
        full = np.concatenate([self.res, data], axis=1)
        keep = ost.residual_length(full.shape[1], self.fft, self.hop)
        self.res = full[:, full.shape[1] - keep:]
        softmax, state, _ = deploy_forward(full, self.state, self.w, self.fft, self.hop, self.dtype)
        self.state = state
        trigger = np.zeros(self.S, dtype=np.int32)
        labels = []
        for s in range(self.S):
            q = self.queues[s]
            q.add(softmax[s])
            seq = op.ctc_decode2(np.concatenate(q.get_all(), axis=0), self.w.num_classes, self.decode_thres)
            labels.append(seq)
            if op.ctc_predict(seq, self.label):
                trigger[s] = 1
                q.clear()
                self.state[:, s, :] = 0
        return dict(speech=speech, softmax=softmax, trigger=trigger, labels=labels, state=self.state.copy())


def stream_vs_offline(pcm_f32, w, fft, hop, seg_len=3600, dtype=np.float32):
    """ost.stream_vs_offline with the model's frame: one utterance fed in seg_len pieces with carried tail and state."""
    pcm_f32 = np.asarray(pcm_f32, dtype=np.float32)
    state = np.zeros((w.num_layers, 1, w.hidden), dtype=dtype)
    res = np.zeros(0, dtype=np.float32)
    outs = []
    seg_num = len(pcm_f32) // seg_len
    for i in range(seg_num + 1):
        feed = pcm_f32[i * seg_len:] if i == seg_num else pcm_f32[i * seg_len:(i + 1) * seg_len]
        data = np.concatenate([res, feed])
        if len(data) < fft:
            res = data
            continue
        res = data[len(data) - ost.residual_length(len(data), fft, hop):]
        used = len(data) - (len(data) - fft) % hop
        sm, state, _ = deploy_forward(data[:used], state, w, fft, hop, dtype)
        outs.append(sm[0])
    return np.concatenate(outs, axis=0), state


def tail_capacity(fft):
    """Carried-tail samples a stream object keeps per stream: max(400, fft rounded up to 8)."""
    return max(400, (fft + 7) // 8 * 8)


def record_bytes(fft, layers=2, W=15, max_chunk=4800, hop=160):
    """Bytes of one per-stream record (include/kws_b200.h)."""
    mf = max(0, 1 + (max_chunk + fft - 1 - fft) // hop)
    fpad = max(16, (mf + 15) // 16 * 16)
    return 48 + 512 * layers + 2 * tail_capacity(fft) + (W + 15) // 16 * 16 + W * fpad
