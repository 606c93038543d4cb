"""Teacher driver with the flags of the reference's teacher.py (teacher.py:14-33): the generator entry points
``--test-fast`` (one teacher-forced pass + parallel sampling, teacher.py:117-138) and ``--test-slow`` (sample-by-sample
generation, teacher.py:140-170) on the CUDA hot path.

Differences, all host-side: audio comes from ``--data``: an NSynth TFRecord (read without TensorFlow), a directory of
.wav files, or synthetic waves; results are written as .wav (no matplotlib windows); ``--test-slow`` runs the dilation-queue kernel
(one call, O(T)) and, with ``--check-naive N``, also the reference's literal loop (one full decoder pass per sample,
teacher.py:153-170) on the first N samples with the same noise to show that both produce the same audio.
``--train`` is not offered: teacher training (model.py:242-248) is outside the hot path of this build."""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DILATIONS = [1, 2, 4, 8, 16, 32, 64, 128, 256, 512] * 3          # teacher.py:55-57


def build_parser():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument('--teacher', type=str, default='teachers/%d' % int(time.time() * 1000), help='Directory where checkpoint and summary is stored')
    p.add_argument('--student', type=str, default='students/%d' % int(time.time() * 1000), help='Directory where checkpoint and summary is stored')
    p.add_argument('--start', type=int, default=0, help='Starting index')
    p.add_argument('--train', action='store_true', help='Train teacher (not part of this build)')
    p.add_argument('--test-fast', action='store_true', help='Test teacher (fast generation)')
    p.add_argument('--test-slow', action='store_true', help='Test teacher (slow generation)')
    p.add_argument('--latent-channels', type=int, default=32, help='Number of latent channel per time slice')
    p.add_argument('--pool-stride', type=int, default=128, help='Number of samples to use per time slice')
    p.add_argument('--batch-size', type=int, default=4, help='Batch size')
    # additions (the reference hard-codes these: teacher.py:42-47)
    p.add_argument('--num-samples', type=int, default=4096)
    p.add_argument('--sample-rate', type=int, default=4000)
    p.add_argument('--data', type=str, default='synthetic', help='"synthetic", an NSynth .tfrecord file (nsynth.py) or a directory of .wav files')
    p.add_argument('--audio-max-length', type=int, default=16000, help='length of the audio feature in the TFRecord (nsynth.py:6)')
    p.add_argument('--out-dir', type=str, default='.')
    p.add_argument('--clips', type=int, default=None, help='number of clips (default: 10 for --test-fast, 1 for --test-slow)')
    p.add_argument('--precision', type=str, default='fp16', choices=['fp32', 'fp16'])
    p.add_argument('--check-naive', type=int, default=0, help='--test-slow: also run the per-sample loop on the first N samples')
    p.add_argument('--prime', type=int, default=0,
                   help='--test-slow: the first N samples of each clip are the clip itself (N a multiple of --pool-stride); '
                        'generation continues from there')
    p.add_argument('--chunk', type=int, default=0,
                   help='--test-slow: generate in calls of S samples (a multiple of --pool-stride) through one state')
    p.add_argument('--prefill', action='store_true',
                   help='--test-slow --prime N: prime the state in one parallel pass instead of step by step (same audio)')
    return p


def generate_chunked(teacher, encoding, u1, u2, precision, prefix, chunk, pool_stride):
    """--test-slow in calls of `chunk` samples through one generation state: the same audio as one call."""
    B, T = u1.shape[0], u1.shape[1]
    state = teacher.generation_state(B, precision)
    n = 0 if prefix is None else prefix.shape[1]
    parts = []
    for a in range(0, T, chunk):
        b = min(a + chunk, T)
        parts.append(teacher.generate(encoding[:, a // pool_stride:b // pool_stride], u1=u1[:, a:b], u2=u2[:, a:b],
                                      precision=precision, zero_last=b == T, state=state,
                                      prefix=prefix[:, a:min(b, n)] if a < n else None))
    return np.concatenate(parts, axis=1)


def generate_prefilled(teacher, encoding, u1, u2, precision, prefix, chunk, pool_stride):
    """--test-slow --prime N --prefill: prime a state with the N samples in one parallel pass, then generate the rest
    from it (in calls of `chunk` samples if given).  The same audio as priming step by step."""
    B, T, n = u1.shape[0], u1.shape[1], prefix.shape[1]
    state = teacher.generation_state(B, precision)
    teacher.prefill(state, prefix, encoding[:, :n // pool_stride])
    parts = [np.asarray(prefix, dtype=np.float32)]
    step = chunk or T - n
    for a in range(n, T, step):
        b = min(a + step, T)
        parts.append(teacher.generate(encoding[:, a // pool_stride:b // pool_stride], u1=u1[:, a:b], u2=u2[:, a:b],
                                      precision=precision, zero_last=b == T, state=state))
    out = np.concatenate(parts, axis=1)
    if n == T:
        out[:, T - 1:] = 0                                      # teacher.py:170, as the one-call path does
    return out


def main(argv=None):
    args = build_parser().parse_args(argv)
    import sr_wavenet_b200 as srwn
    from sr_wavenet_b200 import synth
    from sr_wavenet_b200.audio_data import AudioReader, write_wav

    if args.train:
        raise SystemExit("teacher training (model.py:242-248) is outside the hot path of this build")
    num_samples, batch = args.num_samples, args.batch_size
    for flag, v in (('--prime', args.prime), ('--chunk', args.chunk)):
        if v < 0 or v % args.pool_stride or v > num_samples:
            raise SystemExit('%s %d must be a multiple of --pool-stride %d and at most --num-samples %d'
                             % (flag, v, args.pool_stride, num_samples))
    audio_data = AudioReader(args.data, batch, num_samples, audio_max_length=args.audio_max_length)
    teacher = srwn.WaveNetAutoEncoder(input_size=num_samples, condition_size=0, num_mixtures=5, dilations=DILATIONS,
                                      latent_channels=args.latent_channels, skip_channels=128,
                                      pool_stride=args.pool_stride, learning_rate=1e-4)
    teacher.load(args.teacher)
    os.makedirs(args.out_dir, exist_ok=True)
    results = {}

    if args.test_fast:                                          # teacher.py:117-138
        t0, n = time.time(), 0
        for step in range(args.clips or 10):
            x, _ = audio_data.next()
            regen = teacher.reconstruct(x, None, precision=args.precision)
            write_wav(os.path.join(args.out_dir, 'test_wav_%d.wav' % step), args.sample_rate, x[0])
            write_wav(os.path.join(args.out_dir, 'regen_wav_%d.wav' % step), args.sample_rate, regen[0])
            n += x.size
        results['test_fast_samples_per_s'] = n / (time.time() - t0)
        print('test-fast: %d samples, %.3g samples/s (host time, includes wav output)' % (n, results['test_fast_samples_per_s']))

    if args.test_slow:                                          # teacher.py:140-170
        for count in range(args.clips or 1):
            x, _ = audio_data.next()
            write_wav(os.path.join(args.out_dir, 'test_wav_%d.wav' % count), args.sample_rate, x[0])
            encoding = teacher.encode(x, None, precision=args.precision)
            u1, u2 = synth.sampler_uniforms(x.shape[0], num_samples, 5, seed=999 + count)
            ar_prec = 'fp32' if args.precision == 'fp32' else 'fp16'    # the queue kernel keeps fp16 state on the 16-bit path
            prefix = x[:, :args.prime] if args.prime else None
            t0 = time.time()
            if args.prefill and args.prime:
                regen = generate_prefilled(teacher, encoding, u1, u2, ar_prec, prefix, args.chunk, args.pool_stride)
            elif args.chunk:
                regen = generate_chunked(teacher, encoding, u1, u2, ar_prec, prefix, args.chunk, args.pool_stride)
            else:
                regen = teacher.generate(encoding, u1=u1, u2=u2, precision=ar_prec, zero_last=True, prefix=prefix)
            dt = time.time() - t0
            results['test_slow_samples_per_s'] = regen.size / dt
            print('test-slow: %d x %d samples in %.3f s (%.3g samples/s)' % (regen.shape[0], regen.shape[1], dt, regen.size / dt))
            if args.check_naive:
                n = min(args.check_naive, num_samples)
                x_so_far = np.zeros((x.shape[0], num_samples), dtype=np.float32)
                x_so_far[:, :args.prime] = x[:, :args.prime]    # primed: those samples are kept, not drawn
                for i in range(min(args.prime, n), n):          # the reference's loop, verbatim semantics
                    x_so_far[:, i:] = 0
                    x_so_far[:, i] = teacher.reconstruct_with_encoding(x_so_far, encoding, u1=u1, u2=u2,
                                                                       precision=args.precision)[:, i]
                diff = float(np.abs(x_so_far[:, :n] - regen[:, :n]).max())
                results['naive_max_abs_diff'] = diff
                print('naive loop vs queue kernel on the first %d samples: max |diff| = %.3g' % (n, diff))
            write_wav(os.path.join(args.out_dir, 'regen_wav_%d.wav' % count), args.sample_rate, regen[0])
    return results


if __name__ == '__main__':
    main()
