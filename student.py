"""Student driver with the flags of the reference's student.py (student.py:14-36): ``--train`` runs distillation steps
(student.py:89-160: encode -> logistic noise -> train_fast; every print_steps the entropy, a synthesis and a
reconstruction) and ``--test`` the synthesis entry point (student.py:163-197), on the CUDA hot path.

Host-side differences: audio comes from ``--data``: an NSynth TFRecord (read without TensorFlow), a directory of .wav
files, or synthetic waves; results are written as .wav (no matplotlib windows); ``--steps`` bounds the training loop (the reference's
literal is 1000000).  ``--teacher`` is a checkpoint directory written by teacher.py / WaveNetAutoEncoder.save; without
one a randomly initialised teacher is used and the driver says so."""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DILATIONS = [1, 2, 4, 8, 16, 32, 64, 128, 256, 512] * 3          # student.py:57-59


def build_parser():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument('--teacher', type=str, default=None, help='Directory where checkpoint and summary is stored')
    p.add_argument('--student', type=str, default='students/%d' % int(time.time() * 1000), help='Directory where checkpoint and summary is stored')
    p.add_argument('--start', type=int, default=0, help='Starting index')
    p.add_argument('--train', action='store_true', help='Train student')
    p.add_argument('--test', action='store_true', help='Test student')
    p.add_argument('--latent-channels', type=int, default=32, help='Number of latent channel per time slice')
    p.add_argument('--pool-stride', type=int, default=128, help='Number of samples to use per time slice')
    p.add_argument('--batch-size', type=int, default=4, help='Batch size')
    p.add_argument('--entropy-weight', type=float, default=0.25, help='Weight of entropy term in loss function')
    p.add_argument('--cross-entropy-weight', type=float, default=1.0, help='Weight of cross entropy term in loss function')
    p.add_argument('--power-weight', type=float, default=1.0, help='Weight of power loss term in loss function')
    p.add_argument('--learning-rate', type=float, default=1e-4, help='Learning rate')
    # additions (the reference hard-codes these: student.py:42-50)
    p.add_argument('--num-samples', type=int, default=4096)
    p.add_argument('--sample-rate', type=int, default=4000)
    p.add_argument('--steps', type=int, default=1000000, help='last training step (exclusive)')
    p.add_argument('--print-steps', type=int, default=25)
    p.add_argument('--data', type=str, default='synthetic', help='"synthetic", an NSynth .tfrecord file (nsynth.py) or a directory of .wav files')
    p.add_argument('--audio-max-length', type=int, default=16000, help='length of the audio feature in the TFRecord (nsynth.py:6)')
    p.add_argument('--out-dir', type=str, default='.')
    p.add_argument('--clips', type=int, default=20, help='--test: number of clips')
    p.add_argument('--precision', type=str, default='fp16', choices=['fp32', 'fp16'])
    p.add_argument('--seed', type=int, default=None, help='seed of the host-side logistic noise (student.py:104 leaves it unseeded)')
    p.add_argument('--chunk', type=int, default=0,
                   help='--test: synthesize each clip in calls of S samples (a multiple of --pool-stride) through one '
                        'synthesis state; the same audio as one call')
    return p


def generate_chunked(student, noise, encoding, precision, chunk, pool_stride):
    """--test --chunk: the clip in calls of `chunk` samples through one synthesis state: the same audio as one call."""
    B, T = noise.shape
    state = student.synthesis_state(B, precision)
    parts = [student.generate(None, noise[:, a:a + chunk], encoding[:, a // pool_stride:(a + chunk) // pool_stride], None,
                              state=state) for a in range(0, T, chunk)]
    return np.concatenate(parts, axis=1)


def main(argv=None):
    args = build_parser().parse_args(argv)
    import sr_wavenet_b200 as srwn
    from sr_wavenet_b200.audio_data import AudioReader, write_wav

    num_samples, batch = args.num_samples, args.batch_size
    if args.chunk < 0 or args.chunk % args.pool_stride:
        raise SystemExit('--chunk %d must be a multiple of --pool-stride %d' % (args.chunk, args.pool_stride))
    audio_data = AudioReader(args.data, batch, num_samples, audio_max_length=args.audio_max_length)
    teacher = args.teacher
    if teacher is None or not os.path.exists(os.path.join(teacher, 'checkpoint')):
        print('no teacher checkpoint under %r: using a randomly initialised teacher' % (teacher,))
        teacher = srwn.WaveNetAutoEncoder(input_size=num_samples, condition_size=0, num_mixtures=5, dilations=DILATIONS,
                                          latent_channels=args.latent_channels, skip_channels=128,
                                          pool_stride=args.pool_stride)
    student = srwn.ParallelWaveNet(input_size=num_samples, condition_size=0, dilations=DILATIONS, teacher=teacher,
                                   dilation_channels=32, skip_channels=128, num_flows=4,
                                   latent_channels=args.latent_channels, pool_stride=args.pool_stride,
                                   alpha=args.entropy_weight, beta=args.cross_entropy_weight, gamma=args.power_weight,
                                   learning_rate=args.learning_rate)
    print('initailized')
    student.load(None, args.student)
    print('loaded')
    rng = np.random.default_rng(args.seed)
    os.makedirs(args.out_dir, exist_ok=True)
    results = {'losses': []}

    if args.train:                                              # student.py:89-160
        global_step = args.start
        for global_step in range(args.start, args.steps):
            x, _ = audio_data.next()
            encoding = student.encode(None, x, None, precision=args.precision)
            noise = rng.logistic(0, 1, [batch, num_samples]).astype(np.float32)
            loss, power_loss = student.train_fast(None, noise, x, encoding, None)
            results['losses'].append(loss)
            if global_step % args.print_steps == 0:
                entropy = student.getEntropy_fast(None, noise, encoding, None)
                print('Step: {:6d} | Entropy: {} | Power Loss: {:.4f} | Total Loss: {:.4f}'.format(global_step, str(entropy), power_loss, loss))
                output = student.generate(None, noise, encoding, None, precision=args.precision)
                regen = student.reconstruct(None, x, None, precision=args.precision)
                write_wav(os.path.join(args.out_dir, 'student_wav_%d.wav' % global_step), args.sample_rate, output[0, :, 0])
                write_wav(os.path.join(args.out_dir, 'regen_wav_%d.wav' % global_step), args.sample_rate, regen[0])
            student.save(None, args.student, global_step, force=False)     # checkpoint once per minute
        student.save(None, args.student, global_step, force=True)

    if args.test:                                               # student.py:163-197
        for step in range(args.clips):
            x, _ = audio_data.next()
            encoding = student.encode(None, x, None, precision=args.precision)
            regen = student.reconstruct(None, x, None, precision=args.precision)
            noise = rng.logistic(0, 1, x.shape).astype(np.float32)
            entropy = student.getEntropy(None, noise, encoding, None)
            if args.chunk:
                output = generate_chunked(student, noise, encoding, args.precision, args.chunk, args.pool_stride)
            else:
                output = student.generate(None, noise, encoding, None, precision=args.precision)
            print('Entropy', entropy)
            write_wav(os.path.join(args.out_dir, 'test_wav_%d.wav' % step), args.sample_rate, x[0])
            write_wav(os.path.join(args.out_dir, 'regen_wav_%d.wav' % step), args.sample_rate, regen[0])
            write_wav(os.path.join(args.out_dir, 'student_wav_%d.wav' % step), args.sample_rate, output[0, :, 0])
            results['output_shape'] = tuple(output.shape)
    return results


if __name__ == '__main__':
    main()
