// phase-rotate — the reference's command line tool on top of libphaserot_cuda.
//
// Same options, messages, exit codes and result lines as the reference CLI
// (cli/phase-rotate.cc:489-539 help text, :608-661 option parsing, :663-766
// validation, :815-947 minimum search and report, :950-1003 render loop).  What
// differs is where the audio work happens:
//
//   * analysis: the reference re-reads the file once for a coarse pass and once
//     more per candidate window (cli:784, 871-880).  A per-angle peak is a pure
//     function of (file, channel, angle), so this program asks the GPU for the
//     whole 360-entry table in ONE phaserot_sweep() pass and replays the
//     reference's coarse / refine bookkeeping against that table, including
//     which channels a refine pass would have analysed (cli:880).
//   * render: all full blocks go through one phaserot_render() call; only the
//     short last block and the flush block use the block-wise phaserot_apply(),
//     because the reference feeds stale rendered samples back in there (cli:973).
//
// The write loop keeps the reference's latency trim and its quirks (float
// offset into the interleaved buffer, cli:985; stale tail, cli:973).
// There is no CPU DSP in this file: without a usable GPU it exits with an error.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <getopt.h>
#include <limits>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include <chrono>

#include <sndfile.h>

#include "phaserot_cuda.h"

#ifndef VERSION
#define VERSION "0.5-cuda"
#endif

namespace {

// Angle grid: SUBSAMPLE 2 / MAXSAMPLE 360 in the reference (cli:38-39), i.e. half
// degrees.  `--subsample N` (long option of this backend only) selects 1/N degree
// steps; every place the reference uses the two constants reads these instead.
int kSubsample = 2;
int kMaxSample = 180 * 2;

struct Options {
	const char*  angles_arg = nullptr;
	int          stride     = 0;
	bool         stride_set = false; // default: 12 degrees (cli:597)
	int          verbose    = 0;
	bool         link       = false;
	unsigned int blksiz     = 0;
	const char*  in_path    = nullptr;
	const char*  out_path   = nullptr;
	// opt-in long options of this backend; the reference's own options are unchanged
	int          oversample  = 0;     // --true-peak[=2|4]
	int          subsample   = 2;     // --subsample N: 1/N degree grid (BASELINE configs 3 and 5 use 10 and 100)
	int          gpus        = 1;     // --gpus N: sample-range shards over N devices (0 = all)
	bool         fixed_write = false; // --fixed-write: write loop without the reference's two quirks (cli:985, cli:973)
	double       sections    = 0;     // --sections SECONDS: one angle per section of the file (0 = one for the whole file)
	bool         loudness    = false; // --loudness: BS.1770-4 integrated loudness and PLR of the input and of the output
	bool         overs       = false; // --overs DBFS: samples above the ceiling at the input, the output angle and the best angle
	double       overs_db    = 0;
	int          nth_peak    = 0;     // --nth-peak N: minimise the level of the N-th largest sample instead of the peak (0: off)
};

// PHASEROT_CLI_TIMING=1: wall-clock breakdown of the process on stderr (file read, CUDA
// context + module load inside phaserot_create, analysis, render, write)
struct StageTimer {
	bool                                  on;
	std::chrono::steady_clock::time_point t0, last;
	StageTimer () : on (getenv ("PHASEROT_CLI_TIMING") != nullptr), t0 (std::chrono::steady_clock::now ()), last (t0) {}
	void mark (const char* what)
	{
		if (!on) return;
		const auto now = std::chrono::steady_clock::now ();
		fprintf (stderr, "[timing] %-28s %8.1f ms  (at %8.1f ms)\n", what, std::chrono::duration<double, std::milli> (now - last).count (),
		         std::chrono::duration<double, std::milli> (now - t0).count ());
		last = now;
	}
};

float
to_dB (float coeff) // cli:76-83
{
	if (coeff < 1e-15) {
		return -std::numeric_limits<float>::infinity ();
	}
	return 20.0f * log10f (coeff);
}

std::thread g_cuda_warm; // CUDA context creation, see main()

void
join_cuda_warm ()
{
	if (g_cuda_warm.joinable ()) {
		g_cuda_warm.join ();
	}
}

[[noreturn]] void
die (const char* msg)
{
	join_cuda_warm ();
	fputs (msg, stderr);
	::exit (EXIT_FAILURE);
}

void
print_help ()
{
	// text kept identical to the reference so that help2man output and user
	// scripts do not change (cli/phase-rotate.cc:489-539)
	fputs ("phase-rotate - Audio File Phase Rotation Util.\n\n"
	       "Usage: phase-rotate [ OPTIONS ] <file> [out-file]\n\n"
	       "Options:\n"
	       "  -a, --angle <n>[,<n>]*     specify phase angle to apply\n"
	       "  -f, --fftlen <num>         process-block size, freq. resolution\n"
	       "  -h, --help                 display this help and exit\n"
	       "  -l, --link-channels        use downmixed mono peak for analysis\n"
	       "  -s, --stride <num>         analysis step-size\n"
	       "  -v, --verbose              show processing information\n"
	       "  -V, --version              print version information and exit\n"
	       "\n"
	       "\n"
	       "This utility analyzes the given audio file to find a phase-rotation\n"
	       "angle that results in minimal digital-peak, while retaining overall\n"
	       "sound and loudness.\n"
	       "\n"
	       "If both input and output file are given, the analysis results applied, and\n"
	       "a new file with optimized phase is written. Otherwise the analysis results\n"
	       "are only printed to standard output.\n"
	       "\n"
	       "Analysis is performed in two steps, first a coarse analysis is performed,\n"
	       "calculating peak for angles distanced `stride' degrees apart. Then local\n"
	       "minimums are explored in a second step.\n"
	       "\n"
	       "Verbose analysis allows to plot the digital peak vs phase-rotation.\n"
	       "The output is in gnuplot(1) data file format.\n"
	       "\n"
	       "If the -a option is specified, no analysis is performed but the given,\n"
	       "phase-angle(s) are directly applied. This requires both input and output\n"
	       "files to be given. If a single angle is given it is applied to all channels\n"
	       "of the file. Otherwise one has to specify the same number of phase-angles as\n"
	       "there are channels in the file.\n"
	       "\n"
	       "\n"
	       "Examples:\n"
	       "phase-rotate -l my-music.wav out-file.wav\n\n"
	       "phase-rotate -vv -s 3 my-music.wav\n\n"
	       "phase-rotate -a 10,20 in.wav out.wav\n\n"
	       "Report bugs to <https://github.com/x42/phaserotate.lv2/issues>\n"
	       "Website: <https://github.com/x42/phaserotate.lv2/>\n",
	       stdout);
	::exit (EXIT_SUCCESS);
}

Options
parse_options (int argc, char** argv)
{
	Options o;
	static const struct option longopts[] = {
		{ "angle", required_argument, 0, 'a' },
		{ "fftlen", required_argument, 0, 'f' },
		{ "stride", required_argument, 0, 's' },
		{ "help", no_argument, 0, 'h' },
		{ "link-channels", no_argument, 0, 'l' },
		{ "version", no_argument, 0, 'V' },
		{ "verbose", no_argument, 0, 'v' },
		{ "true-peak", optional_argument, 0, 1000 }, // new, long-only: the reference's options are unchanged
		{ "subsample", required_argument, 0, 1001 },
		{ "gpus", required_argument, 0, 1002 },
		{ "fixed-write", no_argument, 0, 1003 },
		{ "sections", required_argument, 0, 1004 },
		{ "loudness", no_argument, 0, 1005 },
		{ "overs", required_argument, 0, 1006 },
		{ "nth-peak", required_argument, 0, 1007 },
		{ 0, 0, 0, 0 },
	};
	int c;
	while ((c = getopt_long (argc, argv, "a:f:hls:Vv", longopts, nullptr)) != EOF) {
		switch (c) {
			case 'a': o.angles_arg = optarg; break;
			case 'f': o.blksiz = (unsigned int)atoi (optarg); break;
			case 'h': print_help (); break;
			case 'l': o.link = true; break;
			case 's':
				o.stride     = atoi (optarg);
				o.stride_set = true;
				break;
			case 'V':
				printf ("phase-rotate version %s\n\n", VERSION);
				printf ("Copyright (C) GPL 2021 Robin Gareus <robin@gareus.org>\n");
				::exit (EXIT_SUCCESS);
			case 'v': ++o.verbose; break;
			case 1000:
				o.oversample = optarg ? atoi (optarg) : 4;
				if (o.oversample != 2 && o.oversample != 4) {
					die ("Error: --true-peak takes an oversampling factor of 2 or 4.\n");
				}
				break;
			case 1001:
				o.subsample = atoi (optarg);
				if (o.subsample < 1 || o.subsample > 1000) {
					die ("Error: --subsample takes a grid density of 1 .. 1000 steps per degree.\n");
				}
				break;
			case 1002:
				o.gpus = atoi (optarg);
				if (o.gpus < 0 || o.gpus > 16) {
					die ("Error: --gpus takes a device count of 0 (all) .. 16.\n");
				}
				break;
			case 1003: o.fixed_write = true; break;
			case 1004: {
				char* ep    = nullptr;
				o.sections = strtod (optarg, &ep);
				if (*ep != '\0' || !(o.sections > 0) || !std::isfinite (o.sections)) {
					die ("Error: --sections takes a section length in seconds > 0.\n");
				}
				break;
			}
			case 1005: o.loudness = true; break;
			case 1006: {
				char* ep   = nullptr;
				o.overs    = true;
				o.overs_db = strtod (optarg, &ep);
				if (*ep != '\0' || ep == optarg || !std::isfinite (o.overs_db) || o.overs_db < -60 || o.overs_db > 20) {
					die ("Error: --overs takes a ceiling in dBFS from -60 to 20.\n");
				}
				break;
			}
			case 1007: {
				char*      ep = nullptr;
				const long n  = strtol (optarg, &ep, 10);
				if (*ep != '\0' || ep == optarg || n < 1 || n > 256) {
					die ("Error: --nth-peak takes a rank of 1 .. 256.\n");
				}
				o.nth_peak = (int)n;
				break;
			}
			default: die ("Error: unrecognized option. See --help for usage information.\n");
		}
	}
	if (o.sections > 0 && (o.angles_arg || o.oversample || o.gpus != 1)) {
		die ("Error: --sections cannot be combined with -a, --true-peak or --gpus.\n");
	}
	if (o.loudness && (o.angles_arg || o.sections > 0 || o.gpus != 1)) {
		die ("Error: --loudness cannot be combined with -a, --sections or --gpus.\n");
	}
	if (o.overs && (o.sections > 0 || o.gpus != 1)) {
		die ("Error: --overs cannot be combined with --sections or --gpus.\n");
	}
	if (o.nth_peak && (o.angles_arg || o.sections > 0 || o.gpus != 1 || o.loudness)) {
		// (--loudness: its PLR lines are defined on the rank-1 peaks)
		die ("Error: --nth-peak cannot be combined with -a, --sections, --gpus or --loudness.\n");
	}
	kSubsample = o.subsample;
	kMaxSample = 180 * kSubsample;
	if (!o.stride_set) {
		o.stride = 12 * kSubsample;
	}
	if (optind + 1 > argc) {
		die ("Error: Missing parameter. See --help for usage information.\n");
	}
	if (o.stride < 1 || o.stride > 45 * kSubsample || (kMaxSample % o.stride) != 0) {
		die ("Error: 180 deg is not evenly dividable by given stride.\n");
	}
	if (o.blksiz != 0 && (o.blksiz < 1024 || o.blksiz > 32768)) {
		die ("Error: fft-len is out of bounds; valid range 1024..32768\n");
	}
	if (o.angles_arg && optind + 2 > argc) {
		die ("Error: -a, --angle option requires an output file to be given.\n");
	}
	o.in_path = argv[optind];
	if (optind + 1 < argc) {
		o.out_path = argv[optind + 1];
	}
	return o;
}

// "-a n[,n]*" -> grid steps (cli:718-747)
std::vector<int>
parse_angles (const char* arg, int channels)
{
	std::vector<int> angles;
	std::string      s (arg);
	size_t           pos = 0;
	while (pos <= s.size ()) {
		size_t comma = s.find (',', pos);
		if (comma == std::string::npos) {
			comma = s.size ();
		}
		if (comma > pos) { // strtok skips empty fields
			const std::string tok = s.substr (pos, comma - pos);
			char*             ep  = nullptr;
			const double      a   = strtod (tok.c_str (), &ep);
			if (*ep != '\0' || a < -180 || a > 180) {
				die ("Error: Invalid angle speficied, value needs to be -180 .. +180.\n");
			}
			angles.push_back ((int)round (a * (float)kSubsample));
		}
		pos = comma + 1;
	}
	if (angles.size () == 1) {
		while (angles.size () < (size_t)channels) {
			angles.push_back (angles.back ());
		}
	}
	if (angles.size () < (size_t)channels) {
		die ("Error: file has more channels than angles were specified.\n");
	}
	return angles;
}

void
copy_metadata (SNDFILE* in, SNDFILE* out) // cli:541-563
{
	for (int k = SF_STR_FIRST; k <= SF_STR_LAST; ++k) {
		if (const char* str = sf_get_string (in, k)) {
			sf_set_string (out, k, str);
		}
	}
	SF_CUES cues;
	memset (&cues, 0, sizeof (cues));
	if (sf_command (in, SFC_GET_CUE, &cues, sizeof (cues)) == SF_TRUE) {
		sf_command (out, SFC_SET_CUE, &cues, sizeof (cues));
	}
	SF_BROADCAST_INFO binfo;
	memset (&binfo, 0, sizeof (binfo));
	if (sf_command (in, SFC_GET_BROADCAST_INFO, &binfo, sizeof (binfo)) == SF_TRUE) {
		sf_command (out, SFC_SET_BROADCAST_INFO, &binfo, sizeof (binfo));
	}
}

void
check (int rc, const char* what)
{
	if (rc != PHASEROT_OK) {
		join_cuda_warm ();
		fprintf (stderr, "Error: %s: %s (%s)\n", what, phaserot_strerror (rc), phaserot_last_error ());
		::exit (EXIT_FAILURE);
	}
}

/*
 * The GPU's full table, read the way the reference reads PhaseRotate::_peak
 * after a pass that analysed only the channels in `mask` (others are zero after
 * PhaseRotate::reset, cli:355-366).
 */
struct PeakTable {
	int                channels = 0;
	std::vector<float> t; // [channels][kMaxSample]

	float one (int c, int a) const
	{
		if (a < 0) {
			a += kMaxSample;
		}
		return t[(size_t)c * kMaxSample + (size_t)(a % kMaxSample)];
	}
	// PhaseRotate::peak (cli:275-285) / peak_all (cli:287-299)
	float peak (int c, int a, const std::vector<bool>& mask) const
	{
		if (c < 0) {
			float p = 0;
			for (int k = 0; k < channels; ++k) {
				p = std::max (p, mask[(size_t)k] ? one (k, a) : 0.f);
			}
			return p;
		}
		return mask[(size_t)c] ? one (c, a) : 0.f;
	}
};

// Angle search on one peak table: the coarse pass over every `stride`-th angle, then the refine pass
// around its local minima, replayed on the table (cli:815-929).  angle[c] is what the reference applies
// (channels without a minimum: 0, p_min = +inf).
struct MinResult {
	std::vector<int>   angle;
	std::vector<float> p_min, r_zro, r_min;
};

MinResult
find_min_angles (const PeakTable& tab, const Options& opt, FILE* vfd)
{
const int               C      = tab.channels;
const int               stride = opt.stride;
const std::vector<bool> all ((size_t)C, true);

	if (opt.verbose > 1) { // gnuplot table of the coarse pass (cli:800-813)
		printf ("# Angle mono-peak");
		for (int c = 0; c < C; ++c) {
			printf (" chn-%d", c + 1);
		}
		printf ("\n");
		for (int a = 0; a < kMaxSample; a += stride) {
			printf ("%.2f %.4f", a / (float)kSubsample, to_dB (tab.peak (-1, a, all)));
			for (int c = 0; c < C; ++c) {
				printf (" %.4f", to_dB (tab.peak (c, a, all)));
			}
			printf ("\n");
		}
	}

	const float inf = std::numeric_limits<float>::infinity ();
	std::map<int, std::vector<int>> mins; // coarse angle -> channels to refine there
	std::vector<int>   min_angle ((size_t)C, 0);
	// The reference leaves p_min / min_angle uninitialised for a channel whose
	// coarse peaks are all equal (cli:835-839); +inf / 0 is the evident intent.
	std::vector<float> p_min ((size_t)C, inf), r_zro ((size_t)C, 0.f), r_min ((size_t)C, 0.f);

	for (int c = 0; c < C; ++c) {
		const int pc   = opt.link ? -1 : c;
		float     cmin = inf, cmax = 0;
		r_zro[(size_t)c] = tab.peak (c, 0, all);
		for (int a = 0; a < kMaxSample; a += stride) {
			cmin = std::min (cmin, tab.peak (pc, a, all));
			cmax = std::max (cmax, tab.peak (pc, a, all));
		}
		float range = cmax - cmin;
		if (range == 0) {
			mins[0].push_back (c);
			continue;
		}
		if (stride > 1) {
			range *= .07;
			p_min[(size_t)c] = inf;
		} else {
			range            = 0;
			p_min[(size_t)c] = cmin;
		}
		for (int a = 0; a < kMaxSample; a += stride) {
			const float p = tab.peak (pc, a, all);
			if (p <= cmin + range) {
				mins[a].push_back (c);
				if (opt.verbose > 1) {
					fprintf (vfd, "Consider min: %f (< %f) chn: %d @ %.2f deg\n", p, cmin + range, c, a / (float)kSubsample);
				}
			}
		}
	}

	if (stride == 1) {
		for (auto& mp : mins) { // ascending: the largest angle wins (cli:859-865)
			for (int cn : mp.second) {
				min_angle[(size_t)cn] = mp.first;
				r_min[(size_t)cn]     = tab.peak (cn, mp.first, all);
			}
		}
	} else {
		const int s2 = (stride + 1) / 2;
		for (auto& mp : mins) {
			// which channels the reference's refine pass analyses (cli:880)
			std::vector<bool> mask ((size_t)C, mp.second.size () > 1);
			if (mp.second.size () == 1) {
				mask[(size_t)mp.second.front ()] = true;
			}
			const int ma = mp.first;
			for (int cn : mp.second) {
				for (int a = ma - s2; a < ma + s2 + 1; ++a) {
					const float p = tab.peak (opt.link ? -1 : cn, a, mask);
					if (p <= p_min[(size_t)cn]) { // ties: the later angle wins (cli:885)
						p_min[(size_t)cn]     = p;
						r_min[(size_t)cn]     = tab.peak (cn, a, mask);
						min_angle[(size_t)cn] = (a + kMaxSample) % kMaxSample;
					}
					if (opt.verbose > 1) {
						printf ("%.2f %.4f", ((a + kMaxSample) % kMaxSample) / (float)kSubsample, to_dB (tab.peak (-1, a, mask)));
						for (int c = 0; c < C; ++c) {
							printf (" %.4f", to_dB (tab.peak (c, a, mask)));
						}
						printf ("\n");
					}
				}
			}
		}
	}

	// minimise the channel phase distance (cli:905-929)
	float avg_rotate = 0;
	int   avg_count  = 0;
	for (int c = 0; c < C; ++c) {
		if (p_min[(size_t)c] != inf) {
			avg_rotate += min_angle[(size_t)c];
			++avg_count;
		}
	}
	avg_rotate /= avg_count;
	const float avg_dist = kMaxSample / (float)avg_count;
	for (int c = 0; c < C; ++c) {
		if (p_min[(size_t)c] == inf) {
			continue;
		}
		if (min_angle[(size_t)c] > 90 * kSubsample && fabsf (min_angle[(size_t)c] - avg_rotate) > avg_dist) {
			min_angle[(size_t)c] -= kMaxSample;
		} else if (avg_rotate > 90 * kSubsample) {
			min_angle[(size_t)c] -= kMaxSample;
		}
	}
	return MinResult { min_angle, p_min, r_zro, r_min };
}

// the per-channel result lines of the report (cli:931-947)
void
report_channels (const MinResult& r, FILE* vfd)
{
	const float inf = std::numeric_limits<float>::infinity ();
	for (size_t c = 0; c < r.angle.size (); ++c) {
		if (r.p_min[c] == inf) {
			fprintf (vfd, "Channel: %2d Phase:   0 deg # cannot find min.\n", (int)c + 1);
			continue;
		}
		fprintf (vfd, "Channel: %2d Phase: %5.2f deg", (int)c + 1, r.angle[c] / (float)kSubsample);
		if (r.angle[c] != 0) {
			fprintf (vfd, ", gain: %5.2f dB (att. %4.2f to %4.2f dBFS)", to_dB (r.r_zro[c]) - to_dB (r.r_min[c]), to_dB (r.r_zro[c]), to_dB (r.r_min[c]));
		}
		fprintf (vfd, "\n");
	}
}

} // namespace

int
main (int argc, char** argv)
{
	StageTimer timer;
	Options    opt = parse_options (argc, argv);
	if (opt.gpus == 1 && !getenv ("CUDA_VISIBLE_DEVICES")) {
		// one device is used: do not let the driver bring up every GPU of the box (most of the
		// process start-up on an 8-GPU node); an explicit CUDA_VISIBLE_DEVICES is respected
		setenv ("CUDA_VISIBLE_DEVICES", "0", 0);
	}

	SF_INFO nfo;
	memset (&nfo, 0, sizeof (nfo));
	SNDFILE* infile = sf_open (opt.in_path, SFM_READ, &nfo);
	if (!infile) {
		fprintf (stderr, "Cannot open '%s' for reading: ", opt.in_path);
		fputs (sf_strerror (NULL), stderr);
		::exit (EXIT_FAILURE);
	}
	const bool find_min = opt.angles_arg == nullptr;
	if (!nfo.seekable) { // the reference tests `find_min && !seekable` with find_min still true (cli:691)
		fprintf (stderr, "File '%s' is not seekable. ", opt.in_path);
		::exit (EXIT_FAILURE);
	}
	SNDFILE* outfile = nullptr;
	if (opt.out_path) {
		outfile = sf_open (opt.out_path, SFM_WRITE, &nfo);
		if (!outfile) {
			fprintf (stderr, "Cannot open '%s' for writing: ", opt.out_path);
			fputs (sf_strerror (NULL), stderr);
			::exit (EXIT_FAILURE);
		}
	}

	// Bringing up the CUDA context takes ~0.7 s on a B200 - longer than the whole reference run
	// on a one-minute file.  It needs nothing from the file, so it runs on its own thread while
	// the main thread opens, reads and decodes the audio (into ordinary memory: the library
	// stages it through its own page-locked chunk buffers during the upload).
	// (started once the files are open: the error exits above stay trivial; later ones join it first)
	g_cuda_warm = std::thread ([] { phaserot_free_host (phaserot_alloc_host (64)); });

	FILE* vfd = opt.verbose > 1 ? stderr : stdout;
	if (opt.verbose > 2) {
		std::vector<char> log (65536);
		sf_command (infile, SFC_GET_LOG_INFO, log.data (), (int)log.size ());
		fputs (log.data (), vfd);
	} else if (opt.verbose) {
		fprintf (vfd, "Input File      : %s\n", opt.in_path);
		fprintf (vfd, "Sample Rate     : %d Hz\n", nfo.samplerate);
		fprintf (vfd, "Channels        : %d\n", nfo.channels);
	}

	const int        C = nfo.channels;
	std::vector<int> angles;
	if (opt.angles_arg) {
		angles = parse_angles (opt.angles_arg, C);
		if (opt.verbose) {
			fprintf (vfd, "# Apply phase-shift\n");
			for (int c = 0; c < C; ++c) {
				fprintf (vfd, "Channel: %2d Phase: %5.2f deg\n", c + 1, angles[(size_t)c] / (float)kSubsample);
			}
		}
	}

	// block size (cli:749-755)
	unsigned int blksiz = opt.blksiz;
	if (blksiz == 0 || blksiz > 32768) {
		blksiz = (unsigned int)nfo.samplerate / 8;
	}
	unsigned p2;
	for (p2 = 1; 1U << p2 < blksiz; ++p2)
		;
	blksiz = (unsigned int)std::min (32768, std::max (1024, 1 << p2));
	if (opt.verbose > 1) {
		fprintf (vfd, "Process block-size %d\n", blksiz);
	}

	// the whole file in page-locked memory.  Analysis only of an integer PCM file:
	// the samples stay integers on the host and on the bus (2 bytes per sample for
	// 16 bit) and are widened on the device exactly as sf_readf_float would
	// (phaserot_sweep_pcm); everything else is read as float like the reference
	// does (cli:573).
	const uint64_t frames  = nfo.frames > 0 ? (uint64_t)nfo.frames : 0;
	const int      subfmt  = nfo.format & SF_FORMAT_SUBMASK;
	// 24-bit samples of a little-endian container (WAV, RF64, W64; format word without an
	// endianness override) travel packed, 3 bytes each, exactly as sf_read_raw delivers them
	const int      major   = nfo.format & SF_FORMAT_TYPEMASK;
	const bool     raw24   = subfmt == SF_FORMAT_PCM_24 && (nfo.format & 0x30000000) == 0 && (major == SF_FORMAT_WAV || major == 0x220000 /* RF64 */ || major == 0x0B0000 /* W64 */);
	const int      pcm_fmt = (find_min && !opt.out_path && subfmt == SF_FORMAT_PCM_16)                                 ? PHASEROT_PCM_S16
	                         : (find_min && !opt.out_path && raw24)                                                     ? PHASEROT_PCM_S24
	                         : (find_min && !opt.out_path && (subfmt == SF_FORMAT_PCM_24 || subfmt == SF_FORMAT_PCM_32)) ? PHASEROT_PCM_S32
	                                                                                                                      : 0;
	const size_t   ssize   = pcm_fmt == PHASEROT_PCM_S16 ? sizeof (short) : pcm_fmt == PHASEROT_PCM_S24 ? 3 : sizeof (float); // int and float are both 4 bytes
	const size_t   fbytes  = std::max<size_t> (ssize * (size_t)frames * (size_t)C, 16);
	timer.mark ("open file");
	float*         audio   = (float*)malloc (fbytes);
	bool           pinned  = false;
	if (!audio) {
		die ("Out of memory\n");
	}
	uint64_t got = 0;
	while (got < frames) {
		const sf_count_t want = (sf_count_t)std::min<uint64_t> (frames - got, 1u << 20);
		sf_count_t       n;
		if (pcm_fmt == PHASEROT_PCM_S16) {
			n = sf_readf_short (infile, (short*)audio + got * (uint64_t)C, want);
		} else if (pcm_fmt == PHASEROT_PCM_S24) {
			n = sf_read_raw (infile, (char*)audio + 3 * got * (uint64_t)C, want * 3 * (sf_count_t)C) / (3 * (sf_count_t)C);
		} else if (pcm_fmt == PHASEROT_PCM_S32) {
			n = sf_readf_int (infile, (int*)audio + got * (uint64_t)C, want);
		} else {
			n = sf_readf_float (infile, audio + got * (uint64_t)C, want);
		}
		if (n <= 0) {
			break;
		}
		got += (uint64_t)n;
	}
	const uint64_t F = got;
	timer.mark ("read + decode file");

	phaserot_cfg_t cfg;
	memset (&cfg, 0, sizeof (cfg));
	cfg.abi_version = PHASEROT_ABI_VERSION;
	cfg.mode        = PHASEROT_MODE_CLI;
	cfg.n_channels  = C;
	cfg.blksiz      = (int32_t)blksiz;
	cfg.subsample   = kSubsample;
	cfg.device      = -1;
	cfg.oversample  = opt.oversample;
	join_cuda_warm ();
	timer.mark ("wait for CUDA init");
	phaserot_t*       pr  = nullptr;
	phaserot_group_t* grp = nullptr;
	if (opt.gpus != 1) {
		// --gpus N: one contiguous shard of the file per device, tables combined on the
		// first device over NVLink (phaserot_group_sweep); rendering stays on the first device
		int ndev = opt.gpus;
		if (ndev == 0) {
			phaserot_group_t* probe = nullptr;
			for (ndev = 16; ndev > 1; --ndev) { // the largest group the box can form
				if (phaserot_group_create (&probe, &cfg, nullptr, ndev) == PHASEROT_OK) {
					break;
				}
			}
			grp = probe;
		}
		if (!grp) {
			check (phaserot_group_create (&grp, &cfg, nullptr, ndev), "cannot initialise the CUDA backend");
		}
		pr = phaserot_group_handle (grp, 0);
		if (opt.verbose > 1) {
			fprintf (vfd, "Analyzing on %d GPUs\n", phaserot_group_size (grp));
		}
	} else {
		check (phaserot_create (&pr, &cfg), "cannot initialise the CUDA backend");
	}
	timer.mark ("phaserot_create (tables, kernels)");

	MinResult        res;          // whole-file analysis: what the result lines report
	uint64_t         sect_len = 0; // --sections: frames per section
	std::vector<int> sect_angles;  // --sections: [section][channel] in grid steps on the full circle
	if (find_min && opt.sections > 0) {
		// one sweep, one table per section; the search of the whole-file analysis runs on each of them
		const uint64_t al = phaserot_shard_align (pr);
		sect_len          = std::max<uint64_t> (1, (uint64_t)ceil (ceil (opt.sections * nfo.samplerate) / (double)al)) * al; // rounded up
		if (opt.verbose) {
			fprintf (vfd, "Section length  : %.3f s (%llu frames)\n", sect_len / (double)nfo.samplerate, (unsigned long long)sect_len);
		}
		check (phaserot_sweep_sections (pr, audio, pcm_fmt, F, sect_len, 0, kMaxSample, 1, -1), "analysis failed");
		int ns = 0;
		check (phaserot_section_peaks (pr, &ns, nullptr), "analysis failed");
		const size_t       per = (size_t)C * kMaxSample;
		std::vector<float> tables ((size_t)ns * per);
		check (phaserot_section_peaks (pr, &ns, tables.data ()), "analysis failed");
		timer.mark ("analysis (upload + sweep)");
		if (!outfile || opt.verbose) {
			fprintf (vfd, "# Result -- Minimize digital peak\n");
		}
		PeakTable tab;
		tab.channels = C;
		for (int k = 0; k < ns; ++k) {
			tab.t.assign (tables.begin () + (std::ptrdiff_t)(k * per), tables.begin () + (std::ptrdiff_t)((k + 1) * per));
			const MinResult r = find_min_angles (tab, opt, vfd);
			if (!outfile || opt.verbose) {
				fprintf (vfd, "# Section %d: %.3f - %.3f s\n", k + 1, (double)k * sect_len / nfo.samplerate,
				         (double)std::min<uint64_t> (F, (uint64_t)(k + 1) * sect_len) / nfo.samplerate);
				report_channels (r, vfd);
			}
			for (int c = 0; c < C; ++c) {
				// section 0 renders at the index the whole-file render uses (cli:463); every following section
				// at whichever of a, a - 180 deg (the same peak) is nearer to the angle before it: a ramp
				// between sections never turns more than 90 degrees
				int a = ((r.angle[(size_t)c] % kMaxSample) + kMaxSample) % kMaxSample;
				if (k > 0) {
					a += kMaxSample * (int)lround ((sect_angles[(size_t)(k - 1) * C + c] - a) / (double)kMaxSample);
				}
				sect_angles.push_back (a);
			}
		}
	} else if (find_min) {
		const int stride = opt.stride;
		if (opt.verbose > 1) {
			fprintf (vfd, "Analyzing using %d process threads, stride = %d\n", C, stride);
		}
		PeakTable tab;
		tab.channels = C;
		tab.t.resize ((size_t)C * kMaxSample);
		if (opt.nth_peak) {
			// --nth-peak N: one pass, the N largest samples at every grid index (index 0 = the input); the search
			// and the report run on the rank-N levels as they would on the peaks (rank 1 is the peak table)
			const size_t       N = (size_t)opt.nth_peak;
			std::vector<float> ranks (tab.t.size () * N, 0.f);
			if (F > 0) {
				check (phaserot_nth_peaks (pr, audio, pcm_fmt, F, opt.nth_peak, 0, kMaxSample, 1, -1, ranks.data ()), "analysis failed");
			}
			for (size_t i = 0; i < tab.t.size (); ++i) tab.t[i] = ranks[i * N + N - 1];
		} else {
			// one pass, every grid index (index 0 = raw peak, cli:413-414)
			if (grp) {
				check (phaserot_group_sweep (grp, audio, pcm_fmt, F, 0, kMaxSample, 1, -1), "analysis failed");
			} else if (pcm_fmt) {
				check (phaserot_sweep_pcm (pr, audio, pcm_fmt, F, 0, kMaxSample, 1, -1), "analysis failed");
			} else {
				check (phaserot_sweep (pr, audio, F, 0, kMaxSample, 1, -1), "analysis failed");
			}
			check (phaserot_peaks (pr, tab.t.data ()), "analysis failed");
		}
		timer.mark ("analysis (upload + sweep)");
		res    = find_min_angles (tab, opt, vfd);
		angles = res.angle;
		if (!outfile || opt.verbose) { // report (cli:931-947)
			if (opt.nth_peak > 1) {
				fprintf (vfd, "# Result -- Minimize digital peak, rank %d\n", opt.nth_peak);
			} else {
				fprintf (vfd, "# Result -- Minimize digital peak\n");
			}
			report_channels (res, vfd);
		}
	}

	if (opt.loudness) {
		// BS.1770-4 integrated loudness of the input (set 0: angle 0) and of the --fixed-write render at the
		// applied angles (set 1), and the peak-to-loudness ratios with the peaks of the result lines
		std::vector<int> sets ((size_t)2 * C, 0);
		std::copy (angles.begin (), angles.end (), sets.begin () + C);
		std::vector<float> w ((size_t)C, 1.f);
		if (C == 6) {
			w = { 1.f, 1.f, 1.f, 0.f, 1.41f, 1.41f }; // BS.1770 5.1 weights, WAV order L R C LFE Ls Rs
		}
		double lufs[2] = { -std::numeric_limits<double>::infinity (), -std::numeric_limits<double>::infinity () };
		if (F > 0) {
			check (phaserot_loudness (pr, audio, pcm_fmt, F, (double)nfo.samplerate, w.data (), sets.data (), 2, lufs), "loudness failed");
		}
		float pk_in = 0.f, pk_out = 0.f;
		for (int c = 0; c < C; ++c) {
			pk_in  = std::max (pk_in, res.r_zro[(size_t)c]);
			pk_out = std::max (pk_out, res.p_min[(size_t)c] == std::numeric_limits<float>::infinity () ? res.r_zro[(size_t)c] : res.r_min[(size_t)c]);
		}
		printf ("# Loudness -- ITU-R BS.1770-4 integrated\n");
		printf ("Input : %.2f LUFS, PLR %.2f dB\n", lufs[0], to_dB (pk_in) - lufs[0]);
		printf ("Output: %.2f LUFS, PLR %.2f dB\n", lufs[1], to_dB (pk_out) - lufs[1]);
		timer.mark ("loudness");
	}

	if (opt.overs) {
		// samples above the ceiling at every grid angle (index 0: the input), reported at the input, at the
		// applied angle (a and a + 180 deg give the same |y|) and at the angle with the fewest
		const float           T = (float)pow (10.0, opt.overs_db / 20.0);
		std::vector<uint64_t> n ((size_t)C * kMaxSample, 0);
		if (F > 0) {
			check (phaserot_overs (pr, audio, pcm_fmt, F, T, 0, kMaxSample, 1, -1, n.data (), nullptr), "overs failed");
		}
		printf ("# Overs -- samples above %.2f %s\n", opt.overs_db, opt.oversample ? "dBTP" : "dBFS");
		for (int c = 0; c < C; ++c) {
			const uint64_t* row  = n.data () + (size_t)c * kMaxSample;
			const int       out  = ((angles[(size_t)c] % kMaxSample) + kMaxSample) % kMaxSample;
			int             best = 0;
			for (int a = 1; a < kMaxSample; ++a) {
				if (row[a] <= row[best]) best = a; // ties: the largest index, like the reference's search
			}
			printf ("Channel: %2d Input: %llu Output: %llu Fewest: %llu at %.2f deg\n", c + 1, (unsigned long long)row[0], (unsigned long long)row[out],
			        (unsigned long long)row[best], best / (float)kSubsample);
		}
		timer.mark ("overs");
	}

	if (outfile) {
		copy_metadata (infile, outfile);
		check (phaserot_reset (pr), "reset failed");

		const uint32_t L       = blksiz;
		const uint32_t latency = L / 2; // cli:963
		const size_t   bs      = (size_t)L * (size_t)C;
		const uint64_t n_full  = F / L;              // blocks made of file data only
		const uint32_t rem     = (uint32_t)(F % L);  // frames in the short last block
		bool           failed  = false;
		uint32_t       pad     = 0;
		uint32_t       off     = latency;

		// what the reference passes to sf_writef_float for one processed block
		auto write_block = [&] (const float* blk, sf_count_t n) {
			n -= off;
			if (!failed && n != sf_writef_float (outfile, &blk[off], n)) { // float offset, like cli:985
				fprintf (stderr, "Error writing to output file.\n");
				pad    = latency;
				failed = true;
			}
			off = 0;
		};

		std::vector<float> last_out (bs, 0.f); // processed block the reference would still hold in `buf`
		if (opt.fixed_write || sect_len) {
			// --fixed-write: the latency-compensated render y[t + L/2], t in [0, F), as the
			// write loop intends it: the trim counts FRAMES (the reference offsets the
			// interleaved buffer by `latency` floats, cli:985: channels > 1 start at frame
			// latency / channels) and a short last block is always zero padded (cli:973
			// leaves the previous block's output behind it when it is longer than the latency)
			const uint64_t nb = (F + L - 1) / L + 1;
			float*         y  = (float*)phaserot_alloc_host (sizeof (float) * bs * nb);
			const bool     yp = y != nullptr;
			if (!y) {
				y = (float*)malloc (sizeof (float) * bs * nb);
			}
			if (!y) {
				die ("Out of memory\n");
			}
			if (sect_len) { // --sections: always written this way
				check (phaserot_render_sections (pr, audio, F, sect_len, sect_angles.data (), 1, y), "render failed");
			} else {
				check (phaserot_render (pr, audio, F, angles.data (), 1, y), "render failed");
			}
			if ((sf_count_t)F != sf_writef_float (outfile, y + (size_t)latency * (size_t)C, (sf_count_t)F)) {
				fprintf (stderr, "Error writing to output file.\n");
			}
			if (yp) {
				phaserot_free_host (y);
			} else {
				free (y);
			}
			sf_close (outfile);
			outfile = nullptr;
		}
		if (outfile && n_full > 0) {
			float* y = (float*)phaserot_alloc_host (sizeof (float) * bs * n_full);
			bool   y_pinned = y != nullptr;
			if (!y) {
				y = (float*)malloc (sizeof (float) * bs * n_full);
			}
			if (!y) {
				die ("Out of memory\n");
			}
			check (phaserot_render (pr, audio, n_full * L, angles.data (), 0, y), "render failed");
			for (uint64_t b = 0; b < n_full && !failed; ++b) {
				write_block (y + b * bs, (sf_count_t)L);
			}
			memcpy (last_out.data (), y + (n_full - 1) * bs, sizeof (float) * bs);
			if (y_pinned) {
				phaserot_free_host (y);
			} else {
				free (y);
			}
		}
		if (outfile && rem > 0 && !failed) {
			// short last block (cli:968-990): frames beyond `rem` keep the previous
			// processed block unless rem < latency, in which case they are zeroed
			std::vector<float>& buf = last_out;
			memcpy (buf.data (), audio + n_full * bs, sizeof (float) * (size_t)rem * (size_t)C);
			sf_count_t n = rem;
			if (rem < latency) {
				memset (&buf[(size_t)C * rem], 0, sizeof (float) * (size_t)C * (L - rem));
				pad = latency - rem;
				n += pad;
			}
			check (phaserot_apply (pr, buf.data (), angles.data ()), "render failed");
			write_block (buf.data (), n);
		}
		const sf_count_t nflush = outfile ? (sf_count_t)latency - pad : 0; // cli:993-1001
		if (nflush > 0) {
			std::vector<float> z (bs, 0.f);
			check (phaserot_apply (pr, z.data (), angles.data ()), "render failed");
			if (nflush != sf_writef_float (outfile, z.data (), nflush)) {
				fprintf (stderr, "Error writing to output file.\n");
			}
		}
		if (outfile) {
			sf_close (outfile);
		}
	}

	timer.mark ("search + report + render/write");
	if (grp) {
		phaserot_group_destroy (grp);
	} else {
		phaserot_destroy (pr);
	}
	timer.mark ("destroy");
	sf_close (infile);
	if (pinned) {
		phaserot_free_host (audio);
	} else {
		free (audio);
	}
	return 0;
}
