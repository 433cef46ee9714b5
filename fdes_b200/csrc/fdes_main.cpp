// fdes_b200 -- command-line front end with the option set of the reference CLI
// (reference src/FDES.cu:61-263, Useage.txt:26-37):
//   FDES [--input_name f.cnf] [--image_name out.bin] [--emd_name out.emd]
//        [--print_level 0|1|2] [--gpu_index n] [--help] [--version]
// Defaults as in src/FDES.cu:40-44: dataFDES.cnf -> Measurements.bin, results.emd.
#include "../../include/fdes_b200.h"
#include "params.h"
#include "emd.h"
#include <fcntl.h>
#include <getopt.h>
#include <sys/mman.h>
#include <unistd.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <string>
#include <vector>

int main(int argc, char** argv)
{
    std::string input = "dataFDES.cnf", image = "Measurements.bin", emd = "results.emd";
    int gpu_index = 0, print_level = 0;
    bool stem_scan = false;
    std::string stem_4d;
    int stem_4d_bin = 1;
    std::string gpus_spec;
    static struct option opts[] = {{"gpu_index", required_argument, 0, 0},
                                   {"input_name", required_argument, 0, 0},
                                   {"image_name", required_argument, 0, 0},
                                   {"emd_name", required_argument, 0, 0},
                                   {"print_level", required_argument, 0, 0},
                                   {"help", no_argument, 0, 0},
                                   {"version", no_argument, 0, 0},
                                   {"stem_scan", no_argument, 0, 0},   // extension, see below
                                   {"gpus", required_argument, 0, 0},  // extension: shard the run over several GPUs
                                   {"stem_4d", required_argument, 0, 0},       // extension: 4D-STEM data set of --stem_scan
                                   {"stem_4d_bin", required_argument, 0, 0},
                                   {NULL, 0, 0, 0}};
    while (true) {
        int idx = 0;
        const int c = getopt_long(argc, argv, "", opts, &idx);
        if (c == -1) break;
        if (c != 0) { fprintf(stderr, "  unknown option, try --help\n"); return EXIT_FAILURE; }
        switch (idx) {
            case 0: gpu_index = atoi(optarg); break;
            case 1: input = optarg; fprintf(stderr, "  input_name %s  \n", optarg); break;
            case 2: image = optarg; break;
            case 3: emd = optarg; break;
            case 4:
                print_level = atoi(optarg);
                if (print_level < 0 || print_level > 2) {
                    fprintf(stderr, " \n printLevel error %s  \n", input.c_str());
                    return EXIT_FAILURE;
                }
                break;
            case 5:
                fprintf(stderr,
                        " \nUsage: \n"
                        "  [ --input_name  <parameter file (.cnf)> ]\n"
                        "  [ --image_name  <raw float32 image output, default Measurements.bin> ]\n"
                        "  [ --emd_name    <results name, default results.emd> ]\n"
                        "  [ --print_level <0 images | 1 + potential slices | 2 + exit waves> ]\n"
                        "  [ --gpu_index   <CUDA device ordinal, default 0> ]\n"
                        "  [ --help ] [ --version ]\n"
                        "  [ --gpus        extension: <count> (gpu_index, gpu_index + 1, ...) or a list i,j,... -- frozen-phonon\n"
                        "                  configurations, tilt/defocus series or STEM probes are sharded over these GPUs ]\n"
                        "  [ --stem_scan   extension: run the probe scan a `mode: STEM` .qsc describes (scan_* and\n"
                        "                  detector: keys); image_name receives float32 [detector][x][y] ]\n"
                        "  [ --stem_4d     extension, with --stem_scan: <path> receives the diffraction pattern of every probe\n"
                        "                  of the same scan, raw float32 [x][y][qy][qx]: fftshifted, cropped to the smallest\n"
                        "                  centred window that holds the band limit, binned; image_name as without it ]\n"
                        "  [ --stem_4d_bin <b>: pattern pixels summed b x b (default 1) ]\n");
                return EXIT_FAILURE;
            case 7: stem_scan = true; break;
            case 8: gpus_spec = optarg; break;
            case 9: stem_4d = optarg; break;
            case 10: stem_4d_bin = atoi(optarg); break;
            case 6: fprintf(stderr, " \n FDES (fdes_b200) Version : %1.1f  \n", fdes_b200_version() / 100.0); return EXIT_FAILURE;
        }
    }
    // The CLI takes the atoms from the file; FDES() wants them as an array (atomsFromExternal).
    fdes::Params p;
    fdes::Atoms atoms;
    bool ok = false;
    try { ok = fdes::read_input(input.c_str(), p, &atoms, false); }
    catch (const std::exception& e) { fprintf(stderr, " \n fdes_b200: %s \n", e.what()); }
    if (!ok) {
        fprintf(stderr, " \n Errors occur when reading \"%s\" \n", input.c_str());
        return EXIT_FAILURE;
    }
    if (atoms.size() == 0) { fprintf(stderr, "No valid configuration for simulation!.\n"); return EXIT_FAILURE; }
    std::vector<float> a6(6 * (size_t)atoms.size());
    for (int i = 0; i < atoms.size(); i++) {
        a6[6 * i + 0] = (float)atoms.Z[i];
        a6[6 * i + 1] = atoms.xyz[3 * i + 0];
        a6[6 * i + 2] = atoms.xyz[3 * i + 1];
        a6[6 * i + 3] = atoms.xyz[3 * i + 2];
        a6[6 * i + 4] = atoms.dwf[i];
        a6[6 * i + 5] = atoms.occ[i];
    }
    // devices of the run: --gpus, else the environment (FDES_B200_GPUS, as FDES() reads it), else gpu_index
    const char* spec = !gpus_spec.empty() ? gpus_spec.c_str() : getenv("FDES_B200_GPUS");
    std::vector<int> gpus((size_t)std::max(1, fdes_b200_parse_gpu_list(spec, gpu_index, nullptr, 0)));
    fdes_b200_parse_gpu_list(spec, gpu_index, gpus.data(), (int)gpus.size());
    if (!stem_4d.empty() && !stem_scan) { fprintf(stderr, " \n --stem_4d needs --stem_scan \n"); return EXIT_FAILURE; }
    if (stem_scan) {
        // Extension (FDES has no STEM mode): the raster and detectors of a QSTEM `mode: STEM` file, keys the
        // reference parses and drops (src/rwQsc.cu:444-466, 698-735), drive the batched probe scan.
        int nxy[2] = {0, 0};
        const int ndet = fdes_b200_qsc_scan(input.c_str(), nxy, nullptr, 0, nullptr, 0);
        if (ndet <= 0) {
            fprintf(stderr, " \n fdes_b200: %s \n", ndet < 0 ? fdes_b200_last_error() : "--stem_scan: the file has no `detector:` line");
            return EXIT_FAILURE;
        }
        const int np = nxy[0] * nxy[1];
        std::vector<float> xy(2 * (size_t)np), det(2 * (size_t)ndet), sig((size_t)np * ndet), out((size_t)np * ndet);
        fdes_b200_qsc_scan(input.c_str(), nxy, xy.data(), np, det.data(), ndet);
        fdes_b200_sim* sim = fdes_b200_open_multi(input.c_str(), nullptr, 0, gpus.data(), (int)gpus.size(), 37, 0);   // 37 probes per launch: whole waves of 148 SMs at 512^2
        if (!sim) { fprintf(stderr, " \n fdes_b200: %s \n", fdes_b200_last_error()); return EXIT_FAILURE; }
        double ms = 0.0;
        if (stem_4d.empty()) {
            ms = fdes_b200_stem_scan(sim, 0, np, xy.data(), ndet, det.data(), sig.data());
        } else {
            // the data set goes straight into the mapped output file: [x][y][qy][qx], probe i = x * ny + y
            int dims[10];
            fdes_b200_get_dims(sim, dims);
            const int side = fdes_b200_stem_4d_side(dims[3], 0, stem_4d_bin);
            if (side < 0) { fprintf(stderr, " \n fdes_b200: --stem_4d_bin: %s \n", fdes_b200_last_error()); return EXIT_FAILURE; }
            const size_t bytes = (size_t)np * side * side * sizeof(float);
            const int fd = open(stem_4d.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0644);
            void* map = MAP_FAILED;
            if (fd >= 0 && ftruncate(fd, (off_t)bytes) == 0) map = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
            if (map == MAP_FAILED) {
                fprintf(stderr, " \n fdes_b200: cannot write %s \n", stem_4d.c_str());
                return EXIT_FAILURE;
            }
            ms = fdes_b200_stem_scan_4d(sim, 0, np, xy.data(), 0, stem_4d_bin, ndet, det.data(), 0, static_cast<float*>(map), sig.data());
            const bool synced = msync(map, bytes, MS_SYNC) == 0;
            munmap(map, bytes);
            if (close(fd) != 0 || !synced) {
                fprintf(stderr, " \n fdes_b200: cannot write %s \n", stem_4d.c_str());
                return EXIT_FAILURE;
            }
        }
        if (ms < 0) { fprintf(stderr, " \n fdes_b200: %s \n", fdes_b200_last_error()); return EXIT_FAILURE; }
        for (int i = 0; i < np; i++)
            for (int d = 0; d < ndet; d++) out[(size_t)d * np + i] = sig[(size_t)i * ndet + d];   // [probe][det] -> [det][x][y]
        fdes::write_binary(image.c_str(), out.data(), out.size());
        fdes::write_cnf("ParamsUsedQsc.txt", p, atoms, gpu_index);
        fdes_b200_close(sim);
        fprintf(stderr, "  STEM scan: %d x %d probes, %d detectors, %.2f ms on the device (%.0f probes/s)\n  Done.\n", nxy[0],
                nxy[1], ndet, ms, np / (ms * 1e-3));
        return 0;
    }
    // NOTE: FDES() truncates the occupancy to an integer like the reference's readAtomsFromArray;
    // the file path keeps fractional occupancies, so the CLI goes through the session API.
    fdes_b200_sim* sim = fdes_b200_open_multi(input.c_str(), nullptr, 0, gpus.data(), (int)gpus.size(), 0, print_level > 1);
    if (!sim) { fprintf(stderr, " \n fdes_b200: %s \n", fdes_b200_last_error()); return EXIT_FAILURE; }
    int d[10];
    fdes_b200_get_dims(sim, d);
    const size_t n123 = (size_t)d[0] * d[1] * d[2], m12 = (size_t)d[3] * d[4];
    std::vector<float> img(n123), ew, pot;
    if (print_level > 1) ew.resize(2 * m12 * d[2]);
    if (fdes_b200_simulate(sim, img.data(), ew.empty() ? nullptr : ew.data()) != 0) {
        fprintf(stderr, " \n fdes_b200: %s \n", fdes_b200_last_error());
        return EXIT_FAILURE;
    }
    if (print_level > 0) {
        pot.resize(2 * m12 * (size_t)fdes_b200_potential_slices_count(sim));
        if (fdes_b200_potential(sim, pot.data()) != 0) {
            fprintf(stderr, " \n fdes_b200: %s \n", fdes_b200_last_error());
            return EXIT_FAILURE;
        }
    }
    fdes::write_cnf(strstr(input.c_str(), ".emd") ? "ParamsUsedEmd.txt" : fdes::is_qsc_name(input.c_str()) && !strstr(input.c_str(), ".cnf") ? "ParamsUsedQsc.txt" : "dataFDES_used.cnf", p, atoms, gpu_index);
    fdes::write_binary(image.c_str(), img.data(), n123);
    if (!strstr(input.c_str(), ".emd")) fdes::write_emd("config.emd", p, atoms, nullptr, nullptr, 0, nullptr);   // src/FDES.cu:229-232
    fdes::write_emd(emd.c_str(), p, atoms, img.data(), pot.empty() ? nullptr : pot.data(),
                    pot.empty() ? 0 : fdes_b200_potential_slices_count(sim), ew.empty() ? nullptr : ew.data());
    fdes_b200_close(sim);
    fprintf(stderr, "  Done.\n");
    return 0;
}
