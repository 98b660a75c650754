// AddressSanitizer run of the FLAC decoder's per-frame functions (csrc/emu.cu replays fl_frame, fl_mix_frame and
// fl_divide).  Each frame is decoded alone from a heap buffer that holds exactly its bytes, placed at the frame's
// offset modulo 4 (the bit reader's word alignment) with the bytes before it poisoned, so a read before or past the
// frame is reported; outputs go to a buffer that ends exactly where the file's output does.
//
// Input (argv[1], written by tests/test_flac.py): records of
//   int32 case, int32 n_frames, dspx_flac_file, then per frame: dspx_flac_frame and its in_bytes bytes.
// Output: one line "flac case C frame F status S" per frame.
#include <sanitizer/asan_interface.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../include/dspx.h"
extern "C" int emu_flac_decode(const void *in, const dspx_flac_file *files, int64_t n_files, const dspx_flac_frame *frames,
                               int64_t n_frames, int normalize, float *out, int32_t *status);

int main(int argc, char **argv)
{
    if (argc < 2) return 2;
    FILE *fp = fopen(argv[1], "rb");
    if (!fp) return 2;
    int32_t head[2];
    while (fread(head, sizeof(head), 1, fp) == 1) {
        dspx_flac_file file;
        if (fread(&file, sizeof(file), 1, fp) != 1) return 3;
        file.in_offset = 0;
        file.out_start = 0;
        std::vector<float> out(file.out_length);
        for (int32_t f = 0; f < head[1]; f++) {
            dspx_flac_frame fr;
            if (fread(&fr, sizeof(fr), 1, fp) != 1) return 3;
            const int64_t slack = fr.in_offset & 3;
            unsigned char *buf = static_cast<unsigned char *>(malloc(slack + fr.in_bytes));
            if (fread(buf + slack, 1, fr.in_bytes, fp) != (size_t)fr.in_bytes) return 3;
            ASAN_POISON_MEMORY_REGION(buf, slack);
            fr.in_offset = slack;
            fr.file = 0;
            int32_t status = -1;
            int rc = 0;
            for (int normalize = 0; normalize < 2; normalize++)
                rc |= emu_flac_decode(buf, &file, 1, &fr, 1, normalize, out.data(), &status);
            printf("flac case %d frame %d rc %d status %d\n", head[0], f, rc, status);
            ASAN_UNPOISON_MEMORY_REGION(buf, slack);
            free(buf);
        }
    }
    fclose(fp);
    return 0;
}
