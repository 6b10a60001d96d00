/* fisheye_b200.c — drop-in replacement for TyrQuake/Blinky's engine/NQ/fisheye.c.
 *
 * Same link-level seam as the reference (engine/include/fisheye.h:4-9): exports
 * F_Init, F_Shutdown, F_RenderView, F_WriteConfig and the two globals the
 * renderer reads (fisheye_enabled, fisheye_plate_fov); imports the same engine
 * symbols (Cmd_*, Con_Printf, vid, scr_vrect, r_refdef, R_RenderView, ...).  The
 * host side stays C; everything else goes through the thin C ABI of
 * libblinky_b200.so (include/blinky_b200.h):
 *
 *   scripts / console / zoom / lensmap build  -> blinky_command, blinky_build_lensmap (host)
 *   render_lensmap() (fisheye.c:2406-2424)    -> blinky_warp_host (sm_100a CUDA kernels)
 *
 * Build: compile this file instead of NQ/fisheye.c (engine/Makefile:645) with
 * the engine's include paths plus -I<repo>/include, and add -lblinky_b200 where
 * the reference adds -llua (engine/Makefile:834-841).  See INTEGRATION.md.
 *
 * Differences a maintainer should know about:
 *  - the lensmap is built in one shot — lens_inverse translated to CUDA and evaluated on
 *    the GPU, or interpreted on host threads — instead of being time-sliced over frames
 *    (fisheye.c:301-322, 819-826).  Like the reference's builder it never holds a frame up:
 *    the build runs on a worker thread in a second library context while F_RenderView keeps
 *    warping with the previous lensmap (or draws only the background when the view size or
 *    the globe changed, the reference's freshly wiped map), and the two contexts swap when
 *    the build is done.  BLINKY_SYNC_BUILD=1 restores the blocking build;
 *  - globe.pixels lives in pinned host memory so plates upload with
 *    cudaMemcpyAsync; only plates the lens looks at are uploaded;
 *  - f_saveglobe writes the PCX files itself (into com_gamedir) instead of going
 *    through COM_WriteFile.
 */
#include "bspfile.h"
#include "client.h"
#include "cmd.h"
#include "console.h"
#include "cvar.h"
#include "draw.h"
#include "fisheye.h"
#include "host.h"
#include "mathlib.h"
#include "quakedef.h"
#include "r_local.h"
#include "screen.h"
#include "sys.h"
#include "view.h"

#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "blinky_b200.h"

/* read by view.c / r_main.c / r_misc.c exactly like the reference's (fisheye.c:293, 299) */
qboolean fisheye_enabled;
double fisheye_plate_fov;

/* Two library contexts with the same console state.  ctx[front] owns the lensmap that is on
 * screen; a rebuild happens in the other one on a worker thread, then they swap. */
static blinky_ctx *ctx[2];
static int front;
#define b200 (ctx[front])
static byte *globe_pixels;      /* pinned; [numplates][platesize][platesize] like GLOBEPIXEL (fisheye.c:349) */
static size_t globe_bytes;
static int build_threads = 0; /* 0 = lens evaluated on the GPU (BLINKY_BUILD_THREADS overrides) */
static int sync_build = 0;    /* BLINKY_SYNC_BUILD=1: build inside F_RenderView like round 1 */

/* what the lensmap on screen was built for (cached: the console may already have moved on) */
static struct {
    int valid, width, height, platesize, numplates;
    int display[BLINKY_MAX_PLATES];
    float plates[BLINKY_MAX_PLATES * 11];
    double fov[BLINKY_MAX_PLATES];
} shown;

/* the worker */
static pthread_t build_thread;
static volatile int build_running, build_done;
static int build_w, build_h, build_ps;
#define MAX_QUEUED 64
static char *queued_cmds[MAX_QUEUED]; /* console lines that arrived while the back context was busy */
static int n_queued;

/* exposed for harnesses/tests (not part of the engine seam) */
blinky_ctx *F_B200_Context(void) { return b200; }
int F_B200_Building(void) { return build_running; }
int F_B200_ShownDisplay(int *display, int *numplates)
{
    memcpy(display, shown.display, sizeof shown.display);
    *numplates = shown.valid ? shown.numplates : 0;
    return shown.valid;
}

static void to_console(const char *text, void *user)
{
    (void)user;
    Con_Printf("%s", text);
}

static void to_cmd(const char *command, void *user)
{
    (void)user;
    Cmd_ExecuteString(command, src_command); /* a lens's `onload` may be any console command */
}

/* A context's first blinky_warp_host sets up its copy pipeline (streams, device slots, pinned
 * staging): tens of milliseconds.  The back context pays that here, on the worker, with the kinds of
 * buffers F_RenderView passes (pinned faces, an unpinned screen, keep_unmapped), instead of in the
 * first frame after the swap.  Best effort: a failure here only moves the cost back to that frame. */
static void warm_up(blinky_ctx *c)
{
    size_t faces = (size_t)build_ps * build_ps * BLINKY_MAX_PLATES;
    void *src = NULL;
    byte *dst;

    if (blinky_alloc_pinned(c, faces, &src) != BLINKY_OK) return;
    memset(src, 0, faces);
    dst = malloc((size_t)build_w * build_h);
    if (dst) {
        blinky_warp_host(c, src, faces, dst, 0, build_w, 0, 0, 1, 1);
        free(dst);
    }
    blinky_free_pinned(c, src);
}

static void *build_worker(void *arg)
{
    (void)arg;
    /* errors (invalid lens, zoom failure, ...) are collected in the context's log and printed by the
     * main thread at the swap; like the reference, an empty map simply draws nothing */
    blinky_build_lensmap(ctx[1 - front], build_w, build_h, build_ps, build_threads);
    warm_up(ctx[1 - front]);
    __sync_synchronize();
    build_done = 1;
    return NULL;
}

static void snapshot_shown(int width, int height, int platesize)
{
    int i;
    shown.valid = 1;
    shown.width = width;
    shown.height = height;
    shown.platesize = platesize;
    shown.numplates = blinky_get_plates(b200, shown.plates, BLINKY_MAX_PLATES);
    blinky_get_display(b200, shown.display);
    for (i = 0; i < shown.numplates; ++i) shown.fov[i] = blinky_plate_fov(b200, i);
}

/* the back context caught up: swap, print what the build had to say, replay the queued console lines */
static void finish_build(void)
{
    int i;
    pthread_join(build_thread, NULL);
    build_running = build_done = 0;
    front = 1 - front;
    {
        const char *log = blinky_log(b200);
        if (log && log[0]) Con_Printf("%s", log);
        blinky_log_clear(b200);
    }
    blinky_set_print_callback(b200, to_console, NULL);
    blinky_set_exec_callback(b200, to_cmd, NULL);
    blinky_set_print_callback(ctx[1 - front], NULL, NULL);
    blinky_set_exec_callback(ctx[1 - front], NULL, NULL);
    snapshot_shown(build_w, build_h, build_ps);
    /* lines typed during the build went to the old front only */
    for (i = 0; i < n_queued; ++i) {
        blinky_command(b200, queued_cmds[i]);
        free(queued_cmds[i]);
    }
    n_queued = 0;
    blinky_log_clear(b200); /* their messages were already printed when they were typed */
}

void F_B200_WaitBuild(void)
{
    if (build_running) finish_build(); /* pthread_join blocks until the worker is done */
}

/* Every f_* console command re-assembles its argument line and hands it to the
 * library, which implements the reference's command semantics and messages.  Both contexts
 * hear every line: the front one answers on the console, the back one stays silent (its
 * `onload` is not executed again: the front's already came through here). */
static void forward_command(void)
{
    char line[1024];
    size_t n = 0;
    int i;
    for (i = 0; i < Cmd_Argc() && n < sizeof(line) - 4; i++) {
        const char *a = Cmd_Argv(i);
        int quote = i > 0 && (strchr(a, ' ') != NULL || a[0] == 0);
        n += (size_t)snprintf(line + n, sizeof(line) - n, "%s%s%s%s", i ? " " : "", quote ? "\"" : "", a, quote ? "\"" : "");
    }
    line[n < sizeof(line) ? n : sizeof(line) - 1] = 0;
    blinky_command(b200, line);
    if (ctx[1 - front]) {
        if (build_running) {
            if (n_queued < MAX_QUEUED) queued_cmds[n_queued++] = strdup(line);
        } else {
            blinky_command(ctx[1 - front], line);
            blinky_log_clear(ctx[1 - front]);
        }
    }
    if (!strcasecmp(Cmd_Argv(0), "fisheye") && Cmd_Argc() >= 2) {
        fisheye_enabled = blinky_fisheye_enabled(b200);
        vid.recalc_refdef = true; /* fisheye.c:976 */
    }
}

static struct stree_root *complete_from(const char *dir, const char *arg)
{
    struct stree_root *root = Z_Malloc(sizeof(struct stree_root));
    if (root) {
        *root = STREE_ROOT;
        STree_AllocInit();
        COM_ScanDir(root, dir, arg, ".lua", true);
    }
    return root;
}
static struct stree_root *cmdarg_lens(const char *arg) { return complete_from("../lua-scripts/lenses", arg); }
static struct stree_root *cmdarg_globe(const char *arg) { return complete_from("../lua-scripts/globes", arg); }

void F_Init(void)
{
    static const char *commands[] = {"fisheye", "f_help", "f_dumppal", "f_rubix", "f_rubixgrid", "f_cover", "f_contain",
                                     "f_fov", "f_vfov", "f_lens", "f_globe", "f_saveglobe", "f_shortcutkeys"};
    const char *dev = getenv("BLINKY_DEVICE");
    const char *thr = getenv("BLINKY_BUILD_THREADS");
    const char *syn = getenv("BLINKY_SYNC_BUILD");
    size_t i;
    int rc;
    front = 0;
    memset(&shown, 0, sizeof shown);
    rc = blinky_create(dev ? atoi(dev) : 0, &ctx[0]);
    if (rc != BLINKY_OK) {
        Con_Printf("fisheye_b200: %s\n", ctx[0] ? blinky_last_error(ctx[0]) : "out of memory");
        /* no CPU fallback: leave fisheye off rather than pretend */
        fisheye_enabled = false;
        if (ctx[0]) {
            blinky_destroy(ctx[0]);
            ctx[0] = NULL;
        }
        return;
    }
    if (thr) build_threads = atoi(thr);
    sync_build = syn && atoi(syn) != 0;
    blinky_set_print_callback(b200, to_console, NULL);
    blinky_set_exec_callback(b200, to_cmd, NULL);
    blinky_set_basedir(b200, com_basedir);
    if (!sync_build) { /* the second context rebuilds lensmaps off the frame loop */
        if (blinky_create(dev ? atoi(dev) : 0, &ctx[1]) == BLINKY_OK) {
            blinky_set_basedir(ctx[1], com_basedir);
        } else {
            if (ctx[1]) blinky_destroy(ctx[1]);
            ctx[1] = NULL;
            sync_build = 1;
        }
    }

    for (i = 0; i < sizeof(commands) / sizeof(commands[0]); i++) Cmd_AddCommand(commands[i], forward_command);
    Cmd_SetCompletion("f_lens", cmdarg_lens);
    Cmd_SetCompletion("f_globe", cmdarg_globe);

    /* defaults, through the console like the reference (fisheye.c:668-672) */
    Cmd_ExecuteString("fisheye 1", src_command);
    Cmd_ExecuteString("f_globe cube", src_command);
    Cmd_ExecuteString("f_lens panini", src_command);
    Cmd_ExecuteString("f_fov 180", src_command);
    Cmd_ExecuteString("f_rubixgrid 10 4 1", src_command);

    blinky_set_palette(b200, host_basepal); /* create_palmap, fisheye.c:675 */
    if (ctx[1]) blinky_set_palette(ctx[1], host_basepal);
}

void F_Shutdown(void)
{
    int i;
    if (!b200) return;
    F_B200_WaitBuild();
    if (globe_pixels) blinky_free_pinned(b200, globe_pixels);
    globe_pixels = NULL;
    globe_bytes = 0;
    for (i = 0; i < 2; ++i) {
        if (ctx[i]) blinky_destroy(ctx[i]);
        ctx[i] = NULL;
    }
    front = 0;
    shown.valid = 0;
}

void F_WriteConfig(FILE *f)
{
    char buf[1024];
    if (!b200) return;
    blinky_write_config(b200, buf, sizeof buf);
    fputs(buf, f);
}

/* copy the freshly rendered view out of vid.buffer into this plate's slot (fisheye.c:2427-2450) */
static void render_plate(int plate_index, int platesize, vec3_t forward, vec3_t right, vec3_t up)
{
    byte *pixels = globe_pixels + (size_t)plate_index * platesize * platesize;
    byte *vbuffer = vid.buffer + scr_vrect.x + scr_vrect.y * vid.rowbytes;
    int y;

    VectorCopy(forward, r_refdef.forward);
    VectorCopy(right, r_refdef.right);
    VectorCopy(up, r_refdef.up);

    R_PushDlights();
    R_RenderView();

    for (y = 0; y < platesize; y++) {
        memcpy(pixels, vbuffer, (size_t)platesize);
        vbuffer += vid.rowbytes;
        pixels += platesize;
    }
}

void F_RenderView(void)
{
    extern int sb_lines;
    int width = scr_vrect.width, height = scr_vrect.height;
    int platesize = width < height ? width : height; /* fisheye.c:707 */
    int i, usable;
    vec3_t forward, right, up;
    vrect_t vrect;

    if (!b200) return;

    if (build_running && build_done) finish_build();
    if (!build_running && blinky_needs_rebuild(b200, width, height, platesize)) { /* fisheye.c:730 */
        size_t need = (size_t)platesize * platesize * BLINKY_MAX_PLATES;
        if (need != globe_bytes) {
            if (globe_pixels) blinky_free_pinned(b200, globe_pixels);
            globe_pixels = NULL;
            if (blinky_alloc_pinned(b200, need, (void **)&globe_pixels) != BLINKY_OK) {
                Con_Printf("Quake-Lenses: could not allocate enough memory\n");
                globe_bytes = 0;
                return; /* the reference exit(1)s here (fisheye.c:723-726) */
            }
            globe_bytes = need;
        }
        if (sync_build) {
            /* errors (invalid lens, zoom failure, ...) were already printed through Con_Printf;
             * like the reference, an empty map simply draws nothing */
            blinky_build_lensmap(b200, width, height, platesize, build_threads);
            snapshot_shown(width, height, platesize);
        } else {
            build_w = width;
            build_h = height;
            build_ps = platesize;
            build_done = 0;
            build_running = 1;
            if (pthread_create(&build_thread, NULL, build_worker, NULL) != 0) {
                build_running = 0;
                blinky_build_lensmap(b200, width, height, platesize, build_threads);
                snapshot_shown(width, height, platesize);
            }
        }
    }
    if (!globe_pixels) return;

    AngleVectors(r_refdef.viewangles, forward, right, up);
    vrect.x = 0;
    vrect.y = 0;
    vrect.width = vid.width;
    vrect.height = vid.height;
    R_SetVrect(&vrect, &scr_vrect, sb_lines);

    /* the map on screen can be used while its successor is built as long as it was made for this view
     * size (the plates keep their layout); otherwise this frame shows the cleared background only */
    usable = shown.valid && shown.width == width && shown.height == height && shown.platesize == platesize;
    for (i = 0; usable && i < shown.numplates; ++i) {
        if (shown.display[i]) {
            const float *pf = shown.plates + i * 11, *pr = pf + 3, *pu = pf + 6;
            vec3_t r = {0, 0, 0}, u = {0, 0, 0}, f = {0, 0, 0};

            fisheye_plate_fov = shown.fov[i]; /* fisheye.c:769 */
            R_ViewChanged(&vrect, sb_lines, vid.aspect);

            /* plate basis (relative to the camera) -> world (fisheye.c:777-790) */
            VectorMA(r, pr[0], right, r);
            VectorMA(r, pr[1], up, r);
            VectorMA(r, pr[2], forward, r);
            VectorMA(u, pu[0], right, u);
            VectorMA(u, pu[1], up, u);
            VectorMA(u, pu[2], forward, u);
            VectorMA(f, pf[0], right, f);
            VectorMA(f, pf[1], up, f);
            VectorMA(f, pf[2], forward, f);

            render_plate(i, platesize, f, r, u);
        }
    }

    if (usable && blinky_saveglobe_pending(b200)) { /* fisheye.c:797-799 */
        D_EnableBackBufferAccess();
        blinky_save_globe(b200, globe_pixels, com_gamedir);
        D_DisableBackBufferAccess();
    }

    Draw_TileClear(0, 0, vid.width, vid.height); /* background for pixels the lens does not map */
    if (!usable) return;

    /* render_lensmap() on the GPU; keep_unmapped=1: only mapped pixels are written */
    if (blinky_warp_host(b200, globe_pixels, globe_bytes, vid.buffer, 0, vid.rowbytes, scr_vrect.x, scr_vrect.y, 1, 1) != BLINKY_OK)
        Con_Printf("fisheye_b200: %s\n", blinky_last_error(b200));
}
